// Beam search on the device (SURVEY.md §8f rank 1: `num_beams=5` is what the reference's literal pipeline call runs under
// transformers >= 4.53).  Restates GenerationMixin._beam_search ($TF/generation/utils.py:3076-3400; helpers :2876-3075)
// and the three Whisper logits processors applied to LOG-PROBABILITIES ($TF/generation/logits_process.py:1812-2043)
// for `windows x beams` decode rows, early_stopping=False, do_sample=False, one returned sequence per window.
//
// One search step = three launches appended to the decode step (all inside one CUDA graph, no host control):
//   beam_row_topk_kernel   one CTA per decode row: fp32 log-softmax over the whole vocabulary of the row's raw logits
//                          (the LM head's tap), THEN the processors (suppress lists, timestamp grammar from the row's
//                          carried state, the sum-of-timestamp-probability rule), + the row's running score; the row
//                          is staged once in shared memory and its best 2K continuations are extracted by 2K block
//                          arg-max rounds (any of the window's best 2K of K*V lies in its row's best 2K).
//   beam_advance_kernel    one CTA per window: K-way merge of the rows' lists into the window's best 2K, the
//                          running / finished bookkeeping of _beam_search (hits, 2K -> K running, finished-slot merge
//                          ranked by score / generated_length**length_penalty, `improvable`, the global stop test),
//                          the token / beam-index histories (double-buffered, gathered by beam of origin), the next
//                          token and grammar state of every decode row, and the self-attention KV cache re-gather as a
//                          BLOCK-TABLE PERMUTATION: full pages are inherited by pointer, only the partial current page
//                          is copied (into the row's own slot of the other bank), by
//   beam_copy_pages_kernel one CTA per (row, layer, k|v).
// The scalar logic is `__host__ __device__` so that the same code runs on the CPU behind tw_beam_step_host, where
// tests/test_beam_cpu.py checks it token-exactly against the oracle's beam search (itself pinned to transformers).
#include "common.cuh"
#include "twb200_internal.h"
#include <math.h>
#include <string.h>
#include <vector>

namespace tw {
namespace beam {

constexpr int MAXK = 8;          // beams per window
constexpr int MAXC = 2 * MAXK;   // candidates per window
constexpr float NEG = -1.0e9f;
constexpr int PAGE = 64;

struct Cfg {
    int K, V, L, P, eos, pad, no_ts, max_initial_ts, timestamps, track;
    float length_penalty;
};

#define HD __host__ __device__ __forceinline__

// grammar state carried per running row: what WhisperTimeStampLogitsProcessor derives from the generated ids
struct Gram {
    int last_is_ts;   // last generated token is a timestamp
    int pen_is_ts;    // the one before it is (true while fewer than two tokens were generated)
    int last_ts;      // value of the last timestamp token generated so far, -1: none
    int pad_;
};

HD bool bit(const uint32_t* bits, int v) { return (bits[v >> 5] >> (v & 31)) & 1u; }

// SuppressTokens -> SuppressTokensAtBegin -> WhisperTimeStamp (everything but the probability rule)
HD bool allowed(int v, const Gram& g, int n_gen, const Cfg& c, const uint32_t* sup, const uint32_t* bsup) {
    if (bit(sup, v)) return false;
    if (n_gen == 0 && bit(bsup, v)) return false;
    if (!c.timestamps) return true;
    if (v == c.no_ts) return false;
    const int TB = c.no_ts + 1;
    if (n_gen == 0) {
        if (v < TB) return false;
        return c.max_initial_ts < 0 || v <= TB + c.max_initial_ts;
    }
    if (g.last_is_ts) {
        if (g.pen_is_ts) { if (v >= TB) return false; }
        else if (v < c.eos) return false;
    }
    if (g.last_ts >= 0 && v >= TB) {
        const int bound = (g.last_is_ts && !g.pen_is_ts) ? g.last_ts : g.last_ts + 1;
        if (v < bound) return false;
    }
    return true;
}

HD Gram gram_after(const Gram& g, int n_gen_before, int tok, const Cfg& c) {
    Gram o;
    const bool is_ts = tok >= c.no_ts + 1;
    o.pen_is_ts = (n_gen_before == 0) ? 1 : g.last_is_ts;
    o.last_is_ts = is_ts ? 1 : 0;
    o.last_ts = is_ts ? tok : g.last_ts;
    o.pad_ = 0;
    return o;
}

// ---------------------------------------------------------------------------------------------------------------
// window bookkeeping (scalar; one thread on the device)
// ---------------------------------------------------------------------------------------------------------------
struct Plan {
    int n_cand;
    float top_lp[MAXC];
    int origin[MAXC], tok[MAXC], hit[MAXC];
    int run_src[MAXK];      // candidate index each new running slot continues
    float run_score[MAXK];
    int fin_src[MAXK];      // < K: old finished slot; >= K: candidate (fin_src - K)
    float fin_score[MAXK];
    int fin_flag[MAXK], fin_len[MAXK];
    int improvable, hits_all;
};

// descending by value, earlier index first on ties; selects the best `k` of `n` into idx[]
HD void top_k_small(const float* val, int n, int k, int* idx) {
    bool used[MAXK + MAXC];
    for (int i = 0; i < n; ++i) used[i] = false;
    for (int s = 0; s < k; ++s) {
        int best = -1;
        for (int i = 0; i < n; ++i)
            if (!used[i] && (best < 0 || val[i] > val[best])) best = i;
        used[best] = true;
        idx[s] = best;
    }
}

// cand_val / cand_tok: the K rows' sorted lists [K][2K].  cur = index the new token is written to.
HD void plan_window(const Cfg& c, int cur, const float* cand_val, const int* cand_tok, const float* old_fin_score,
                    const int* old_fin_flag, const int* old_fin_len, int old_improvable, Plan& p) {
    const int K = c.K, C = 2 * c.K;
    // K-way merge of the rows' descending lists: the window's best 2K of K*V, ties -> lower flat index k*V + tok
    int head[MAXK];
    for (int k = 0; k < K; ++k) head[k] = 0;
    for (int s = 0; s < C; ++s) {
        int bk = -1;
        for (int k = 0; k < K; ++k) {
            if (head[k] >= C) continue;
            if (bk < 0) { bk = k; continue; }
            const float a = cand_val[k * C + head[k]], b = cand_val[bk * C + head[bk]];
            if (a > b) bk = k;   // equal values: the lower row index (lower flat index) stays
        }
        p.top_lp[s] = cand_val[bk * C + head[bk]];
        p.tok[s] = cand_tok[bk * C + head[bk]];
        p.origin[s] = bk;
        ++head[bk];
    }
    p.n_cand = C;
    float run_lp[MAXC];
    bool all_hit = true;
    for (int s = 0; s < C; ++s) {
        p.hit[s] = (p.tok[s] == c.eos) || (cur + 1 >= c.L);
        all_hit = all_hit && p.hit[s];
        run_lp[s] = p.hit[s] ? p.top_lp[s] + NEG : p.top_lp[s];
    }
    p.hits_all = all_hit;
    top_k_small(run_lp, C, K, p.run_src);
    for (int i = 0; i < K; ++i) p.run_score[i] = run_lp[p.run_src[i]];
    // finished slots: the old K and the candidates that just finished among the best K, ranked by
    // score / generated_length ** length_penalty
    const int gen_len = cur + 1 - c.P;
    const float denom = (float)pow((double)gen_len, (double)c.length_penalty);
    float m_lp[MAXK + MAXC];
    for (int k = 0; k < K; ++k) m_lp[k] = old_fin_score[k];
    for (int s = 0; s < C; ++s) {
        const bool just = p.hit[s] && s < K;
        float f = p.top_lp[s] / denom;
        if (!old_improvable) f += NEG;
        if (!just) f += NEG;
        m_lp[K + s] = f;
    }
    top_k_small(m_lp, K + C, K, p.fin_src);
    for (int i = 0; i < K; ++i) {
        const int j = p.fin_src[i];
        p.fin_score[i] = m_lp[j];
        if (j < K) { p.fin_flag[i] = old_fin_flag[j]; p.fin_len[i] = old_fin_len[j]; }
        else { p.fin_flag[i] = (p.hit[j - K] && (j - K) < K) ? 1 : 0; p.fin_len[i] = gen_len; }
    }
    // can a running beam still beat the worst finished one?
    const float best_possible = p.run_score[0] / denom;
    float worst = p.fin_score[0];
    for (int i = 1; i < K; ++i) worst = fminf(worst, p.fin_score[i]);
    bool any = false;
    for (int i = 0; i < K; ++i) any = any || (best_possible > (p.fin_flag[i] ? worst : NEG));
    p.improvable = (old_improvable && any) ? 1 : 0;
}

// record of one hypothesis: [0, L) tokens, [L, 2L) HF's beam_indices (only when tracked)
HD int rec_width(const Cfg& c) { return c.track ? 2 * c.L : c.L; }

struct State {
    int* hist;          // [2][n][K][W] running hypotheses (double-buffered by ctrl[0])
    int* fin;           // [2][n][K][W] finished hypotheses
    float* run_score;   // [n][K]
    float* fin_score;   // [n][K]
    int* fin_flag;      // [n][K]
    int* fin_len;       // [n][K]
    Gram* gram;         // [n][K]
    int* improvable;    // [n]
    int* hits_all;      // [n]
    int* ctrl;          // [0] history parity, [1] done, [2] arrival counter, [3] KV bank, [4] steps taken
};

// copies performed for window w once its plan is known; (tid, nt) = cooperating thread and count
HD void apply_plan_rows(const Cfg& c, const State& s, const Plan& p, int n, int w, int cur, int par, int tid, int nt) {
    const int K = c.K, W = rec_width(c), L = c.L;
    const size_t half = (size_t)n * K * W;
    const int* old_run = s.hist + par * half + (size_t)w * K * W;
    int* new_run = s.hist + (par ^ 1) * half + (size_t)w * K * W;
    const int* old_fin = s.fin + par * half + (size_t)w * K * W;
    int* new_fin = s.fin + (par ^ 1) * half + (size_t)w * K * W;
    const int g = cur - c.P;   // generated index of the new token
    for (int i = 0; i < K; ++i) {
        const int cs = p.run_src[i], o = p.origin[cs];
        for (int t = tid; t < cur; t += nt) new_run[i * W + t] = old_run[o * W + t];
        if (c.track)
            for (int t = tid; t < g; t += nt) new_run[i * W + L + t] = old_run[o * W + L + t];
        if (tid == 0) {
            new_run[i * W + cur] = p.tok[cs];
            if (c.track) new_run[i * W + L + g] = w * K + o;
        }
        const int j = p.fin_src[i];
        if (j < K) {
            for (int t = tid; t < W; t += nt) new_fin[i * W + t] = old_fin[j * W + t];
        } else {
            const int fo = p.origin[j - K];
            for (int t = tid; t < L; t += nt)
                new_fin[i * W + t] = t < cur ? old_run[fo * W + t] : (t == cur ? p.tok[j - K] : c.pad);
            if (c.track)
                for (int t = tid; t < L; t += nt)
                    new_fin[i * W + L + t] = t < g ? old_run[fo * W + L + t] : (t == g ? w * K + fo : -1);
        }
    }
}

#ifndef TW_HOST_TEST
// ---------------------------------------------------------------------------------------------------------------
// device kernels
// ---------------------------------------------------------------------------------------------------------------
constexpr int TOPK_THREADS = 1024;

struct TopkParams {
    const float* logits;      // [R][V] raw fp32 logits of this step
    const tw_row_state* st;   // [R]
    const float* run_score;   // [R]
    const Gram* gram;         // [R]
    const uint32_t* sup;
    const uint32_t* bsup;
    const int* ctrl;
    float* cand_val;          // [R][2K]
    int* cand_tok;            // [R][2K]
    Cfg c;
};

TW_DEVINL float block_max(float v, float* red) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    v = warp_max(v);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float m = red[0];
    for (int i = 1; i < (int)(blockDim.x >> 5); ++i) m = fmaxf(m, red[i]);
    return m;
}
TW_DEVINL float block_sum(float v, float* red) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float m = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) m += red[i];
    return m;
}

__global__ void __launch_bounds__(TOPK_THREADS, 1) beam_row_topk_kernel(const TopkParams p) {
    extern __shared__ float row[];            // [V] processed, accumulated scores of this row
    __shared__ float red[32];
    __shared__ int redi[32];
    const Cfg& c = p.c;
    const int r = blockIdx.x, tid = threadIdx.x;
    const int V = c.V, TB = c.no_ts + 1, C = 2 * c.K;
    if (p.ctrl[1]) return;                    // search over: state is frozen
    const int n_gen = p.st[r].pos + 1 - c.P;
    const Gram g = p.gram[r];
    const float* x = p.logits + (size_t)r * V;
    // log-softmax over the WHOLE vocabulary first ($TF/generation/utils.py:3230: log_softmax, then the processors)
    float mx = -INFINITY;
    for (int v = tid; v < V; v += TOPK_THREADS) { const float t = x[v]; row[v] = t; mx = fmaxf(mx, t); }
    mx = block_max(mx, red);
    float sum = 0.f;
    for (int v = tid; v < V; v += TOPK_THREADS) sum += expf(row[v] - mx);
    sum = block_sum(sum, red);
    const float lse = logf(sum);
    // processors on the log-probabilities; statistics of the timestamp-probability rule
    float mt = -INFINITY, ms = -INFINITY;
    for (int v = tid; v < V; v += TOPK_THREADS) {
        float lp = (row[v] - mx) - lse;
        if (!allowed(v, g, n_gen, c, p.sup, p.bsup)) lp = -INFINITY;
        row[v] = lp;
        if (v >= TB) ms = fmaxf(ms, lp); else mt = fmaxf(mt, lp);
    }
    if (c.timestamps) {
        mt = block_max(mt, red);
        ms = block_max(ms, red);
        float ss = 0.f;
        if (ms > -INFINITY)
            for (int v = TB + tid; v < V; v += TOPK_THREADS) ss += expf(row[v] - ms);   // exp(-inf) = 0 for masked ids
        ss = block_sum(ss, red);
        const bool ts_heavier = (ms > -INFINITY) && (ms + logf(ss) > mt);
        if (ts_heavier)
            for (int v = tid; v < TB; v += TOPK_THREADS) row[v] = -INFINITY;
    }
    const float base = p.run_score[r];
    __syncthreads();
    for (int v = tid; v < V; v += TOPK_THREADS) row[v] += base;
    __syncthreads();
    // 2K rounds of block arg-max (value desc, lower id on ties); each thread re-scans its ~51 strided entries
    for (int s = 0; s < C; ++s) {
        float bv = -INFINITY;
        int bi = 0x7fffffff;
        for (int v = tid; v < V; v += TOPK_THREADS) {
            const float t = row[v];
            if (t > bv) { bv = t; bi = v; }        // ascending v: the first maximum is the lowest id
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bv, d);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, d);
            if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
        }
        if ((tid & 31) == 0) { red[tid >> 5] = bv; redi[tid >> 5] = bi; }
        __syncthreads();
        if (tid < 32) {
            bv = red[tid]; bi = redi[tid];
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
                const float ov = __shfl_xor_sync(0xffffffffu, bv, d);
                const int oi = __shfl_xor_sync(0xffffffffu, bi, d);
                if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
            }
            if (tid == 0) {
                if (bi == 0x7fffffff) { bi = 0; }      // fewer than 2K admissible ids: -inf filler
                p.cand_val[r * C + s] = bv;
                p.cand_tok[r * C + s] = bi;
                if (bv > -INFINITY) row[bi] = -INFINITY;
            }
        }
        __syncthreads();
    }
}

struct AdvanceParams {
    State s;
    const float* cand_val;
    const int* cand_tok;
    tw_row_state* st;      // [R]
    int* tokens;           // [R][tokens_ld]: the token every decode row feeds next is written at index cur
    int tokens_ld;
    int* block_table;      // [R][ppr]
    int ppr, bank_pages;   // pages per row; pages per bank (= max rows * ppr)
    int* copy_src;         // [R] page the row's partial current page is copied from (-1: none)
    int* copy_dst;         // [R]
    int* copy_len;         // [1] positions to copy
    int* origin_out;       // [R] previous row each new row continues
    int n;
    Cfg c;
};

__global__ void __launch_bounds__(128) beam_advance_kernel(const AdvanceParams p) {
    __shared__ Plan plan;
    __shared__ int s_bt[MAXK * 8];
    __shared__ int s_last;
    const Cfg& c = p.c;
    const int w = blockIdx.x, tid = threadIdx.x, K = c.K, C = 2 * c.K;
    if (p.s.ctrl[1]) return;                     // search over: nothing changes any more
    const int par = p.s.ctrl[0], bank = p.s.ctrl[3];
    const int cur = p.st[w * K].pos + 1;         // index the new token is written to (same for every row)
    for (int i = tid; i < K * p.ppr; i += 128) s_bt[i] = p.block_table[w * K * p.ppr + i];
    if (tid == 0)
        plan_window(c, cur, p.cand_val + (size_t)w * K * C, p.cand_tok + (size_t)w * K * C, p.s.fin_score + w * K,
                    p.s.fin_flag + w * K, p.s.fin_len + w * K, p.s.improvable[w], plan);
    __syncthreads();
    apply_plan_rows(c, p.s, plan, p.n, w, cur, par, tid, 128);
    // KV cache: positions 0..cur-1 are cached; the next step writes position cur into page cur / 64
    const int pn = cur / PAGE, fill = cur % PAGE;
    if (tid < K) {
        const int i = tid, r = w * K + i, cs = plan.run_src[i], o = plan.origin[cs];
        for (int q = 0; q < pn && q < p.ppr; ++q) p.block_table[r * p.ppr + q] = s_bt[o * p.ppr + q];
        if (pn < p.ppr) {
            const int dst = (bank ^ 1) * p.bank_pages + r * p.ppr + pn;   // the row's own slot in the other bank
            p.block_table[r * p.ppr + pn] = dst;
            p.copy_dst[r] = dst;
            p.copy_src[r] = fill ? s_bt[o * p.ppr + pn] : -1;
        } else {
            p.copy_src[r] = -1;
        }
        p.origin_out[r] = w * K + o;
        // the decode row: next token, position, grammar state
        if (cur < p.tokens_ld) p.tokens[(size_t)r * p.tokens_ld + cur] = plan.tok[cs];
        tw_row_state st = p.st[r];
        st.pos = cur;
        st.finished = 0;
        p.st[r] = st;
    }
    __shared__ Gram s_gram[MAXK];
    if (tid < K) s_gram[tid] = p.s.gram[w * K + tid];
    __syncthreads();
    if (tid < K) {
        const int cs = plan.run_src[tid];
        p.s.gram[w * K + tid] = gram_after(s_gram[plan.origin[cs]], cur - c.P, plan.tok[cs], c);
        p.s.run_score[w * K + tid] = plan.run_score[tid];
        p.s.fin_score[w * K + tid] = plan.fin_score[tid];
        p.s.fin_flag[w * K + tid] = plan.fin_flag[tid];
        p.s.fin_len[w * K + tid] = plan.fin_len[tid];
    }
    if (tid == 0) {
        p.s.improvable[w] = plan.improvable;
        p.s.hits_all[w] = plan.hits_all;
    }
    // the last window to finish evaluates the global stop test and flips the double buffers
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const int prev = atomicAdd(&p.s.ctrl[2], 1);
        s_last = (prev == (int)gridDim.x - 1);
    }
    __syncthreads();
    if (s_last && tid == 0) {
        __threadfence();
        bool any_improvable = false, all_hits = true;
        for (int i = 0; i < p.n; ++i) {
            any_improvable = any_improvable || __ldcg(&p.s.improvable[i]);
            all_hits = all_hits && __ldcg(&p.s.hits_all[i]);
        }
        p.s.ctrl[0] = par ^ 1;
        p.s.ctrl[3] = bank ^ 1;
        p.s.ctrl[4] += 1;
        p.s.ctrl[2] = 0;
        *p.copy_len = fill;
        if (!(any_improvable && !all_hits)) p.s.ctrl[1] = 1;
    }
}

struct CopyParams {
    __nv_bfloat16* pool;     // [L][2][n_pages][PAGE][D]
    const int* copy_src;
    const int* copy_dst;
    const int* copy_len;
    const int* ctrl;
    int n_pages, D;
};

__global__ void __launch_bounds__(256) beam_copy_pages_kernel(const CopyParams p) {
    const int r = blockIdx.x, lk = blockIdx.y;
    const int src = p.copy_src[r], len = *p.copy_len;
    if (src < 0 || len <= 0) return;
    const int dst = p.copy_dst[r];
    const uint4* s = reinterpret_cast<const uint4*>(p.pool + ((size_t)lk * p.n_pages + src) * PAGE * p.D);
    uint4* d = reinterpret_cast<uint4*>(p.pool + ((size_t)lk * p.n_pages + dst) * PAGE * p.D);
    const int n16 = len * p.D / 8;
    for (int i = threadIdx.x; i < n16; i += 256) d[i] = s[i];
}
#endif  // TW_HOST_TEST

}  // namespace beam
}  // namespace tw

// ================================================================================================
// C ABI
// ================================================================================================
using namespace tw;
using namespace tw::beam;

static int to_cfg(const tw_beam_config* b, Cfg& c, const char* who) {
    TW_REQUIRE(b, "%s: null config", who);
    TW_REQUIRE(b->num_beams >= 1 && b->num_beams <= MAXK, "%s: num_beams %d not in [1,%d]", who, b->num_beams, MAXK);
    TW_REQUIRE(b->prompt_len >= 1 && b->prompt_len < b->max_length, "%s: bad prompt / max length", who);
    c.K = b->num_beams; c.V = b->vocab; c.L = b->max_length; c.P = b->prompt_len; c.eos = b->eos; c.pad = b->pad;
    c.no_ts = b->no_timestamps; c.max_initial_ts = b->max_initial_ts; c.timestamps = b->timestamps;
    c.track = b->track_indices; c.length_penalty = b->length_penalty;
    return 0;
}

static State to_state(const tw_beam_state* s) {
    State o;
    o.hist = s->hist; o.fin = s->fin; o.run_score = s->run_score; o.fin_score = s->fin_score; o.fin_flag = s->fin_flag;
    o.fin_len = s->fin_len; o.gram = (Gram*)s->gram; o.improvable = s->improvable; o.hits_all = s->hits_all; o.ctrl = s->ctrl;
    return o;
}

extern "C" int32_t tw_beam_record_width(const tw_beam_config* b) { return b->track_indices ? 2 * b->max_length : b->max_length; }

extern "C" int tw_beam_step(const tw_beam_config* b, const tw_beam_state* state, const float* logits, void* row_state,
                            const uint32_t* suppress_bits, const uint32_t* begin_suppress_bits, float* cand_val,
                            int32_t* cand_tok, int32_t* tokens, int32_t tokens_ld, int32_t* block_table,
                            int32_t pages_per_row, int32_t bank_pages, void* kv_pool, int32_t n_pages, int32_t layers,
                            int32_t d_model, int32_t* copy_src, int32_t* copy_dst, int32_t* copy_len,
                            int32_t* origin_out, int32_t n_windows, void* stream) {
    Cfg c;
    if (int rc = to_cfg(b, c, "tw_beam_step")) return rc;
    TW_REQUIRE(state && logits && row_state && suppress_bits && begin_suppress_bits && cand_val && cand_tok && tokens &&
               block_table && kv_pool && copy_src && copy_dst && copy_len && origin_out, "tw_beam_step: null argument");
    if (tw::ensure_device(logits)) return 1;
    TW_REQUIRE(pages_per_row <= 8, "tw_beam_step: more than 8 pages per row");
    TW_REQUIRE(n_pages >= 2 * bank_pages, "tw_beam_step: the KV pool needs two banks of %d pages", bank_pages);
    TW_REQUIRE(d_model % 8 == 0, "tw_beam_step: d_model must be a multiple of 8");
    if (n_windows <= 0) return 0;
    const size_t smem = (size_t)c.V * sizeof(float);
    TW_REQUIRE(smem <= 220 * 1024, "tw_beam_step: vocabulary of %d does not fit the row buffer", c.V);
    static std::atomic<unsigned long long> attr_done{0};
    if (device_needs_setup(attr_done)) {
        TW_CUDA_CHECK(cudaFuncSetAttribute(beam_row_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        mark_device_done(attr_done);
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int R = n_windows * c.K;
    TopkParams tp;
    tp.logits = logits; tp.st = (const tw_row_state*)row_state; tp.run_score = state->run_score; tp.gram = (const Gram*)state->gram;
    tp.sup = suppress_bits; tp.bsup = begin_suppress_bits; tp.ctrl = state->ctrl; tp.cand_val = cand_val; tp.cand_tok = cand_tok;
    tp.c = c;
    beam_row_topk_kernel<<<R, TOPK_THREADS, smem, st>>>(tp);
    AdvanceParams ap;
    ap.s = to_state(state); ap.cand_val = cand_val; ap.cand_tok = cand_tok; ap.st = (tw_row_state*)row_state; ap.tokens = tokens;
    ap.tokens_ld = tokens_ld; ap.block_table = block_table; ap.ppr = pages_per_row; ap.bank_pages = bank_pages;
    ap.copy_src = copy_src; ap.copy_dst = copy_dst; ap.copy_len = copy_len; ap.origin_out = origin_out; ap.n = n_windows;
    ap.c = c;
    beam_advance_kernel<<<n_windows, 128, 0, st>>>(ap);
    CopyParams cp;
    cp.pool = (__nv_bfloat16*)kv_pool; cp.copy_src = copy_src; cp.copy_dst = copy_dst; cp.copy_len = copy_len;
    cp.ctrl = state->ctrl; cp.n_pages = n_pages; cp.D = d_model;
    beam_copy_pages_kernel<<<dim3(R, layers * 2), 256, 0, st>>>(cp);
    TW_CUDA_CHECK(cudaGetLastError());
    return 0;
}

// Host restatement of one search step on host buffers (same scalar code as the kernels; the per-row selection runs
// serially).  Test infrastructure for the CPU suite: no device is touched.
extern "C" int tw_beam_step_host(const tw_beam_config* b, const tw_beam_state* state, const float* logits, int32_t cur,
                                 const uint32_t* suppress_bits, const uint32_t* begin_suppress_bits, int32_t* next_tokens,
                                 int32_t* origin_out, int32_t n_windows) {
    Cfg c;
    if (int rc = to_cfg(b, c, "tw_beam_step_host")) return rc;
    TW_REQUIRE(state && logits && suppress_bits && begin_suppress_bits && next_tokens && origin_out,
               "tw_beam_step_host: null argument");
    State s = to_state(state);
    if (s.ctrl[1]) return 0;
    const int K = c.K, C = 2 * K, V = c.V, TB = c.no_ts + 1, R = n_windows * K;
    std::vector<float> cand_val((size_t)R * C), row(V);
    std::vector<int> cand_tok((size_t)R * C);
    const int n_gen = cur - c.P;
    for (int r = 0; r < R; ++r) {
        const float* x = logits + (size_t)r * V;
        float mx = -INFINITY;
        for (int v = 0; v < V; ++v) mx = fmaxf(mx, x[v]);
        double sum = 0.0;
        for (int v = 0; v < V; ++v) sum += exp((double)(x[v] - mx));
        const float lse = (float)log(sum);
        float mt = -INFINITY, ms = -INFINITY;
        for (int v = 0; v < V; ++v) {
            float lp = (x[v] - mx) - lse;
            if (!allowed(v, s.gram[r], n_gen, c, suppress_bits, begin_suppress_bits)) lp = -INFINITY;
            row[v] = lp;
            if (v >= TB) ms = fmaxf(ms, lp); else mt = fmaxf(mt, lp);
        }
        if (c.timestamps && ms > -INFINITY) {
            double ss = 0.0;
            for (int v = TB; v < V; ++v) ss += exp((double)(row[v] - ms));
            if (ms + (float)log(ss) > mt)
                for (int v = 0; v < TB; ++v) row[v] = -INFINITY;
        }
        for (int v = 0; v < V; ++v) row[v] += s.run_score[r];
        for (int k = 0; k < C; ++k) {
            int bi = -1;
            for (int v = 0; v < V; ++v)
                if (row[v] > -INFINITY && (bi < 0 || row[v] > row[bi])) bi = v;
            cand_val[(size_t)r * C + k] = bi < 0 ? -INFINITY : row[bi];
            cand_tok[(size_t)r * C + k] = bi < 0 ? 0 : bi;
            if (bi >= 0) row[bi] = -INFINITY;
        }
    }
    const int par = s.ctrl[0];
    bool any_improvable = false, all_hits = true;
    std::vector<Gram> old_gram(s.gram, s.gram + R);
    for (int w = 0; w < n_windows; ++w) {
        Plan p;
        plan_window(c, cur, cand_val.data() + (size_t)w * K * C, cand_tok.data() + (size_t)w * K * C, s.fin_score + w * K,
                    s.fin_flag + w * K, s.fin_len + w * K, s.improvable[w], p);
        apply_plan_rows(c, s, p, n_windows, w, cur, par, 0, 1);
        for (int i = 0; i < K; ++i) {
            const int cs = p.run_src[i], o = p.origin[cs];
            next_tokens[w * K + i] = p.tok[cs];
            origin_out[w * K + i] = w * K + o;
            s.gram[w * K + i] = gram_after(old_gram[w * K + o], n_gen, p.tok[cs], c);
            s.run_score[w * K + i] = p.run_score[i];
            s.fin_score[w * K + i] = p.fin_score[i];
            s.fin_flag[w * K + i] = p.fin_flag[i];
            s.fin_len[w * K + i] = p.fin_len[i];
        }
        s.improvable[w] = p.improvable;
        s.hits_all[w] = p.hits_all;
        any_improvable = any_improvable || p.improvable;
        all_hits = all_hits && p.hits_all;
    }
    s.ctrl[0] = par ^ 1;
    s.ctrl[4] += 1;
    if (!(any_improvable && !all_hits)) s.ctrl[1] = 1;
    return 0;
}
