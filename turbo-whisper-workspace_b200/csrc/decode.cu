// K7 / K8 — batched greedy decode step (SURVEY.md §8 a8-a10).  HBM-bound by design: every kernel
// streams weights or KV once with 16-byte loads and keeps all per-row state on the device, so one
// step is a fixed kernel sequence (CUDA-graph friendly; positions are read from device memory).
//
//   decode_embed_kernel   tok-embed + learned pos-embed -> fp32 residual stream
//                         ($TF/models/whisper/modeling_whisper.py:736-759)
//   skinny_gemm_kernel    out[b,n] = sum_k x[b,k] W[n,k] for B <= 32 rows: the weight is the M side
//                         of mma.sync.m16n8k16 (16 output features x 8 batch rows per instruction),
//                         K is split over the 8 warps of a CTA, fragments are loaded straight from
//                         global memory with a k-permutation that makes both operands 16-byte
//                         vector loads.  Epilogues: bias->bf16, QKV scatter into the paged
//                         self-attention KV cache, residual add (fp32, in place), GELU->bf16, and
//                         the LM head epilogue (Whisper logits processors + per-CTA arg-max /
//                         log-sum-exp partials).
//   decode_attn_kernel    one query per (row, head) against a key range: self-attention over the
//                         paged cache, cross-attention over the per-window encoder K/V with a
//                         split over the 1500 keys and a last-CTA-done combine.
//   decode_finalize_kernel  combines the LM-head partials, applies the timestamp probability
//                         rule, picks the token, handles forced tokens / finished rows and
//                         advances the per-row grammar state
//                         ($TF/generation/logits_process.py:1812-2043, $TF/generation/utils.py:2762-2797).
#include "common.cuh"
#include "twb200_internal.h"

namespace tw {
namespace dec {

constexpr int MAXB = 128;  // decode rows per launch (ln_part / ln_stats strides; engine.MAX_DECODE_BATCH <= this)
constexpr int PAGE = 64;  // positions per KV page

struct GrammarConst {
    int eos, pad, no_timestamps, ts_begin, vocab, lang_first, lang_last, max_initial_ts, begin_index;
};

// ------------------------------------------------------------------------------------------------
// embedding
// ------------------------------------------------------------------------------------------------
// also emits LayerNorm(x) (first decoder layer's self_attn_layer_norm) as bf16 when ln_out is given
__global__ void __launch_bounds__(256) decode_embed_kernel(const int* __restrict__ tokens, int tokens_ld,
                                                          const tw_row_state* __restrict__ st,
                                                          const __nv_bfloat16* __restrict__ tok_emb,
                                                          const float* __restrict__ pos_emb,
                                                          float* __restrict__ x, int D,
                                                          const float* __restrict__ ln_g,
                                                          const float* __restrict__ ln_b,
                                                          __nv_bfloat16* __restrict__ ln_out) {
    __shared__ float s_red[2][8];
    pdl_launch_dependents();
    pdl_wait();
    const int b = blockIdx.x;
    const int pos = st[b].pos;
    const int tok = tokens[b * tokens_ld + pos];
    float v[8];  // D <= 2048
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int c = threadIdx.x + i * 256;
        v[i] = 0.f;
        if (c < D) {
            v[i] = __bfloat162float(tok_emb[(size_t)tok * D + c]) + pos_emb[(size_t)pos * D + c];
            x[(size_t)b * D + c] = v[i];
            sum += v[i];
        }
    }
    if (!ln_out) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    sum = warp_sum(sum);
    if (lane == 0) s_red[0][warp] = sum;
    __syncthreads();
    float tot = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) tot += s_red[0][w];
    const float mean = tot / (float)D;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int c = threadIdx.x + i * 256;
        if (c < D) { const float d = v[i] - mean; q += d * d; }
    }
    q = warp_sum(q);
    if (lane == 0) s_red[1][warp] = q;
    __syncthreads();
    float qt = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) qt += s_red[1][w];
    const float rstd = rsqrtf(qt / (float)D + 1e-5f);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int c = threadIdx.x + i * 256;
        if (c < D) ln_out[(size_t)b * D + c] = __float2bfloat16((v[i] - mean) * rstd * ln_g[c] + ln_b[c]);
    }
}

// ------------------------------------------------------------------------------------------------
// skinny GEMM
// ------------------------------------------------------------------------------------------------
enum Epi { EPI_BF16 = 0, EPI_QKV = 1, EPI_RESID = 2, EPI_GELU_BF16 = 3, EPI_LOGITS = 4 };

struct SkinnyParams {
    const __nv_bfloat16* W;  // [N, K]
    const __nv_bfloat16* X;  // [B, ldx]
    int ldx;
    // EPI_RESID only: after the in-place residual update the last CTA to finish LayerNorms the updated
    // fp32 rows into ln_out (the operand of the next projection), so no LayerNorm launch is needed
    const float* ln_g;
    const float* ln_b;
    __nv_bfloat16* ln_out;       // [B, N] or null
    unsigned int* ln_counter;    // zero-initialised, self re-arming
    const float* bias;       // [N] or null
    int B, N, K;
    int chunk_grid;          // 1: blockIdx.y selects the row chunk (NB * 8 rows) — the chunks of a wide launch run as
                             // separate CTAs instead of a serial loop inside one CTA
    // LayerNorm folded into the consumer (round 2; removes the serial last-CTA LayerNorm tail of the producer):
    //   W (LN(x)) + b  =  rstd * (W' x - mean * c) + d,   W' = W diag(gamma), c = W' 1, d = W beta + b
    // Producer (EPI_RESID with ln_part_out): besides the fp32 update it stores bf16(x_new) into xb_out (the next
    // projection's operand) and (mean, M2) of its 16 values per row into ln_part_out[cta][row]; the LAST CTA to finish
    // combines the N / 16 partials of every row (two fixed-order warp reductions: deterministic) into (mean, rstd) —
    // a tail of a few hundred loads instead of a full LayerNorm over B x N values.  Consumer (LNF instantiations,
    // weights = W', bias = d): reads the B (mean, rstd) pairs and applies rstd / mean / c in its epilogue.
    float2* ln_part_out;         // [N/16][MAXB] scratch or null
    __nv_bfloat16* xb_out;       // [B, N]
    float2* ln_stats_out;        // [MAXB] (mean, rstd) per row, written by the producer's last CTA
    const float2* ln_stats_in;   // [MAXB] (consumer)
    const float* ln_c;           // [N]: row sums of the bf16 W'
    // EPI_BF16 / EPI_GELU_BF16
    __nv_bfloat16* out_bf16;
    int ldo;
    // EPI_RESID
    float* resid;            // [B, N] fp32, updated in place
    // EPI_QKV
    __nv_bfloat16* q_out;    // [B, D]
    __nv_bfloat16* kv_pool;  // layer base: [2][n_pages][PAGE][D]
    const int* block_table;  // [B, pages_per_row]
    int pages_per_row, n_pages, D;
    const tw_row_state* st;
    // EPI_LOGITS
    float* logits_out;       // optional raw logits [B, N]
    const uint32_t* suppress_bits;        // vocab bitmap
    const uint32_t* begin_suppress_bits;  // vocab bitmap
    GrammarConst gc;
    float* part_val;         // [B][n_ctas][3]  (max_text, max_ts, sumexp_ts)
    int* part_idx;           // [B][n_ctas][2]
};

// Decoder weights are stored FRAGMENT-MAJOR (packed once at load time, engine.pack_skinny_weight): for every slab of
// 16 output rows and every k-step of 32, the 32 lanes' A-fragments of mma.m16n8k16 are contiguous —
//   [slab][k-step][half: rows g | rows g+8][lane = g*4 + tg][8 bf16 = W[16*slab + g + 8*half][32*kstep + 8*tg ..]]
// so a warp's 16-byte-per-lane load covers 512 contiguous bytes (four full 128-byte lines) instead of sixteen 64-byte
// pieces 2*K bytes apart.  Rows beyond N are zero padding.
constexpr int FRAG_STEP = 512;   // elements per (slab, k-step) block
constexpr int FRAG_HALF = 256;   // offset of the rows g+8 half
TW_DEVINL const __nv_bfloat16* frag_ptr(const __nv_bfloat16* W, int K, int slab, int kstep, int lane) {
    return W + ((size_t)slab * (K >> 5) + kstep) * FRAG_STEP + lane * 8;
}
// `volatile`: a plain asm is a pure function to the compiler, which may then execute it speculatively ABOVE the
// condition that guards it (next-slab / next-round prefetches) — an out-of-range address that way is a real fault
// (seen as a layout-dependent illegal access when the weight buffer started a fresh memory segment).  The mma asm
// stays non-volatile, so only the loads keep their program order, which is the order they are written in anyway.
TW_DEVINL uint4 ldg_stream(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
TW_DEVINL void mma_bf16_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                              uint32_t b1) {
    asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
        "{%0, %1, %2, %3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

TW_DEVINL bool token_allowed(int v, const tw_row_state& s, const GrammarConst& gc, const uint32_t* sup,
                             const uint32_t* bsup) {
    if (s.mode & 1) return v >= gc.lang_first && v <= gc.lang_last;
    if (s.mode & 2) return !((sup[v >> 5] >> (v & 31)) & 1u) && !(s.begin && ((bsup[v >> 5] >> (v & 31)) & 1u));
    if ((sup[v >> 5] >> (v & 31)) & 1u) return false;
    if (s.begin && ((bsup[v >> 5] >> (v & 31)) & 1u)) return false;
    if (v == gc.no_timestamps) return false;
    if (v >= gc.ts_begin) return v >= s.ts_lo && v <= s.ts_hi;
    return v >= s.text_lo;
}

// One warp-row LayerNorm (fp32 two-pass statistics, eps 1e-5) of x[0..K) -> bf16; K <= 1280, K % 128 == 0.
// LOADCG: read through L2 (rows just written by other CTAs).
template <bool LOADCG>
TW_DEVINL void warp_layernorm_row(const float* __restrict__ x, const float* __restrict__ gamma,
                                  const float* __restrict__ beta, __nv_bfloat16* __restrict__ out, int K, int lane) {
    const int nvec = K >> 7;
    const float4* xr = reinterpret_cast<const float4*>(x);
    float4 v[10];
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < 10; ++i)
        if (i < nvec) {
            v[i] = LOADCG ? __ldcg(xr + lane + i * 32) : xr[lane + i * 32];
            sum += (v[i].x + v[i].y) + (v[i].z + v[i].w);
        }
    const float mean = warp_sum(sum) / (float)K;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 10; ++i)
        if (i < nvec) {
            const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
            q += (a * a + b * b) + (c * c + d * d);
        }
    const float rstd = rsqrtf(warp_sum(q) / (float)K + 1e-5f);
    uint2* dst = reinterpret_cast<uint2*>(out);
#pragma unroll
    for (int i = 0; i < 10; ++i)
        if (i < nvec) {
            const float4 ga = __ldg(reinterpret_cast<const float4*>(gamma) + lane + i * 32);
            const float4 be = __ldg(reinterpret_cast<const float4*>(beta) + lane + i * 32);
            uint2 pk;
            pk.x = pack_bf16x2((v[i].x - mean) * rstd * ga.x + be.x, (v[i].y - mean) * rstd * ga.y + be.y);
            pk.y = pack_bf16x2((v[i].z - mean) * rstd * ga.z + be.z, (v[i].w - mean) * rstd * ga.w + be.w);
            dst[lane + i * 32] = pk;
        }
}

template <int NB, int EPI, int WARPS, bool LNF = false>
__global__ void __launch_bounds__(WARPS * 32, (WARPS == 8) ? 2 : 1) skinny_gemm_kernel(const SkinnyParams p) {
    constexpr int NT = WARPS * 32;
    __shared__ float red[WARPS][NB * 8][17];
    __shared__ int s_last;
    __shared__ float s_mu[LNF ? MAXB : 1], s_rs[LNF ? MAXB : 1];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, tg = lane & 3;
    const int kw = p.K / WARPS;  // K per warp (multiple of 32)
    const int k_begin = warp * kw;
    const int steps = kw >> 5;
    constexpr int UN = 5;  // k-steps per round: their 16-byte fragment loads are all issued before the first mma

    const int n0 = blockIdx.x * 16;
    const int ra = min(n0 + g, p.N - 1), rb = min(n0 + g + 8, p.N - 1);
    // fragment-major weights (see frag_ptr): one 16-byte fragment per lane, 512 contiguous bytes per warp load
    const __nv_bfloat16* wa = frag_ptr(p.W, p.K, blockIdx.x, k_begin >> 5, lane);
    const __nv_bfloat16* wb = wa + FRAG_HALF;

    // the weights do not depend on the previous kernel: the first round of weight fragments is requested
    // before the programmatic-dependency wait, so the stream overlaps the predecessor's tail
    pdl_launch_dependents();
    uint4 alo[UN], ahi[UN];
#pragma unroll
    for (int u = 0; u < UN; ++u)
        if (u < steps) { alo[u] = ldg_stream(wa + u * FRAG_STEP); ahi[u] = ldg_stream(wb + u * FRAG_STEP); }
    pdl_wait();
    if (LNF && threadIdx.x < p.B) {     // (mean, rstd) of every row, left by the producer's last CTA
        const float2 st2 = __ldcg(p.ln_stats_in + threadIdx.x);
        s_mu[threadIdx.x] = st2.x;
        s_rs[threadIdx.x] = st2.y;
    }
    // Row chunks of NB * 8 decode rows: with more than 32 rows in a launch (several micro-batches decoded together) the
    // CTA's weight slab is streamed from DRAM ONCE — it stays in registers when K fits one round (K = 1280), later
    // chunks of a longer K re-read it from L2 — so the weight bytes per decode step do not grow with the rows.
    const int rb0 = p.chunk_grid ? blockIdx.y * NB * 8 : 0;
    const int rb1 = p.chunk_grid ? min(p.B, rb0 + NB * 8) : p.B;
    for (int rb = rb0; rb < rb1; rb += NB * 8) {
    if (rb > rb0) __syncthreads();      // `red` of the previous chunk has been consumed
    const __nv_bfloat16* xr[NB];
#pragma unroll
    for (int j = 0; j < NB; ++j) xr[j] = p.X + (size_t)min(rb + j * 8 + g, p.B - 1) * p.ldx + k_begin + tg * 8;
    float acc[NB][4];
#pragma unroll
    for (int j = 0; j < NB; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
    for (int s0 = 0; s0 < steps; s0 += UN) {
        uint4 xb[UN][NB];
#pragma unroll
        for (int u = 0; u < UN; ++u) {
            if (s0 + u < steps) {
                if (s0 > 0 || (rb > rb0 && steps > UN)) { alo[u] = ldg_stream(wa + (s0 + u) * FRAG_STEP); ahi[u] = ldg_stream(wb + (s0 + u) * FRAG_STEP); }
#pragma unroll
                for (int j = 0; j < NB; ++j) xb[u][j] = __ldg(reinterpret_cast<const uint4*>(xr[j] + (s0 + u) * 32));
            }
        }
#pragma unroll
        for (int u = 0; u < UN; ++u) {
            if (s0 + u < steps) {
#pragma unroll
                for (int j = 0; j < NB; ++j) {
                    mma_bf16_16816(acc[j], alo[u].x, ahi[u].x, alo[u].y, ahi[u].y, xb[u][j].x, xb[u][j].y);
                    mma_bf16_16816(acc[j], alo[u].z, ahi[u].z, alo[u].w, ahi[u].w, xb[u][j].z, xb[u][j].w);
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < NB; ++j) {
        red[warp][j * 8 + 2 * tg][g] = acc[j][0];
        red[warp][j * 8 + 2 * tg + 1][g] = acc[j][1];
        red[warp][j * 8 + 2 * tg][g + 8] = acc[j][2];
        red[warp][j * 8 + 2 * tg + 1][g + 8] = acc[j][3];
    }
    __syncthreads();

    for (int o = threadIdx.x; o < NB * 8 * 16; o += NT) {
        const int bl = o >> 4, rr = o & 15;     // row within the chunk / feature within the slab
        const int bb = rb + bl;                 // decode row
        const int n = n0 + rr;
        const bool live = bb < p.B && n < p.N;
        if (EPI == EPI_RESID && p.ln_part_out) {
            // producer of a folded LayerNorm: fp32 update, bf16 copy for the next projection, and (mean, M2) of the 16
            // values of row bb this CTA owns (one half-warp = one row; N % 16 == 0 here).  Whole warps run this branch.
            float x = 0.f;
            if (live) {
                float v = 0.f;
#pragma unroll
                for (int w = 0; w < WARPS; ++w) v += red[w][bl][rr];
                if (p.bias) v += p.bias[n];
                x = p.resid[(size_t)bb * p.N + n] + v;
                p.resid[(size_t)bb * p.N + n] = x;
                p.xb_out[(size_t)bb * p.N + n] = __float2bfloat16(x);
            }
            float sm = x;
#pragma unroll
            for (int d = 1; d < 16; d <<= 1) sm += __shfl_xor_sync(0xffffffffu, sm, d);
            const float mc = sm * (1.0f / 16.0f);
            float dq = (x - mc) * (x - mc);
#pragma unroll
            for (int d = 1; d < 16; d <<= 1) dq += __shfl_xor_sync(0xffffffffu, dq, d);
            if (live && rr == 0) p.ln_part_out[(size_t)blockIdx.x * MAXB + bb] = make_float2(mc, dq);
            continue;
        }
        if (!live) continue;
        float v = 0.f;
#pragma unroll
        for (int w = 0; w < WARPS; ++w) v += red[w][bl][rr];
        if (LNF) v = s_rs[bb] * (v - s_mu[bb] * p.ln_c[n]);
        if (p.bias) v += p.bias[n];
        if (EPI == EPI_BF16) {
            p.out_bf16[(size_t)bb * p.ldo + n] = __float2bfloat16(v);
        } else if (EPI == EPI_GELU_BF16) {
            p.out_bf16[(size_t)bb * p.ldo + n] = __float2bfloat16(gelu_erf(v));
        } else if (EPI == EPI_RESID) {
            p.resid[(size_t)bb * p.N + n] += v;
        } else if (EPI == EPI_QKV) {
            const int which = n / p.D, c = n - which * p.D;
            if (which == 0) {
                p.q_out[(size_t)bb * p.D + c] = __float2bfloat16(v);
            } else {
                const int pos = p.st[bb].pos;
                const int page = p.block_table[bb * p.pages_per_row + pos / PAGE];
                __nv_bfloat16* dst = p.kv_pool + ((size_t)(which - 1) * p.n_pages + page) * PAGE * p.D +
                                     (size_t)(pos % PAGE) * p.D + c;
                *dst = __float2bfloat16(v);
            }
        }
    }
    }   // row chunks
    if (EPI == EPI_RESID && p.ln_stats_out) {
        // last CTA: (mean, rstd) of every row from the N / 16 per-CTA partials.  All partials count 16 values, so
        // mean = avg(m_c) and M2 = sum(M2_c + 16 (m_c - mean)^2): two fixed-order warp reductions per row.
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) {
            const unsigned int prev = atomicAdd(p.ln_counter, 1u);
            s_last = (prev == gridDim.x * gridDim.y - 1);
            if (s_last) *p.ln_counter = 0;  // re-arm for the next launch
        }
        __syncthreads();
        if (s_last) {
            __threadfence();
            const int parts = gridDim.x;
            constexpr int RPW = (NB * 8 + WARPS - 1) / WARPS;
            constexpr int PPL = 3;           // partials per lane (N <= 1536)
            for (int rw = warp; rw < p.B; rw += WARPS * RPW) {     // one pass per row chunk
            float2 pr[RPW][PPL];
#pragma unroll
            for (int i = 0; i < RPW; ++i) {
                const int r = rw + i * WARPS;
#pragma unroll
                for (int t = 0; t < PPL; ++t) {
                    const int c = lane + 32 * t;
                    pr[i][t] = (r < p.B && c < parts) ? __ldcg(p.ln_part_out + (size_t)c * MAXB + r) : make_float2(0.f, 0.f);
                }
            }
            const float inv_parts = 1.0f / (float)parts;
#pragma unroll
            for (int i = 0; i < RPW; ++i) {
                const int r = rw + i * WARPS;
                const float mean = warp_sum((pr[i][0].x + pr[i][1].x) + pr[i][2].x) * inv_parts;
                float q = 0.f;
#pragma unroll
                for (int t = 0; t < PPL; ++t) {
                    const float d = pr[i][t].x - mean;
                    if (lane + 32 * t < parts) q += fmaf(16.0f * d, d, pr[i][t].y);
                }
                q = warp_sum(q);
                if (lane == 0 && r < p.B) p.ln_stats_out[r] = make_float2(mean, rsqrtf(q / (float)p.N + 1e-5f));
            }
            }
        }
    }
    if (EPI == EPI_RESID && p.ln_out) {
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) {
            const unsigned int prev = atomicAdd(p.ln_counter, 1u);
            s_last = (prev == gridDim.x * gridDim.y - 1);
            if (s_last) *p.ln_counter = 0;  // re-arm for the next launch
        }
        __syncthreads();
        if (s_last) {
            __threadfence();
            // (batching the rows of a warp, or 8 lanes per row, both measured slower than this simple form)
            for (int r = warp; r < p.B; r += WARPS)
                warp_layernorm_row<true>(p.resid + (size_t)r * p.N, p.ln_g, p.ln_b, p.ln_out + (size_t)r * p.N, p.N, lane);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// LM head: logits = x W^T over the tied embedding (51866 x 1280) + logits processors + partial arg-max /
// log-sum-exp.  Persistent grid, one 16-row slab per WARP and the full K per warp: no block-level
// synchronisation in the streaming loop, weight fragments double-buffered in registers (the next round of
// 16-byte loads is in flight while the current round's mma run).  The mma accumulator layout already has
// every (vocab row, batch row) logit in a known lane, so masks and reductions are warp shuffles.
// ------------------------------------------------------------------------------------------------
#ifndef LMH_WARPS_DEF
#define LMH_WARPS_DEF 8
#endif
constexpr int LMH_WARPS = LMH_WARPS_DEF;   // warps per CTA of the persistent LM-head grid (one CTA per SM)

template <int NB>
__global__ void __launch_bounds__(LMH_WARPS * 32, 1) lmhead_kernel(const SkinnyParams p) {
    // grammar state of the batch rows: shared memory, not 6 register copies per thread (the registers go to fragments)
    __shared__ tw_row_state s_st[MAXB];
    constexpr int UN = 4;  // k-steps (of 32) per round
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, tg = lane & 3;
    const int gwarp = blockIdx.x * LMH_WARPS + warp, nwarps = gridDim.x * LMH_WARPS;
    const int n_slabs = (p.N + 15) >> 4;
    const int rounds = p.K / (32 * UN);  // K % 128 == 0

    pdl_launch_dependents();
    // two named fragment buffers (no dynamically indexed arrays: those would live in local memory)
    uint4 a0lo[UN], a0hi[UN], a1lo[UN], a1hi[UN];
    if (gwarp < n_slabs) {  // round 0 of this warp's first slab: independent of the previous kernel
        const __nv_bfloat16* wa0 = frag_ptr(p.W, p.K, gwarp, 0, lane);
        const __nv_bfloat16* wb0 = wa0 + FRAG_HALF;
#pragma unroll
        for (int u = 0; u < UN; ++u) { a0lo[u] = ldg_stream(wa0 + u * FRAG_STEP); a0hi[u] = ldg_stream(wb0 + u * FRAG_STEP); }
    }
    pdl_wait();
    for (int i = threadIdx.x; i < p.B; i += LMH_WARPS * 32) s_st[i] = p.st[i];
    __syncthreads();
    // per-thread running partials for its 2*NB batch columns (j*8 + 2*tg + e)
    float bt[NB * 2], bs[NB * 2], sm[NB * 2];
    int it[NB * 2], is[NB * 2];
#pragma unroll
    for (int c = 0; c < NB * 2; ++c) {
        bt[c] = -INFINITY; bs[c] = -INFINITY; sm[c] = 0.f; it[c] = 0x7fffffff; is[c] = 0x7fffffff;
    }
    // rows in language-detection or no-timestamp mode rank EVERY id in the "text" class, timestamp slabs included
    bool flat = false;
    for (int i = lane; i < p.B; i += 32) flat = flat || (s_st[i].mode != 0);
    const bool any_flat = __any_sync(0xffffffffu, flat);
    const __nv_bfloat16* xr[NB];
#pragma unroll
    for (int j = 0; j < NB; ++j) xr[j] = p.X + (size_t)min(j * 8 + g, p.B - 1) * p.ldx + tg * 8;

    // Buffer 0 always holds the round about to be computed.  When a slab's last round sits in buffer 1 (even number
    // of rounds) buffer 0 receives round 0 of the warp's NEXT slab meanwhile, so the weight stream does not stop
    // while the logits of this slab are masked and reduced.
    bool have_first = true;   // buffer 0 already holds round 0 of the current slab
    for (int slab = gwarp; slab < n_slabs; slab += nwarps) {
        const int n0 = slab * 16;
        const __nv_bfloat16* wa = frag_ptr(p.W, p.K, slab, 0, lane);
        const __nv_bfloat16* wb = wa + FRAG_HALF;
        const int nslab = slab + nwarps;
        float acc[NB][4];
#pragma unroll
        for (int j = 0; j < NB; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
        if (!have_first) {
#pragma unroll
            for (int u = 0; u < UN; ++u) { a0lo[u] = ldg_stream(wa + u * FRAG_STEP); a0hi[u] = ldg_stream(wb + u * FRAG_STEP); }
        }
        have_first = false;
        auto compute = [&](const uint4 (&lo)[UN], const uint4 (&hi)[UN], int r) {
#pragma unroll
            for (int u = 0; u < UN; ++u) {
#pragma unroll
                for (int j = 0; j < NB; ++j) {
                    const uint4 xb = __ldg(reinterpret_cast<const uint4*>(xr[j] + (r * UN + u) * 32));
                    mma_bf16_16816(acc[j], lo[u].x, hi[u].x, lo[u].y, hi[u].y, xb.x, xb.y);
                    mma_bf16_16816(acc[j], lo[u].z, hi[u].z, lo[u].w, hi[u].w, xb.z, xb.w);
                }
            }
        };
        int r = 0;
        for (; r + 1 < rounds; r += 2) {
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                a1lo[u] = ldg_stream(wa + ((r + 1) * UN + u) * FRAG_STEP);
                a1hi[u] = ldg_stream(wb + ((r + 1) * UN + u) * FRAG_STEP);
            }
            compute(a0lo, a0hi, r);
            if (r + 2 < rounds) {
#pragma unroll
                for (int u = 0; u < UN; ++u) {
                    a0lo[u] = ldg_stream(wa + ((r + 2) * UN + u) * FRAG_STEP);
                    a0hi[u] = ldg_stream(wb + ((r + 2) * UN + u) * FRAG_STEP);
                }
            } else if (nslab < n_slabs) {
                const __nv_bfloat16* na = frag_ptr(p.W, p.K, nslab, 0, lane);
                const __nv_bfloat16* nb = na + FRAG_HALF;
#pragma unroll
                for (int u = 0; u < UN; ++u) { a0lo[u] = ldg_stream(na + u * FRAG_STEP); a0hi[u] = ldg_stream(nb + u * FRAG_STEP); }
                have_first = true;
            }
            compute(a1lo, a1hi, r + 1);
        }
        if (r < rounds) compute(a0lo, a0hi, r);   // odd number of rounds: the last one is in buffer 0
        // acc[j][e]: vocab row n0+g (e<2) / n0+g+8 (e>=2), batch row j*8 + 2*tg + (e&1)
        // Slab-level facts are warp-uniform: the 16 suppress bits of the slab come from one 32-bit word, and a slab
        // is all-text (99 % of them), all-timestamp or the single mixed one, so the unused reduction is skipped.
        const uint32_t sup16 = (p.suppress_bits[n0 >> 5] >> (n0 & 16)) & 0xffffu;
        const uint32_t bsup16 = (p.begin_suppress_bits[n0 >> 5] >> (n0 & 16)) & 0xffffu;
        const bool slab_has_text = n0 < p.gc.ts_begin || any_flat;
        const bool slab_has_ts = n0 + 16 > p.gc.ts_begin;
#pragma unroll
        for (int c = 0; c < NB * 2; ++c) {
            const int j = c >> 1, e = c & 1;
            const int bb = j * 8 + 2 * tg + e;
            const tw_row_state& rs = s_st[min(bb, p.B - 1)];
            float vt = -INFINITY, vs = -INFINITY;
            int jt = 0x7fffffff, js = 0x7fffffff;
            bool ts_ok[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int rr = g + 8 * h;
                const int n = n0 + rr;
                const float v = acc[j][e + 2 * h];
                ts_ok[h] = false;
                if (bb < p.B && n < p.N) {
                    if (p.logits_out) p.logits_out[(size_t)bb * p.N + n] = v;
                    bool ok;
                    if (rs.mode & 1) ok = n >= p.gc.lang_first && n <= p.gc.lang_last;
                    else if (rs.mode & 2) ok = !((sup16 >> rr) & 1u) && !(rs.begin && ((bsup16 >> rr) & 1u));
                    else ok = !((sup16 >> rr) & 1u) && !(rs.begin && ((bsup16 >> rr) & 1u)) && n != p.gc.no_timestamps &&
                              (n >= p.gc.ts_begin ? (n >= rs.ts_lo && n <= rs.ts_hi) : n >= rs.text_lo);
                    if (ok) {
                        if (n >= p.gc.ts_begin && rs.mode == 0) {
                            ts_ok[h] = true;
                            if (v > vs) { vs = v; js = n; }   // rows ascend with h: ties keep the lower id
                        } else if (v > vt) { vt = v; jt = n; }
                    }
                }
            }
            // reduce over the 8 lanes that share tg (vocab rows g = 0..7): xor 4, 8, 16
            if (slab_has_text) {
#pragma unroll
                for (int d = 4; d < 32; d <<= 1) {
                    const float ot = __shfl_xor_sync(0xffffffffu, vt, d);
                    const int oi = __shfl_xor_sync(0xffffffffu, jt, d);
                    if (ot > vt || (ot == vt && oi < jt)) { vt = ot; jt = oi; }
                }
                if (vt > bt[c] || (vt == bt[c] && jt < it[c])) { bt[c] = vt; it[c] = jt; }
            }
            if (slab_has_ts) {
                float ms = vs;
                int ks = js;
#pragma unroll
                for (int d = 4; d < 32; d <<= 1) {
                    const float os = __shfl_xor_sync(0xffffffffu, ms, d);
                    const int oj = __shfl_xor_sync(0xffffffffu, ks, d);
                    if (os > ms || (os == ms && oj < ks)) { ms = os; ks = oj; }
                }
                // sum of exp(ts logit - slab max) over this thread's (up to 2) timestamp entries, then over lanes
                float ex = (ts_ok[0] ? __expf(acc[j][e] - ms) : 0.f) + (ts_ok[1] ? __expf(acc[j][e + 2] - ms) : 0.f);
#pragma unroll
                for (int d = 4; d < 32; d <<= 1) ex += __shfl_xor_sync(0xffffffffu, ex, d);
                if (ms > -INFINITY) {
                    if (ms > bs[c]) {
                        sm[c] = (bs[c] > -INFINITY ? sm[c] * __expf(bs[c] - ms) : 0.f) + ex;
                        bs[c] = ms;
                        is[c] = ks;
                    } else {
                        sm[c] += ex * __expf(ms - bs[c]);
                        if (ms == bs[c] && ks < is[c]) is[c] = ks;
                    }
                }
            }
        }
    }
    // one partial per (batch row, warp): lanes g == 0 hold the reduced values of their 2*NB columns
    if (g == 0) {
#pragma unroll
        for (int c = 0; c < NB * 2; ++c) {
            const int bb = (c >> 1) * 8 + 2 * tg + (c & 1);
            if (bb < p.B) {
                const size_t o = (size_t)bb * nwarps + gwarp;
                p.part_val[o * 3 + 0] = bt[c];
                p.part_val[o * 3 + 1] = bs[c];
                p.part_val[o * 3 + 2] = sm[c];
                p.part_idx[o * 2 + 0] = it[c];
                p.part_idx[o * 2 + 1] = is[c];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// finalize: combine partials, choose the token, advance the grammar state
// ------------------------------------------------------------------------------------------------
struct FinalizeParams {
    const float* part_val;
    const int* part_idx;
    int n_parts;
    int* tokens;        // [B, tokens_ld]
    int tokens_ld;
    const int* forced;  // [B, tokens_ld]: forced[b][i] >= 0 overrides the token written at index i
    int* choices;       // optional [B, tokens_ld]: the engine's own pick before the forced override
    tw_row_state* st;
    GrammarConst gc;
    int max_len;        // generation stops writing at tokens_ld / max_length
};

__global__ void __launch_bounds__(128) decode_finalize_kernel(const FinalizeParams p) {
    __shared__ float s_text[128], s_ts[128], s_sum[128];
    __shared__ int s_itext[128], s_its[128];
    const int b = blockIdx.x, tid = threadIdx.x;
    pdl_launch_dependents();
    pdl_wait();
    float bt = -INFINITY, bs = -INFINITY, sm = 0.f;
    int it = 0x7fffffff, is = 0x7fffffff;
    for (int i = tid; i < p.n_parts; i += 128) {
        const size_t o = (size_t)b * p.n_parts + i;
        const float vt = p.part_val[o * 3 + 0], vs = p.part_val[o * 3 + 1], ss = p.part_val[o * 3 + 2];
        const int xt = p.part_idx[o * 2 + 0], xs = p.part_idx[o * 2 + 1];
        if (vt > bt || (vt == bt && xt < it)) { bt = vt; it = xt; }
        if (vs > -INFINITY) {
            if (vs > bs || (vs == bs && xs < is)) {
                sm = (bs > -INFINITY ? sm * __expf(bs - vs) : 0.f) + ss;
                bs = vs;
                is = xs;
            } else {
                sm += ss * __expf(vs - bs);
            }
        }
    }
    // combine the 128 per-thread partials: shuffles within each warp, then 4 warp results through smem
    auto merge = [&](float vt, int xt, float vs, int xs, float ss) {
        if (vt > bt || (vt == bt && xt < it)) { bt = vt; it = xt; }
        if (vs > -INFINITY) {
            if (vs > bs || (vs == bs && xs < is)) {
                sm = (bs > -INFINITY ? sm * __expf(bs - vs) : 0.f) + ss;
                bs = vs;
                is = xs;
            } else {
                sm += ss * __expf(vs - bs);
            }
        }
    };
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const float vt = __shfl_xor_sync(0xffffffffu, bt, d);
        const int xt = __shfl_xor_sync(0xffffffffu, it, d);
        const float vs = __shfl_xor_sync(0xffffffffu, bs, d);
        const int xs = __shfl_xor_sync(0xffffffffu, is, d);
        const float ss = __shfl_xor_sync(0xffffffffu, sm, d);
        merge(vt, xt, vs, xs, ss);
    }
    if ((tid & 31) == 0) {
        const int w = tid >> 5;
        s_text[w] = bt; s_ts[w] = bs; s_sum[w] = sm; s_itext[w] = it; s_its[w] = is;
    }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < 4; ++w) merge(s_text[w], s_itext[w], s_ts[w], s_its[w], s_sum[w]);
        tw_row_state s = p.st[b];
        const GrammarConst& gc = p.gc;
        int tok;
        if (s.mode != 0) {
            tok = it;  // language id arg-max / plain arg-max of the no-timestamp mode (every id is in the text class)
        } else {
            // sum of timestamp probability above every text token -> sample a timestamp
            // (log-softmax normaliser cancels on both sides of the comparison)
            const float lse_ts = (bs > -INFINITY) ? bs + logf(sm) : -INFINITY;
            if (lse_ts > bt) tok = is;
            else tok = (bs > bt) ? is : it;  // ties resolve to the lower (text) id, as torch.argmax
        }
        const int wi = s.pos + 1;  // index the new token is written to
        if (s.finished) tok = gc.pad;
        if (p.choices && wi < p.tokens_ld) p.choices[b * p.tokens_ld + wi] = tok;
        const int f = (wi < p.tokens_ld) ? p.forced[b * p.tokens_ld + wi] : -1;
        if (f >= 0) tok = f;
        if (wi < p.tokens_ld) p.tokens[b * p.tokens_ld + wi] = tok;

        // ---- advance the state for the step that will feed `tok` ----
        const int gen_before = wi - gc.begin_index;  // generated tokens before this one (may be < 0)
        if (gen_before >= 0 && tok == gc.eos) s.finished = 1;
        s.pos = wi;
        s.mode &= 2;   // language detection is over; the no-timestamp flag stays
        const int gen_now = gen_before + 1;  // generated tokens after appending tok
        if (gen_now <= 0) {
            // still inside the prompt: the next token is either forced or the first generated one
            s.last_ts = -1;
            s.begin = (gen_now == 0);
            s.text_lo = gc.ts_begin;  // first generated token must be a timestamp ...
            s.ts_lo = gc.ts_begin;
            s.ts_hi = gc.ts_begin + gc.max_initial_ts;  // ... no later than max_initial_timestamp
        } else {
            const int prev = (gen_now >= 2) ? p.tokens[b * p.tokens_ld + wi - 1] : -1;
            const bool last_is_ts = tok >= gc.ts_begin;
            const bool pen_is_ts = (gen_now < 2) || prev >= gc.ts_begin;
            if (last_is_ts) s.last_ts = tok;
            s.begin = 0;
            s.text_lo = 0;
            s.ts_lo = gc.ts_begin;
            s.ts_hi = gc.vocab - 1;
            if (last_is_ts) {
                if (pen_is_ts) s.ts_hi = gc.ts_begin - 1;  // timestamps forbidden
                else s.text_lo = gc.eos;                    // text below eos forbidden
            }
            if (s.last_ts >= 0) {
                const int bound = (last_is_ts && !pen_is_ts) ? s.last_ts : s.last_ts + 1;
                if (bound > s.ts_lo) s.ts_lo = bound;
            }
        }
        p.st[b] = s;
    }
}

// ------------------------------------------------------------------------------------------------
// decode attention: one query per (row, head); lane-per-key dot products, no shuffles in the loop
// ------------------------------------------------------------------------------------------------
struct AttnParams {
    const __nv_bfloat16* q;   // [B, D]
    __nv_bfloat16* out;       // [B, D]
    int D, H;
    int is_cross;
    // self: paged pool  [2][n_pages][PAGE][D] (layer base)
    const __nv_bfloat16* kv_pool;
    const int* block_table;
    int pages_per_row, n_pages;
    const tw_row_state* st;
    // cross: K row j of (row b, head h) at ck + b*batch_stride + h*head_stride + j*row_stride (elements)
    const __nv_bfloat16* ck;
    const __nv_bfloat16* cv;
    const int* enc_row;       // [B] row of the encoder batch this decode row reads (or null = b)
    long long row_stride, batch_stride, head_stride;
    int S, splits;
    float* part;              // [B][H][splits][66]
    unsigned int* counters;   // [B][H]
};

TW_DEVINL void bf16x8_to_f32(const uint4& u, float* f) {
    f[0] = __uint_as_float(u.x << 16); f[1] = __uint_as_float(u.x & 0xffff0000u);
    f[2] = __uint_as_float(u.y << 16); f[3] = __uint_as_float(u.y & 0xffff0000u);
    f[4] = __uint_as_float(u.z << 16); f[5] = __uint_as_float(u.z & 0xffff0000u);
    f[6] = __uint_as_float(u.w << 16); f[7] = __uint_as_float(u.w & 0xffff0000u);
}

constexpr int ATT_THREADS = 128;
constexpr int ATT_GROUPS = ATT_THREADS / 8;  // 8 lanes share one key row (8 x 16 B = one 128-byte line)
constexpr int ATT_KU = 4;                    // keys in flight per group
constexpr int ATT_MAXKEYS = 512;             // keys handled by one CTA (self: <= 448; cross: S / splits)

__global__ void __launch_bounds__(ATT_THREADS) decode_attn_kernel(const AttnParams p) {
    __shared__ float s_m[ATT_GROUPS], s_l[ATT_GROUPS];
    __shared__ float s_o[ATT_GROUPS][64];
    __shared__ int s_last;
    const int split = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    const int tid = threadIdx.x, grp = tid >> 3, l8 = tid & 7;
    pdl_launch_dependents();
    pdl_wait();

    int j0, j1;
    if (p.is_cross) {
        const int per = (p.S + p.splits - 1) / p.splits;
        j0 = split * per;
        j1 = min(p.S, j0 + per);
    } else {
        j0 = 0;
        j1 = p.st[b].pos + 1;
    }
    float q[8];
    bf16x8_to_f32(__ldg(reinterpret_cast<const uint4*>(p.q + (size_t)b * p.D + h * 64) + l8), q);

    const int eb = (p.is_cross && p.enc_row) ? p.enc_row[b] : b;
    auto row_ptr = [&](int j, int kv) -> const uint4* {
        const __nv_bfloat16* r;
        if (p.is_cross) {
            r = (kv ? p.cv : p.ck) + (size_t)eb * p.batch_stride + (size_t)h * p.head_stride + (size_t)j * p.row_stride;
        } else {
            const int page = p.block_table[b * p.pages_per_row + j / PAGE];
            r = p.kv_pool + ((size_t)kv * p.n_pages + page) * PAGE * p.D + (size_t)(j % PAGE) * p.D + h * 64;
        }
        return reinterpret_cast<const uint4*>(r) + l8;
    };

    float m = -INFINITY, l = 0.f, o[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = 0.f;

    // trip count is uniform over the CTA (the shuffles below need every lane of the warp); key slots past
    // j1 load a clamped row and are masked to -inf
    for (int base = j0; base < j1; base += ATT_GROUPS * ATT_KU) {
        const int jb = base + grp;
        uint4 kr[ATT_KU], vr[ATT_KU];
#pragma unroll
        for (int u = 0; u < ATT_KU; ++u) {
            const int j = min(jb + u * ATT_GROUPS, j1 - 1);
            kr[u] = p.is_cross ? ldg_stream(row_ptr(j, 0)) : *row_ptr(j, 0);
            vr[u] = p.is_cross ? ldg_stream(row_ptr(j, 1)) : *row_ptr(j, 1);
        }
        float sc[ATT_KU];
        float mx = m;
#pragma unroll
        for (int u = 0; u < ATT_KU; ++u) {
            float f[8];
            bf16x8_to_f32(kr[u], f);
            float d = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) d = fmaf(q[i], f[i], d);
            d += __shfl_xor_sync(0xffffffffu, d, 1);
            d += __shfl_xor_sync(0xffffffffu, d, 2);
            d += __shfl_xor_sync(0xffffffffu, d, 4);
            sc[u] = (jb + u * ATT_GROUPS < j1) ? d : -INFINITY;
            mx = fmaxf(mx, sc[u]);
        }
        if (mx == -INFINITY) continue;  // this group has no valid key in the round (no shuffles below)
        const float alpha = (m == -INFINITY) ? 0.f : __expf(m - mx);
        l *= alpha;
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] *= alpha;
#pragma unroll
        for (int u = 0; u < ATT_KU; ++u) {
            const float pj = __expf(sc[u] - mx);  // exp(-inf) = 0 for the padded slots
            l += pj;
            float f[8];
            bf16x8_to_f32(vr[u], f);
#pragma unroll
            for (int i = 0; i < 8; ++i) o[i] = fmaf(pj, f[i], o[i]);
        }
        m = mx;
    }
    if (l8 == 0) { s_m[grp] = m; s_l[grp] = l; }
#pragma unroll
    for (int i = 0; i < 8; ++i) s_o[grp][l8 * 8 + i] = o[i];
    __syncthreads();

    float M = -INFINITY, L = 0.f, O = 0.f;
    if (tid < 64) {
#pragma unroll
        for (int g = 0; g < ATT_GROUPS; ++g) M = fmaxf(M, s_m[g]);
#pragma unroll
        for (int g = 0; g < ATT_GROUPS; ++g) {
            const float w = (s_m[g] == -INFINITY) ? 0.f : __expf(s_m[g] - M);
            L = fmaf(s_l[g], w, L);
            O = fmaf(s_o[g][tid], w, O);
        }
    }
    if (!p.is_cross || p.splits == 1) {
        if (tid < 64) p.out[(size_t)b * p.D + h * 64 + tid] = __float2bfloat16(O / L);
        return;
    }
    // split-K: publish (max, sum, o[64]); the last CTA of this (row, head) combines in split order
    float* my = p.part + (((size_t)b * p.H + h) * p.splits + split) * 66;
    if (tid < 64) my[2 + tid] = O;
    if (tid == 0) { my[0] = M; my[1] = L; }
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const unsigned int prev = atomicAdd(&p.counters[b * p.H + h], 1u);
        s_last = (prev == (unsigned)p.splits - 1);
        if (s_last) p.counters[b * p.H + h] = 0;  // re-arm for the next launch
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    if (tid < 64) {
        const float* base = p.part + ((size_t)b * p.H + h) * p.splits * 66;
        float Mg = -INFINITY;
        for (int s = 0; s < p.splits; ++s) Mg = fmaxf(Mg, __ldcg(base + s * 66));
        float Lg = 0.f, Og = 0.f;
        for (int s = 0; s < p.splits; ++s) {
            const float w = __expf(__ldcg(base + s * 66) - Mg);
            Lg = fmaf(__ldcg(base + s * 66 + 1), w, Lg);
            Og = fmaf(__ldcg(base + s * 66 + 2 + tid), w, Og);
        }
        p.out[(size_t)b * p.D + h * 64 + tid] = __float2bfloat16(Og / Lg);
    }
}

}  // namespace dec
}  // namespace tw

// ================================================================================================
// C ABI
// ================================================================================================
using namespace tw;
using namespace tw::dec;

static int g_use_pdl = 0;  // off by default: inside CUDA graphs plain edges measured faster (212 vs 220 ms / 447 steps); eager stepping gains 10 % with it
extern "C" int tw_set_pdl(int32_t enabled) { g_use_pdl = enabled ? 1 : 0; return 0; }
// wide launches (> 32 decode rows): 0 (default) = serial loop over the 24-row chunks inside one CTA, weights in registers;
// TWB200_SKINNY_CHUNK_GRID=1 = the chunks run as separate CTAs (grid.y).  Measured (profiles/r2x_bench_ab.jsonl): the
// grid form shortens a 96-row step of ONE context (1.21 vs 1.31 ms) but loses 3 % in the five-context bench, where
// CTA residency, not latency, is what the contexts compete for
// TWB200_SKINNY_CHUNK_GRID=2 = grid form only for the launches that leave SMs idle (N / 16 <= 96 CTAs: the N = 1280 projections):
// -8 % per 96-row step alone, no difference in the bench (profiles/r2x3_bench_ab_selective_chunk_grid.jsonl)
static int g_chunk_grid = [] { const char* e = getenv("TWB200_SKINNY_CHUNK_GRID"); return e ? atoi(e) : 0; }();
static int g_cross_stream = [] { const char* e = getenv("TWB200_CROSS_ATTN"); return (e && !strcmp(e, "stream")) ? 1 : 0; }();
extern "C" int tw_set_cross_attn_stream(int32_t enabled) { g_cross_stream = enabled ? 1 : 0; return 0; }

// launch with the programmatic-stream-serialization attribute (the kernel's own griddepcontrol.wait orders it
// after its predecessor); captured into CUDA graphs as a programmatic dependency edge
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = g_use_pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, args...);
}

static_assert(sizeof(tw_row_state) == 32, "tw_row_state layout is part of the ABI (8 x int32)");

template <int EPI, int WARPS, bool LNF = false>
static int launch_nb(const SkinnyParams& p, int grid, cudaStream_t st) {
    // rows per chunk: up to 32 rows one chunk of ceil(B / 8) groups; beyond that chunks of 24 rows (NB = 3: no spills)
    const int nb = p.B <= 32 ? (p.B + 7) / 8 : 3;
    SkinnyParams q = p;
    q.chunk_grid = ((g_chunk_grid == 1 || (g_chunk_grid == 2 && grid <= 96)) && p.B > nb * 8) ? 1 : 0;
    const dim3 g3(grid, q.chunk_grid ? (p.B + nb * 8 - 1) / (nb * 8) : 1);
    switch (nb) {
        case 1: TW_CUDA_CHECK(launch_pdl(skinny_gemm_kernel<1, EPI, WARPS, LNF>, g3, dim3(WARPS * 32), 0, st, q)); break;
        case 2: TW_CUDA_CHECK(launch_pdl(skinny_gemm_kernel<2, EPI, WARPS, LNF>, g3, dim3(WARPS * 32), 0, st, q)); break;
        case 3: TW_CUDA_CHECK(launch_pdl(skinny_gemm_kernel<3, EPI, WARPS, LNF>, g3, dim3(WARPS * 32), 0, st, q)); break;
        case 4: TW_CUDA_CHECK(launch_pdl(skinny_gemm_kernel<4, EPI, WARPS, LNF>, g3, dim3(WARPS * 32), 0, st, q)); break;
        default: set_error("skinny gemm: batch %d > %d", p.B, MAXB); return 2;
    }
    TW_CUDA_CHECK(cudaGetLastError());
    return 0;
}

// the 16-warp K split is used for the long-K residual projection (fc2)
template <int EPI>
static int launch_skinny(const SkinnyParams& p, cudaStream_t st) {
    const int grid = (p.N + 15) / 16;
    if (EPI == EPI_RESID) {
        if (p.K >= 4096 && p.K % 512 == 0) return launch_nb<EPI_RESID, 16>(p, grid, st);
        return launch_nb<EPI_RESID, 8>(p, grid, st);
    }
    if (p.ln_stats_in) return launch_nb<EPI, 8, true>(p, grid, st);   // consumer of a folded LayerNorm
    return launch_nb<EPI, 8>(p, grid, st);
}

extern "C" int tw_dec_embed(const int32_t* tokens, int32_t tokens_ld, const void* row_state, const void* tok_emb_bf16,
                            const float* pos_emb, float* x, int32_t batch, int32_t d_model, const float* ln_gamma,
                            const float* ln_beta, void* ln_out_bf16, void* stream) {
    TW_REQUIRE(tokens && row_state && tok_emb_bf16 && pos_emb && x, "tw_dec_embed: null argument");
    if (tw::ensure_device(x)) return 1;
    TW_REQUIRE(d_model <= 2048, "tw_dec_embed: d_model %d > 2048", d_model);
    TW_REQUIRE(!ln_out_bf16 || (ln_gamma && ln_beta), "tw_dec_embed: LayerNorm output needs gamma and beta");
    if (batch <= 0) return 0;
    TW_CUDA_CHECK(launch_pdl(decode_embed_kernel, dim3(batch), dim3(256), 0, (cudaStream_t)stream, tokens, (int)tokens_ld,
                             (const tw_row_state*)row_state, (const __nv_bfloat16*)tok_emb_bf16, pos_emb, x, (int)d_model,
                             ln_gamma, ln_beta, (__nv_bfloat16*)ln_out_bf16));
    TW_CUDA_CHECK(cudaGetLastError());
    return 0;
}

static int check_skinny(const tw_skinny_args* a, const char* who) {
    TW_REQUIRE(a && a->w && a->x, "%s: null argument", who);
    if (tw::ensure_device(a->w)) return 1;
    TW_REQUIRE(a->batch >= 1 && a->batch <= MAXB, "%s: batch %d not in [1,%d]", who, a->batch, MAXB);
    TW_REQUIRE(a->k % 256 == 0, "%s: K (%d) must be a multiple of 256", who, a->k);
    TW_REQUIRE(a->ldx % 8 == 0 && ((uintptr_t)a->x & 15) == 0 && ((uintptr_t)a->w & 15) == 0, "%s: alignment", who);
    TW_REQUIRE(a->n > 0, "%s: bad N", who);
    if (a->ln_stats_in) TW_REQUIRE(a->ln_c, "%s: a folded LayerNorm needs the W' row sums", who);
    return 0;
}

static void fill_common(SkinnyParams& p, const tw_skinny_args* a) {
    p = SkinnyParams{};
    p.W = (const __nv_bfloat16*)a->w;
    p.X = (const __nv_bfloat16*)a->x;
    p.ldx = a->ldx;
    p.bias = a->bias;
    p.B = a->batch;
    p.N = a->n;
    p.K = a->k;
    if (a->ln_stats_in) {     // consumer of a folded LayerNorm (weights = W diag(gamma), bias = W beta + b)
        p.ln_stats_in = (const float2*)a->ln_stats_in;
        p.ln_c = a->ln_c;
    }
}

extern "C" int tw_dec_linear(const tw_skinny_args* a, int32_t epilogue, void* out, int32_t ldo, void* stream) {
    if (int rc = check_skinny(a, "tw_dec_linear")) return rc;
    TW_REQUIRE(out, "tw_dec_linear: null out");
    SkinnyParams p;
    fill_common(p, a);
    if (epilogue == 0) { p.out_bf16 = (__nv_bfloat16*)out; p.ldo = ldo; return launch_skinny<EPI_BF16>(p, (cudaStream_t)stream); }
    if (epilogue == 3) { p.out_bf16 = (__nv_bfloat16*)out; p.ldo = ldo; return launch_skinny<EPI_GELU_BF16>(p, (cudaStream_t)stream); }
    if (epilogue == 2) {
        p.resid = (float*)out;
        TW_REQUIRE(!a->ln_stats_in, "tw_dec_linear: the residual epilogue cannot consume a folded LayerNorm");
        if (a->ln_part_out) {
            TW_REQUIRE(a->x_bf16_out && a->ln_stats_out && a->ln_counter && a->n % 16 == 0 && a->n <= 1536,
                       "tw_dec_linear: a folded-LayerNorm producer needs x_bf16_out, ln_stats_out, ln_counter, n %% 16 == 0, n <= 1536");
            p.ln_part_out = (float2*)a->ln_part_out;
            p.xb_out = (__nv_bfloat16*)a->x_bf16_out;
            p.ln_stats_out = (float2*)a->ln_stats_out;
            p.ln_counter = a->ln_counter;
        }
        if (a->ln_out_bf16) {
            TW_REQUIRE(a->ln_gamma && a->ln_beta && a->ln_counter, "tw_dec_linear: fused LayerNorm needs gamma, beta, counter");
            TW_REQUIRE(a->n <= 1280 && a->n % 128 == 0, "tw_dec_linear: fused LayerNorm supports n <= 1280, n %% 128 == 0");
            p.ln_g = a->ln_gamma; p.ln_b = a->ln_beta; p.ln_out = (__nv_bfloat16*)a->ln_out_bf16; p.ln_counter = a->ln_counter;
        }
        return launch_skinny<EPI_RESID>(p, (cudaStream_t)stream);
    }
    set_error("tw_dec_linear: unknown epilogue %d", epilogue);
    return 2;
}

extern "C" int tw_dec_qkv(const tw_skinny_args* a, void* q_out_bf16, void* kv_pool_layer, const int32_t* block_table,
                          int32_t pages_per_row, int32_t n_pages, const void* row_state, void* stream) {
    if (int rc = check_skinny(a, "tw_dec_qkv")) return rc;
    TW_REQUIRE(q_out_bf16 && kv_pool_layer && block_table && row_state, "tw_dec_qkv: null argument");
    TW_REQUIRE(a->n % 3 == 0, "tw_dec_qkv: N must be 3*D");
    SkinnyParams p;
    fill_common(p, a);
    p.q_out = (__nv_bfloat16*)q_out_bf16;
    p.kv_pool = (__nv_bfloat16*)kv_pool_layer;
    p.block_table = block_table;
    p.pages_per_row = pages_per_row;
    p.n_pages = n_pages;
    p.D = a->n / 3;
    p.st = (const tw_row_state*)row_state;
    return launch_skinny<EPI_QKV>(p, (cudaStream_t)stream);
}

static GrammarConst to_gc(const tw_grammar* g) {
    GrammarConst gc;
    gc.eos = g->eos; gc.pad = g->pad; gc.no_timestamps = g->no_timestamps; gc.ts_begin = g->ts_begin;
    gc.vocab = g->vocab; gc.lang_first = g->lang_first; gc.lang_last = g->lang_last;
    gc.max_initial_ts = g->max_initial_ts; gc.begin_index = g->begin_index;
    return gc;
}

// number of partial records per batch row = warps of the persistent LM-head grid (one CTA per SM)
static int lmhead_grid() { int n = num_sms(); return n > 0 ? n : 148; }
extern "C" int32_t tw_dec_max_rows(void) { return MAXB; }
extern "C" int32_t tw_dec_lmhead_parts(int32_t vocab) {
    (void)vocab;
    return lmhead_grid() * LMH_WARPS;
}

extern "C" int tw_dec_lmhead(const tw_skinny_args* a, const tw_grammar* g, const void* row_state,
                             const uint32_t* suppress_bits, const uint32_t* begin_suppress_bits, float* part_val,
                             int32_t* part_idx, float* logits_out, void* stream) {
    if (int rc = check_skinny(a, "tw_dec_lmhead")) return rc;
    TW_REQUIRE(g && row_state && suppress_bits && begin_suppress_bits && part_val && part_idx, "tw_dec_lmhead: null argument");
    TW_REQUIRE(a->n == g->vocab, "tw_dec_lmhead: N (%d) != vocab (%d)", a->n, g->vocab);
    SkinnyParams p;
    fill_common(p, a);
    p.st = (const tw_row_state*)row_state;
    p.suppress_bits = suppress_bits;
    p.begin_suppress_bits = begin_suppress_bits;
    p.gc = to_gc(g);
    p.part_val = part_val;
    p.part_idx = part_idx;
    p.logits_out = logits_out;
    const int grid = lmhead_grid();
    cudaStream_t st = (cudaStream_t)stream;
    switch ((p.B + 7) / 8) {
        case 1: TW_CUDA_CHECK(launch_pdl(lmhead_kernel<1>, dim3(grid), dim3(LMH_WARPS * 32), 0, st, p)); break;
        case 2: TW_CUDA_CHECK(launch_pdl(lmhead_kernel<2>, dim3(grid), dim3(LMH_WARPS * 32), 0, st, p)); break;
        case 3: TW_CUDA_CHECK(launch_pdl(lmhead_kernel<3>, dim3(grid), dim3(LMH_WARPS * 32), 0, st, p)); break;
        case 4: TW_CUDA_CHECK(launch_pdl(lmhead_kernel<4>, dim3(grid), dim3(LMH_WARPS * 32), 0, st, p)); break;
        case 5: TW_CUDA_CHECK(launch_pdl(lmhead_kernel<5>, dim3(grid), dim3(LMH_WARPS * 32), 0, st, p)); break;
        case 6: TW_CUDA_CHECK(launch_pdl(lmhead_kernel<6>, dim3(grid), dim3(LMH_WARPS * 32), 0, st, p)); break;
        default: set_error("tw_dec_lmhead: batch %d > 48", p.B); return 2;
    }
    TW_CUDA_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int tw_dec_finalize(const float* part_val, const int32_t* part_idx, int32_t n_parts, int32_t* tokens,
                               int32_t tokens_ld, const int32_t* forced, int32_t* choices, void* row_state,
                               const tw_grammar* g, int32_t batch, void* stream) {
    TW_REQUIRE(part_val && part_idx && tokens && forced && row_state && g, "tw_dec_finalize: null argument");
    if (tw::ensure_device(tokens)) return 1;
    if (batch <= 0) return 0;
    FinalizeParams p;
    p.part_val = part_val; p.part_idx = part_idx; p.n_parts = n_parts; p.tokens = tokens; p.tokens_ld = tokens_ld;
    p.forced = forced; p.choices = choices; p.st = (tw_row_state*)row_state; p.gc = to_gc(g); p.max_len = tokens_ld;
    TW_CUDA_CHECK(launch_pdl(decode_finalize_kernel, dim3(batch), dim3(128), 0, (cudaStream_t)stream, p));
    TW_CUDA_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int tw_dec_self_attn(const void* q_bf16, void* out_bf16, const void* kv_pool_layer, const int32_t* block_table,
                                int32_t pages_per_row, int32_t n_pages, const void* row_state, int32_t batch,
                                int32_t heads, void* stream) {
    TW_REQUIRE(q_bf16 && out_bf16 && kv_pool_layer && block_table && row_state, "tw_dec_self_attn: null argument");
    if (tw::ensure_device(q_bf16)) return 1;
    TW_REQUIRE(pages_per_row * PAGE <= ATT_MAXKEYS, "tw_dec_self_attn: more than %d positions", ATT_MAXKEYS);
    if (batch <= 0) return 0;
    AttnParams p{};
    p.q = (const __nv_bfloat16*)q_bf16; p.out = (__nv_bfloat16*)out_bf16; p.D = heads * 64; p.H = heads;
    p.is_cross = 0; p.kv_pool = (const __nv_bfloat16*)kv_pool_layer; p.block_table = block_table;
    p.pages_per_row = pages_per_row; p.n_pages = n_pages; p.st = (const tw_row_state*)row_state; p.splits = 1;
    TW_CUDA_CHECK(launch_pdl(decode_attn_kernel, dim3(1, heads, batch), dim3(ATT_THREADS), 0, (cudaStream_t)stream, p));
    TW_CUDA_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int tw_dec_cross_attn(const void* q_bf16, void* out_bf16, const void* k_bf16, const void* v_bf16,
                                 int64_t kv_row_stride, int64_t kv_batch_stride, int64_t kv_head_stride,
                                 const int32_t* enc_row, int32_t src_len, int32_t batch, int32_t heads,
                                 int32_t splits, float* part, uint32_t* counters, void* stream) {
    TW_REQUIRE(q_bf16 && out_bf16 && k_bf16 && v_bf16, "tw_dec_cross_attn: null argument");
    if (tw::ensure_device(q_bf16)) return 1;
    TW_REQUIRE(splits >= 1, "tw_dec_cross_attn: splits %d < 1", splits);
    TW_REQUIRE(splits == 1 || (part && counters), "tw_dec_cross_attn: split needs scratch");
    TW_REQUIRE(kv_row_stride % 8 == 0 && kv_batch_stride % 8 == 0 && kv_head_stride % 8 == 0,
               "tw_dec_cross_attn: K/V strides must be multiples of 8 elements");
    if (batch <= 0) return 0;
    // opt-in (tw_set_cross_attn_stream / TWB200_CROSS_ATTN=stream): the persistent TMA-fed streaming kernel of
    // cross_attn.cu; `splits` is then the capacity of `part` and the kernel balances the split count itself.  Measured
    // on B200 (profiles/r2u_cross_probe.jsonl, r2v_bench_ab.jsonl): 4 % faster than the kernel below at >= 72 rows
    // (6.6-6.7 TB/s), 12-20 % slower at <= 24 rows, no difference in the five-context bench — so it is not the default
    if (g_cross_stream) {
        const int rc = tw::cross_attn_stream_launch(q_bf16, out_bf16, k_bf16, v_bf16, kv_row_stride, kv_batch_stride,
                                                    kv_head_stride, enc_row, src_len, batch, heads, splits, part, counters,
                                                    (cudaStream_t)stream, g_use_pdl != 0);
        if (rc >= 0) return rc;
    }
    TW_REQUIRE((src_len + splits - 1) / splits <= ATT_MAXKEYS,
               "tw_dec_cross_attn: %d keys / %d splits exceeds %d per CTA", src_len, splits, ATT_MAXKEYS);
    AttnParams p{};
    p.q = (const __nv_bfloat16*)q_bf16; p.out = (__nv_bfloat16*)out_bf16; p.D = heads * 64; p.H = heads;
    p.is_cross = 1; p.ck = (const __nv_bfloat16*)k_bf16; p.cv = (const __nv_bfloat16*)v_bf16;
    p.row_stride = kv_row_stride; p.batch_stride = kv_batch_stride; p.head_stride = kv_head_stride;
    p.enc_row = enc_row; p.S = src_len; p.splits = splits; p.part = part; p.counters = counters;
    TW_CUDA_CHECK(launch_pdl(decode_attn_kernel, dim3(splits, heads, batch), dim3(ATT_THREADS), 0, (cudaStream_t)stream, p));
    TW_CUDA_CHECK(cudaGetLastError());
    return 0;
}
