// Decoder prefill: all positions of a text prompt (generate(prompt_ids=...)) of R decode rows in one pass, instead of
// one decode step per prompt token.  The projections are tw_gemm_bf16 launches over M = R x (P - 1) rows (engine.py,
// WhisperEngine.prefill); this file holds the rest of the decoder layer for those rows:
//
//   prefill_embed_kernel      x[r, t] = tok_emb[tokens[r, t]] + dec_pos[t]            (fp32 residual stream)
//   prefill_kv_store_kernel   K / V of every prompt position -> the paged self-attention cache, in the layout the
//                             decode step's q|k|v epilogue writes (csrc/decode.cu, EPI_QKV)
//   prefill_attn_kernel       flash attention on mma.sync m16n8k16 (bf16 in, fp32 softmax statistics):
//                             causal self-attention over the prompt, or cross-attention over a window's 1500
//                             encoder positions (head-major K / V, rows mapped to windows by enc_row)
//
// $TF/models/whisper/modeling_whisper.py:449-506 (WhisperDecoderLayer), :736-759 (embeddings).
#include "common.cuh"
#include "twb200_internal.h"

namespace tw {
namespace prefill {

constexpr int PAGE = 64;       // positions per KV page (csrc/decode.cu)
constexpr int QT = 64;         // queries per CTA: 4 warps x 16 rows
constexpr int KT = 64;         // keys per tile
constexpr int LDS = 72;        // smem row stride in elements (144 B: conflict-free fragment loads, 16-B aligned rows)
constexpr int THREADS = 128;

__global__ void __launch_bounds__(256) prefill_embed_kernel(const int* __restrict__ tokens, int tokens_ld, int T,
                                                            const __nv_bfloat16* __restrict__ tok_emb,
                                                            const float* __restrict__ pos_emb, float* __restrict__ x,
                                                            int D) {
    const int t = blockIdx.x, r = blockIdx.y;
    const int tok = tokens[(size_t)r * tokens_ld + t];
    float* xr = x + ((size_t)r * T + t) * D;
    for (int c = threadIdx.x; c < D; c += blockDim.x)
        xr[c] = __bfloat162float(tok_emb[(size_t)tok * D + c]) + pos_emb[(size_t)t * D + c];
}

// one thread per 16-byte chunk of K or V
__global__ void __launch_bounds__(256) prefill_kv_store_kernel(const __nv_bfloat16* __restrict__ qkv, int T, int D,
                                                               __nv_bfloat16* __restrict__ kv_pool,
                                                               const int* __restrict__ block_table, int pages_per_row,
                                                               int n_pages, long long total) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int chunks = D / 8;
    const int c8 = (int)(i % chunks);
    const long long rest = i / chunks;
    const int which = (int)(rest % 2);           // 0: K, 1: V
    const long long m = rest / 2;                // prompt row r * T + t
    const int r = (int)(m / T), t = (int)(m % T);
    const int page = block_table[r * pages_per_row + t / PAGE];
    const uint4 v = *reinterpret_cast<const uint4*>(qkv + (size_t)m * 3 * D + (size_t)(which + 1) * D + c8 * 8);
    *reinterpret_cast<uint4*>(kv_pool + (((size_t)which * n_pages + page) * PAGE + t % PAGE) * D + c8 * 8) = v;
}

struct AttnParams {
    const __nv_bfloat16* q;        // query of (row r, position t) at q + (r * T + t) * q_ld + h * 64
    long long q_ld;
    const __nv_bfloat16* k;        // key j of (row r, head h) at k + kr * kv_batch_stride + h * kv_head_stride + j * kv_row_stride
    const __nv_bfloat16* v;        //   (kr = enc_row[r] when given, else r); V likewise
    long long kv_row_stride, kv_batch_stride, kv_head_stride;
    const int* enc_row;
    int n_keys;                    // keys per (row, head); causal: key j is visible to query t iff j <= t
    __nv_bfloat16* out;            // (r, t) at out + (r * T + t) * out_ld + h * 64
    long long out_ld;
    int T;
};

TW_DEVINL void cp_async16(void* smem, const void* gmem) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
TW_DEVINL void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
TW_DEVINL void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

TW_DEVINL void mma_bf16(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
                 "{%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

TW_DEVINL void ldmatrix_x4_trans(uint32_t* r, const void* smem) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(smem_u32(smem)));
}

// grid (ceil(T / 64), heads, rows); 4 warps, warp w owns queries q0 + 16w .. +15
template <bool CAUSAL>
__global__ void __launch_bounds__(THREADS) prefill_attn_kernel(const AttnParams p) {
    __shared__ __align__(16) __nv_bfloat16 sK[2][KT][LDS];
    __shared__ __align__(16) __nv_bfloat16 sV[2][KT][LDS];
    const int q0 = blockIdx.x * QT, h = blockIdx.y, r = blockIdx.z;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, tg = lane & 3;
    const int kr = p.enc_row ? p.enc_row[r] : r;
    const __nv_bfloat16* kb = p.k + (size_t)kr * p.kv_batch_stride + (size_t)h * p.kv_head_stride;
    const __nv_bfloat16* vb = p.v + (size_t)kr * p.kv_batch_stride + (size_t)h * p.kv_head_stride;
    const int n_keys = CAUSAL ? min(p.n_keys, q0 + QT) : p.n_keys;
    const int n_tiles = (n_keys + KT - 1) / KT;

    // tile loader: 64 keys x 64 dims of K and V = 2 x 512 chunks of 16 B, 8 per thread; rows past n_keys repeat the
    // last key (their scores are masked)
    auto load_tile = [&](int tile, int buf) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int c = tid + i * THREADS;         // 0..511
            const int row = c >> 3, col = (c & 7) * 8;
            const int j = min(tile * KT + row, n_keys - 1);
            cp_async16(&sK[buf][row][col], kb + (size_t)j * p.kv_row_stride + col);
            cp_async16(&sV[buf][row][col], vb + (size_t)j * p.kv_row_stride + col);
        }
        cp_async_commit();
    };
    load_tile(0, 0);

    // Q fragments (A operand, 16 queries x 64 dims) straight from global memory; rows past T repeat the last query
    const int qa = min(q0 + warp * 16 + g, p.T - 1), qb = min(q0 + warp * 16 + g + 8, p.T - 1);
    const __nv_bfloat16* qra = p.q + ((size_t)r * p.T + qa) * p.q_ld + h * 64;
    const __nv_bfloat16* qrb = p.q + ((size_t)r * p.T + qb) * p.q_ld + h * 64;
    uint32_t qf[4][4];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
        qf[kk][0] = *reinterpret_cast<const uint32_t*>(qra + kk * 16 + 2 * tg);
        qf[kk][1] = *reinterpret_cast<const uint32_t*>(qrb + kk * 16 + 2 * tg);
        qf[kk][2] = *reinterpret_cast<const uint32_t*>(qra + kk * 16 + 8 + 2 * tg);
        qf[kk][3] = *reinterpret_cast<const uint32_t*>(qrb + kk * 16 + 8 + 2 * tg);
    }
    const int ta = q0 + warp * 16 + g, tb = ta + 8;   // this thread's two query positions

    constexpr float LOG2E = 1.4426950408889634f;
    float m[2] = {-INFINITY, -INFINITY}, l[2] = {0.f, 0.f};
    float o[8][4];
#pragma unroll
    for (int n = 0; n < 8; ++n) o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f;

    for (int tile = 0; tile < n_tiles; ++tile) {
        const int buf = tile & 1;
        if (tile + 1 < n_tiles) {
            load_tile(tile + 1, buf ^ 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        // S = Q K^T: 16 queries x 64 keys per warp (8 n-tiles of 8 keys)
        float s[8][4];
#pragma unroll
        for (int n = 0; n < 8; ++n) {
            s[n][0] = s[n][1] = s[n][2] = s[n][3] = 0.f;
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const uint32_t b0 = *reinterpret_cast<const uint32_t*>(&sK[buf][n * 8 + g][kk * 16 + 2 * tg]);
                const uint32_t b1 = *reinterpret_cast<const uint32_t*>(&sK[buf][n * 8 + g][kk * 16 + 8 + 2 * tg]);
                mma_bf16(s[n], qf[kk], b0, b1);
            }
        }
        // mask, then the online softmax (base 2) of rows g (ta) and g + 8 (tb)
        float mx[2] = {m[0], m[1]};
#pragma unroll
        for (int n = 0; n < 8; ++n) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int j = tile * KT + n * 8 + 2 * tg + (e & 1);
                const int t = (e < 2) ? ta : tb;
                const bool ok = j < n_keys && (!CAUSAL || j <= t);
                s[n][e] = ok ? s[n][e] * LOG2E : -INFINITY;
                mx[e >> 1] = fmaxf(mx[e >> 1], s[n][e]);
            }
        }
        float alpha[2];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            mx[i] = fmaxf(mx[i], __shfl_xor_sync(0xffffffffu, mx[i], 1));
            mx[i] = fmaxf(mx[i], __shfl_xor_sync(0xffffffffu, mx[i], 2));
            // a row with no visible key yet (only possible for padding rows) keeps m = -inf: use 0 as the reference
            const float ref = (mx[i] == -INFINITY) ? 0.f : mx[i];
            alpha[i] = exp2f(m[i] - ref);      // exp2(-inf) = 0 on the first tile
            m[i] = mx[i];
            mx[i] = ref;
            l[i] *= alpha[i];
        }
        uint32_t pf[4][4];      // P as the A operand of P V: k-chunk kc = keys 16 kc .. 16 kc + 15
#pragma unroll
        for (int n = 0; n < 8; ++n) {
            const float p0 = exp2f(s[n][0] - mx[0]), p1 = exp2f(s[n][1] - mx[0]);
            const float p2 = exp2f(s[n][2] - mx[1]), p3 = exp2f(s[n][3] - mx[1]);
            l[0] += p0 + p1;
            l[1] += p2 + p3;
            pf[n >> 1][(n & 1) * 2 + 0] = pack_bf16x2(p0, p1);
            pf[n >> 1][(n & 1) * 2 + 1] = pack_bf16x2(p2, p3);
        }
#pragma unroll
        for (int n = 0; n < 8; ++n) {
            o[n][0] *= alpha[0]; o[n][1] *= alpha[0];
            o[n][2] *= alpha[1]; o[n][3] *= alpha[1];
        }
        // O += P V; V B-fragments by ldmatrix.trans: matrices (keys +0 / +8) x (dims 8 n / 8 n + 8)
#pragma unroll
        for (int kc = 0; kc < 4; ++kc) {
#pragma unroll
            for (int n = 0; n < 8; n += 2) {
                const int mi = lane >> 3, rr = lane & 7;
                uint32_t b[4];
                ldmatrix_x4_trans(b, &sV[buf][kc * 16 + (mi & 1) * 8 + rr][n * 8 + (mi >> 1) * 8]);
                mma_bf16(o[n], pf[kc], b[0], b[1]);
                mma_bf16(o[n + 1], pf[kc], b[2], b[3]);
            }
        }
        __syncthreads();    // the buffer is refilled by the next iteration's prefetch
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        l[i] += __shfl_xor_sync(0xffffffffu, l[i], 1);
        l[i] += __shfl_xor_sync(0xffffffffu, l[i], 2);
    }
    const float ia = 1.f / l[0], ib = 1.f / l[1];
    __nv_bfloat16* oa = p.out + ((size_t)r * p.T + ta) * p.out_ld + h * 64;
    __nv_bfloat16* ob = p.out + ((size_t)r * p.T + tb) * p.out_ld + h * 64;
#pragma unroll
    for (int n = 0; n < 8; ++n) {
        if (ta < p.T) *reinterpret_cast<uint32_t*>(oa + n * 8 + 2 * tg) = pack_bf16x2(o[n][0] * ia, o[n][1] * ia);
        if (tb < p.T) *reinterpret_cast<uint32_t*>(ob + n * 8 + 2 * tg) = pack_bf16x2(o[n][2] * ib, o[n][3] * ib);
    }
}

}  // namespace prefill
}  // namespace tw

// ================================================================================================
// C ABI
// ================================================================================================
using namespace tw;
using namespace tw::prefill;

static bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

extern "C" int tw_prefill_embed(const int32_t* tokens, int32_t tokens_ld, int32_t rows, int32_t n_pos,
                                const void* tok_emb_bf16, const float* pos_emb, float* x, int32_t d_model,
                                void* stream) {
    TW_REQUIRE(tokens && tok_emb_bf16 && pos_emb && x, "tw_prefill_embed: null argument");
    if (tw::ensure_device(x)) return 1;
    TW_REQUIRE(rows >= 0 && n_pos >= 0 && d_model > 0 && tokens_ld >= n_pos, "tw_prefill_embed: bad shape");
    if (rows == 0 || n_pos == 0) return 0;
    prefill_embed_kernel<<<dim3(n_pos, rows), 256, 0, (cudaStream_t)stream>>>(
        tokens, tokens_ld, n_pos, (const __nv_bfloat16*)tok_emb_bf16, pos_emb, x, d_model);
    TW_CUDA_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int tw_prefill_kv_store(const void* qkv_bf16, int32_t rows, int32_t n_pos, int32_t d_model,
                                   void* kv_pool_layer, const int32_t* block_table, int32_t pages_per_row,
                                   int32_t n_pages, void* stream) {
    TW_REQUIRE(qkv_bf16 && kv_pool_layer && block_table, "tw_prefill_kv_store: null argument");
    if (tw::ensure_device(qkv_bf16)) return 1;
    TW_REQUIRE(d_model > 0 && d_model % 8 == 0, "tw_prefill_kv_store: d_model (%d) must be a multiple of 8", d_model);
    TW_REQUIRE(rows >= 0 && n_pos >= 0 && n_pos <= pages_per_row * PAGE,
               "tw_prefill_kv_store: %d positions do not fit %d pages per row", n_pos, pages_per_row);
    TW_REQUIRE(aligned16(qkv_bf16) && aligned16(kv_pool_layer), "tw_prefill_kv_store: pointers must be 16-byte aligned");
    const long long total = (long long)rows * n_pos * 2 * (d_model / 8);
    if (total == 0) return 0;
    prefill_kv_store_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)qkv_bf16, n_pos, d_model, (__nv_bfloat16*)kv_pool_layer, block_table, pages_per_row,
        n_pages, total);
    TW_CUDA_CHECK(cudaGetLastError());
    return 0;
}

static int launch_attn(const AttnParams& p, bool causal, int rows, int heads, cudaStream_t st, const char* what) {
    TW_REQUIRE(p.q && p.k && p.v && p.out, "%s: null argument", what);
    if (tw::ensure_device(p.out)) return 1;
    TW_REQUIRE(rows >= 0 && heads > 0 && p.T >= 0 && p.n_keys > 0, "%s: bad shape", what);
    TW_REQUIRE(p.q_ld % 8 == 0 && p.out_ld % 8 == 0 && p.kv_row_stride % 8 == 0 && p.kv_batch_stride % 8 == 0 &&
                   p.kv_head_stride % 8 == 0,
               "%s: strides must be multiples of 8 elements", what);
    TW_REQUIRE(aligned16(p.q) && aligned16(p.k) && aligned16(p.v) && aligned16(p.out),
               "%s: pointers must be 16-byte aligned", what);
    if (rows == 0 || p.T == 0) return 0;
    const dim3 grid((p.T + QT - 1) / QT, heads, rows);
    if (causal) prefill_attn_kernel<true><<<grid, THREADS, 0, st>>>(p);
    else prefill_attn_kernel<false><<<grid, THREADS, 0, st>>>(p);
    TW_CUDA_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int tw_prefill_self_attn(const void* qkv_bf16, void* out_bf16, int32_t rows, int32_t n_pos, int32_t heads,
                                    void* stream) {
    AttnParams p = {};
    const long long D = (long long)heads * 64, ld = 3 * D;
    p.q = (const __nv_bfloat16*)qkv_bf16;
    p.q_ld = ld;
    p.k = p.q ? p.q + D : nullptr;
    p.v = p.q ? p.q + 2 * D : nullptr;
    p.kv_row_stride = ld;
    p.kv_batch_stride = (long long)n_pos * ld;
    p.kv_head_stride = 64;
    p.enc_row = nullptr;
    p.n_keys = n_pos;
    p.out = (__nv_bfloat16*)out_bf16;
    p.out_ld = D;
    p.T = n_pos;
    TW_REQUIRE(n_pos <= 448, "tw_prefill_self_attn: %d positions > 448", n_pos);
    return launch_attn(p, true, rows, heads, (cudaStream_t)stream, "tw_prefill_self_attn");
}

extern "C" int tw_prefill_cross_attn(const void* q_bf16, int64_t q_ld, void* out_bf16, const void* k_bf16,
                                     const void* v_bf16, int64_t kv_row_stride, int64_t kv_batch_stride,
                                     int64_t kv_head_stride, const int32_t* enc_row, int32_t src_len, int32_t rows,
                                     int32_t n_pos, int32_t heads, void* stream) {
    AttnParams p = {};
    p.q = (const __nv_bfloat16*)q_bf16;
    p.q_ld = q_ld;
    p.k = (const __nv_bfloat16*)k_bf16;
    p.v = (const __nv_bfloat16*)v_bf16;
    p.kv_row_stride = kv_row_stride;
    p.kv_batch_stride = kv_batch_stride;
    p.kv_head_stride = kv_head_stride;
    p.enc_row = enc_row;
    p.n_keys = src_len;
    p.out = (__nv_bfloat16*)out_bf16;
    p.out_ld = (long long)heads * 64;
    p.T = n_pos;
    return launch_attn(p, false, rows, heads, (cudaStream_t)stream, "tw_prefill_cross_attn");
}
