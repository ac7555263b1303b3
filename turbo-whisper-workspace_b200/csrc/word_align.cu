// Word-level timestamps, device side (SURVEY.md §8f rank 4): the alignment-head cross-attention tap of the decode
// step and the normalise / median-filter / head-mean stage of WhisperGenerationMixin._extract_token_timestamps
// ($TF/models/whisper/generation_whisper.py:241-381).  HBM-bound byte work: the tap re-reads one head's K block
// (src_len x 64 bf16, contiguous in the engine's head-major layout) per (row, alignment head) and writes src_len
// fp32 probabilities; the matrix stage streams the tapped probabilities twice.
//
// HF keeps `cross_attentions` of every decode step (eager attention: softmax(q k^T) per head), stacks the
// (layer, head) pairs of generation_config.alignment_heads, crops to num_frames // 2 encoder positions, drops the
// prompt positions, standardises every (head, frame) column over the token axis (population std), median-filters
// along the frame axis (width config.median_filter_width, reflect padding), averages the heads and runs dynamic
// time warping on the negated matrix.  The DTW itself is host code (csrc/dtw.cpp).
#include "common.cuh"
#include "twb200_internal.h"

#include <cuda_bf16.h>

namespace tw {
namespace align {

constexpr int TAP_THREADS = 256;
constexpr int TAP_MAXKEYS = 2048;   // scores of one (row, head) staged in shared memory

struct TapParams {
    const __nv_bfloat16* q;      // [batch, q_ld], head h at columns 64h..64h+63 (already scaled by head_dim^-0.5)
    const __nv_bfloat16* k;      // this layer's K, element (row, head, j, e) at k + row*bs + head*hs + j*rs + e
    long long rs, bs, hs;
    const int* enc_row;          // decode row -> encoder-batch row
    const tw_row_state* row_state;  // [batch]
    const int* heads;            // device int32 [n_heads]: head index of every alignment slot of this layer
    int slot0, n_slots, max_len, src_len, q_ld;
    float* probs;                // [batch][n_slots][max_len][src_len]
};

__device__ __forceinline__ float block_max(float v, float* red) {
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) red[w] = v;
    __syncthreads();
    float r = red[0];
    for (int i = 1; i < TAP_THREADS / 32; ++i) r = fmaxf(r, red[i]);
    return r;
}

__device__ __forceinline__ float block_sum(float v, float* red) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) red[w] = v;
    __syncthreads();
    float r = 0.f;
    for (int i = 0; i < TAP_THREADS / 32; ++i) r += red[i];
    return r;
}

// grid (alignment heads of this layer, batch); one CTA = softmax(q_h . K_h^T) over src_len positions
__global__ void __launch_bounds__(TAP_THREADS) align_tap_kernel(const TapParams p) {
    __shared__ float qs[64];
    __shared__ float sc[TAP_MAXKEYS];
    __shared__ float red[TAP_THREADS / 32];
    const int b = blockIdx.y, slot = blockIdx.x;
    const int h = p.heads[slot];
    const int pos = p.row_state[b].pos;
    if (pos < 0 || pos >= p.max_len) return;    // uniform per CTA
    if (threadIdx.x < 64) qs[threadIdx.x] = __bfloat162float(p.q[(long long)b * p.q_ld + h * 64 + threadIdx.x]);
    __syncthreads();
    const __nv_bfloat16* kb = p.k + (long long)p.enc_row[b] * p.bs + (long long)h * p.hs;
    float mx = -INFINITY;
    for (int j = threadIdx.x; j < p.src_len; j += TAP_THREADS) {
        const uint4* kr = reinterpret_cast<const uint4*>(kb + (long long)j * p.rs);
        float acc = 0.f;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const uint4 v = kr[c];
            const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float2 f = __bfloat1622float2(h2[e]);
                acc = fmaf(qs[c * 8 + 2 * e], f.x, acc);
                acc = fmaf(qs[c * 8 + 2 * e + 1], f.y, acc);
            }
        }
        sc[j] = acc;
        mx = fmaxf(mx, acc);
    }
    mx = block_max(mx, red);
    float sum = 0.f;
    for (int j = threadIdx.x; j < p.src_len; j += TAP_THREADS) {
        const float e = expf(sc[j] - mx);
        sc[j] = e;
        sum += e;
    }
    sum = block_sum(sum, red);
    float* out = p.probs + (((long long)b * p.n_slots + p.slot0 + slot) * p.max_len + pos) * p.src_len;
    for (int j = threadIdx.x; j < p.src_len; j += TAP_THREADS) out[j] = sc[j] / sum;
}

// ---- column statistics: mean and population std over the token axis for every (row, slot, frame) -------------
struct MatrixParams {
    const float* probs;          // [batch][n_slots][max_len][src_len]
    const int* n_frames;         // device int32 [batch]: frames kept per row (num_frames // 2), <= src_len
    int n_slots, max_len, src_len, t0, n_tok, width;
    float* stats;                // [batch][n_slots][src_len][2] = (mean, std)
    float* matrix;               // [batch][max_len][src_len]; row t - t0 of decode row b at (b*max_len + t - t0)*src_len
};

__global__ void __launch_bounds__(128) align_stats_kernel(const MatrixParams p) {
    const int b = blockIdx.z, s = blockIdx.y;
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= p.n_frames[b]) return;
    const float* col = p.probs + (((long long)b * p.n_slots + s) * p.max_len + p.t0) * p.src_len + f;
    // two-pass in double: the result is the correctly rounded fp32 statistic for any summation order
    double sum = 0.0;
    for (int t = 0; t < p.n_tok; ++t) sum += (double)col[(long long)t * p.src_len];
    const double mean = sum / p.n_tok;
    double var = 0.0;
    for (int t = 0; t < p.n_tok; ++t) {
        const double d = (double)col[(long long)t * p.src_len] - mean;
        var += d * d;
    }
    float* st = p.stats + (((long long)b * p.n_slots + s) * p.src_len + f) * 2;
    st[0] = (float)mean;
    st[1] = (float)sqrt(var / p.n_tok);
}

// one thread per (row, token, frame): median over the reflect-padded window of the standardised column values,
// averaged over the alignment slots
constexpr int MAX_WIDTH = 15;
__global__ void __launch_bounds__(128) align_matrix_kernel(const MatrixParams p) {
    const int b = blockIdx.z, t = blockIdx.y;
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    const int F = p.n_frames[b];
    if (f >= F) return;
    const int half = p.width / 2;
    float acc = 0.f;
    for (int s = 0; s < p.n_slots; ++s) {
        const float* row = p.probs + (((long long)b * p.n_slots + s) * p.max_len + p.t0 + t) * p.src_len;
        const float* st = p.stats + (((long long)b * p.n_slots + s) * p.src_len) * 2;
        float med;
        if (F <= half) {   // _median_filter returns its input when the axis is not longer than the padding
            med = (row[f] - st[2 * f]) / st[2 * f + 1];
        } else {
            float w[MAX_WIDTH];
#pragma unroll
            for (int i = 0; i < MAX_WIDTH; ++i) {
                if (i < p.width) {
                    int g = f - half + i;
                    if (g < 0) g = -g;                       // reflect (no edge repeat)
                    if (g >= F) g = 2 * (F - 1) - g;
                    w[i] = (row[g] - st[2 * g]) / st[2 * g + 1];
                } else {
                    w[i] = INFINITY;
                }
            }
            // rank selection of the (half)-th smallest (ties ordered by index), static indexing only
            med = w[0];
#pragma unroll
            for (int i = 0; i < MAX_WIDTH; ++i) {
                if (i < p.width) {
                    int r = 0;
#pragma unroll
                    for (int j = 0; j < MAX_WIDTH; ++j)
                        if (j < p.width) r += (w[j] < w[i] || (w[j] == w[i] && j < i)) ? 1 : 0;
                    if (r == half) med = w[i];
                }
            }
        }
        acc += med;
    }
    p.matrix[((long long)b * p.max_len + t) * p.src_len + f] = acc / (float)p.n_slots;
}

}  // namespace align
}  // namespace tw

using namespace tw;
using namespace tw::align;

extern "C" int tw_dec_align_tap(const void* q_bf16, int32_t q_ld, const void* k_bf16, int64_t kv_row_stride,
                                int64_t kv_batch_stride, int64_t kv_head_stride, const int32_t* enc_row,
                                const void* row_state, const int32_t* heads_dev, int32_t n_heads, int32_t slot0,
                                int32_t n_slots, int32_t max_len, int32_t src_len, int32_t batch, float* probs,
                                void* stream) {
    TW_REQUIRE(q_bf16 && k_bf16 && enc_row && row_state && heads_dev && probs, "tw_dec_align_tap: null argument");
    TW_REQUIRE(batch >= 1 && batch <= 65535 && n_heads >= 1 && slot0 >= 0 && slot0 + n_heads <= n_slots,
               "tw_dec_align_tap: bad batch / slot range");
    TW_REQUIRE(src_len >= 1 && src_len <= TAP_MAXKEYS, "tw_dec_align_tap: src_len %d exceeds %d", src_len, TAP_MAXKEYS);
    TW_REQUIRE(kv_row_stride % 8 == 0 && kv_batch_stride % 8 == 0 && kv_head_stride % 8 == 0 && q_ld % 8 == 0,
               "tw_dec_align_tap: strides must be multiples of 8 elements");
    if (tw::ensure_device(q_bf16)) return 1;
    TapParams p;
    p.q = (const __nv_bfloat16*)q_bf16;
    p.k = (const __nv_bfloat16*)k_bf16;
    p.rs = kv_row_stride; p.bs = kv_batch_stride; p.hs = kv_head_stride;
    p.enc_row = enc_row; p.row_state = (const tw_row_state*)row_state; p.heads = heads_dev;
    p.slot0 = slot0; p.n_slots = n_slots; p.max_len = max_len; p.src_len = src_len; p.q_ld = q_ld;
    p.probs = probs;
    align_tap_kernel<<<dim3(n_heads, batch), TAP_THREADS, 0, (cudaStream_t)stream>>>(p);
    TW_CUDA_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int tw_align_matrix(const float* probs, const int32_t* n_frames_dev, int32_t batch, int32_t n_slots,
                               int32_t max_len, int32_t src_len, int32_t t0, int32_t n_tok, int32_t filter_width,
                               float* stats, float* matrix, void* stream) {
    TW_REQUIRE(probs && n_frames_dev && stats && matrix, "tw_align_matrix: null argument");
    TW_REQUIRE(batch >= 1 && batch <= 65535 && n_slots >= 1 && n_slots <= 65535, "tw_align_matrix: bad batch / slots");
    TW_REQUIRE(t0 >= 0 && n_tok >= 1 && t0 + n_tok <= max_len && n_tok <= 65535, "tw_align_matrix: bad token range");
    TW_REQUIRE(filter_width >= 1 && filter_width % 2 == 1 && filter_width <= MAX_WIDTH,
               "tw_align_matrix: median filter width must be odd and <= %d", MAX_WIDTH);
    if (tw::ensure_device(probs)) return 1;
    MatrixParams p;
    p.probs = probs; p.n_frames = n_frames_dev; p.n_slots = n_slots; p.max_len = max_len; p.src_len = src_len;
    p.t0 = t0; p.n_tok = n_tok; p.width = filter_width; p.stats = stats; p.matrix = matrix;
    const int fx = (src_len + 127) / 128;
    align_stats_kernel<<<dim3(fx, n_slots, batch), 128, 0, (cudaStream_t)stream>>>(p);
    TW_CUDA_CHECK(cudaGetLastError());
    align_matrix_kernel<<<dim3(fx, n_tok, batch), 128, 0, (cudaStream_t)stream>>>(p);
    TW_CUDA_CHECK(cudaGetLastError());
    return 0;
}
