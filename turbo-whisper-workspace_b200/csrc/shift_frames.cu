// Seek-shifted window gather for the seek loops
// (WhisperGenerationMixin._get_input_segment, $TF/models/whisper/generation_whisper.py:1831-1850):
// the next 30 s window of a row starts at mel frame seek[b] and is zero-padded (feature value 0)
// to 3000 frames.  Operates on the time-major bf16 feature layout [*, rows, cols].  The short-form loop
// (tw_shift_frames) reads the rows' own 3000-frame windows of one batch buffer; the long-form loop
// (tw_gather_frames) reads each row's window out of the whole-clip features of that row's clip.
// dst_row_off skips the leading conv-padding row of the encoder input, which stays zero.
#include "common.cuh"
#include "twb200_internal.h"

namespace tw {
// dst[b, dst_row_off + t] = row b's source frame seek[b] + t for t < min(window, frames_b - seek[b]), zeros up to window.
// Row b's source frame f lives at (src_rows ? src_rows[b] : src + src_row[b] * src_batch_stride) + (src_row_off + f) * cols;
// frames_b = frames ? frames[b] : n_frames.  One launch serves every row of a seek iteration whatever its source.
__global__ void __launch_bounds__(256) shift_frames_kernel(const uint4* __restrict__ src,
                                                          const uint4* const* __restrict__ src_rows,
                                                          const int* __restrict__ src_row, long long src_batch_stride_vec,
                                                          int src_row_off, const int* __restrict__ frames, int n_frames,
                                                          const int* __restrict__ seek, int window, int vec_per_row,
                                                          uint4* __restrict__ dst, long long dst_batch_stride_vec,
                                                          int dst_row_off) {
    const int b = blockIdx.y;
    const uint4* s = src_rows ? src_rows[b] : src + (long long)(src_row ? src_row[b] : b) * src_batch_stride_vec;
    s += (long long)src_row_off * vec_per_row;
    const int sk = seek[b];
    const int avail = (frames ? frames[b] : n_frames) - sk;
    uint4* d = dst + (long long)b * dst_batch_stride_vec + (long long)dst_row_off * vec_per_row;
    const int total = window * vec_per_row;      // < 2^31: checked on the host; the stride is kept in 64 bits
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const int t = (int)i / vec_per_row, c = (int)i % vec_per_row;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (t < avail) v = s[(long long)(sk + t) * vec_per_row + c];
        d[i] = v;
    }
}
}  // namespace tw

extern "C" int tw_shift_frames(const void* src_bf16, void* dst_bf16, const int32_t* src_row, const int32_t* seek,
                               int32_t batch, int32_t frames, int32_t cols, int64_t batch_stride, int32_t row_off,
                               void* stream) {
    using namespace tw;
    TW_REQUIRE(src_bf16 && dst_bf16 && seek, "tw_shift_frames: null argument");
    if (tw::ensure_device(src_bf16)) return 1;
    TW_REQUIRE(cols % 8 == 0 && batch_stride % 8 == 0, "tw_shift_frames: cols and batch_stride must be multiples of 8");
    TW_REQUIRE(src_bf16 != dst_bf16, "tw_shift_frames: in-place shift is not supported");
    TW_REQUIRE(batch >= 0 && batch <= 65535, "tw_shift_frames: bad batch");
    TW_REQUIRE(frames >= 0 && (int64_t)frames * cols < (1LL << 31) * 8, "tw_shift_frames: %d frames out of range", frames);
    if (batch == 0) return 0;
    dim3 grid(148, batch);
    shift_frames_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const uint4*)src_bf16, nullptr, src_row, batch_stride / 8,
                                                               row_off, nullptr, frames, seek, frames, cols / 8,
                                                               (uint4*)dst_bf16, batch_stride / 8, row_off);
    TW_CUDA_CHECK(cudaGetLastError());
    return 0;
}

extern "C" int tw_gather_frames(const void* const* src_rows, const int32_t* frames, const int32_t* seek, int32_t batch,
                                int32_t window, int32_t cols, void* dst_bf16, int64_t dst_batch_stride,
                                int32_t dst_row_off, void* stream) {
    using namespace tw;
    TW_REQUIRE(src_rows && frames && seek && dst_bf16, "tw_gather_frames: null argument");
    if (tw::ensure_device(dst_bf16)) return 1;
    TW_REQUIRE(cols > 0 && cols % 8 == 0 && dst_batch_stride % 8 == 0,
               "tw_gather_frames: cols and dst_batch_stride must be multiples of 8");
    TW_REQUIRE(((uintptr_t)dst_bf16 & 15) == 0, "tw_gather_frames: dst must be 16-byte aligned");
    TW_REQUIRE(window >= 0 && dst_row_off >= 0 && dst_batch_stride >= (int64_t)(dst_row_off + window) * cols,
               "tw_gather_frames: a window of %d frames at row %d does not fit the destination stride", window, dst_row_off);
    TW_REQUIRE(batch >= 0 && batch <= 65535, "tw_gather_frames: %d rows out of range", batch);
    TW_REQUIRE((int64_t)window * cols < (1LL << 31) * 8, "tw_gather_frames: window of %d frames out of range", window);
    if (batch == 0 || window == 0) return 0;
    dim3 grid(148, batch);
    shift_frames_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(nullptr, (const uint4* const*)src_rows, nullptr, 0, 0,
                                                               frames, 0, seek, window, cols / 8, (uint4*)dst_bf16,
                                                               dst_batch_stride / 8, dst_row_off);
    TW_CUDA_CHECK(cudaGetLastError());
    return 0;
}
