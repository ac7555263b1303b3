// K1 — fused log-mel front end (SURVEY.md §8 a4), ONE launch.
//
// Replaces WhisperFeatureExtractor._torch_extract_fbank_features
// ($TF/models/whisper/feature_extraction_whisper.py:135-164): reflect-padded 400-point STFT at
// hop 160 with a periodic Hann window, power spectrum, slaney mel filterbank, log10 clamp at 1e-10,
// per-clip `max - 8` floor and (x + 4) / 4.  The bin count is a template parameter: 128 (large-v3 family) or 80
// (large-v2 and older, WhisperFeatureExtractor(feature_size=80)); see MelLayout.
//
// logmel_kernel: a CTA owns FR = 32 consecutive frames of one clip.  The 5360 samples they touch are staged once in
// shared memory (coalesced; reflect padding and the zero tail are index arithmetic), then every WARP works alone on
// its 4 frames, one frame at a time, in a private shared-memory workspace — the 400-point real FFT as a 200-point
// complex Stockham FFT (radix 8, 5, 5), the real post-process + power, the sparse (<= TAPS taps) mel projection,
// log10 — with __syncwarp between the phases and NO block-wide barrier in the loop (the previous version ran the phases
// CTA-wide behind six __syncthreads per 16 frames and was latency-bound at 0.07 of HBM).  Lane l owns mel bins
// 4l..4l+3, so a frame's bf16 values leave as one coalesced row of the time-major layout the conv stem's TMA view reads
// (256 bytes from 32 lanes at 128 bins, 160 bytes from lanes 0-19 at 80 bins; for the reference layout, as float4 runs
// of 4 frames).  The FFT phases, the staging and the floor do not depend on the bin count.
// The per-clip floor needs the maximum over the WHOLE clip.  (x + 4) / 4 and the bf16 rounding are monotone, so
//   (max(l, m - 8) + 4) / 4 == max((l + 4) / 4, ((m - 8) + 4) / 4)      bit for bit,
// i.e. the kernel can store the un-floored value right away, publish its tile's max / min (ordered-int atomicMax, a
// per-tile min), and the LAST CTA of a clip to finish (per-clip arrival counter) raises the few values that lie below
// the floor — only in tiles whose min is below it, read back from L2.  Counters re-arm themselves: one kernel per call.
//
// The arithmetic phases are __host__ __device__ functions over (tid, nthreads) so that the exact
// index arithmetic is also exercised on the CPU by tests/csrc/logmel_host_test.cu.
#include "common.cuh"
#include "twb200_internal.h"
#include <math.h>
#include <algorithm>

namespace tw {
namespace logmel {

constexpr int N_FFT = 400;
constexpr int HOP = 160;
constexpr int N_BINS = 201;
constexpr int N_FRAMES = 3000;
constexpr int N_SAMPLES = 480000;
constexpr int NC = 200;  // complex FFT length
constexpr int FR = 32;   // frames per CTA
constexpr int NT = 256;  // threads per CTA
constexpr int NWARP = NT / 32;
constexpr int FPW = FR / NWARP;               // consecutive frames per warp
constexpr int SX = FR * HOP + (N_FFT - HOP);  // 5360 staged samples
constexpr int POW_LD = 203;                   // padded row length of the power buffer
constexpr int N_TILES = (N_FRAMES + FR - 1) / FR;   // 94 CTAs per clip
constexpr int NCP = NC + NC / 16 + 1;               // padded FFT workspace length (213), see padi()

// The two filterbanks the kernels are built for.  TAPS bounds the non-zero span of one slaney filter over the 201 FFT
// bins (at most 9 at 128 bins, 14 at 80 bins).  Lane l of a warp owns bins 4l..4l+3: all 32 lanes at 128 bins, lanes
// 0-19 at 80 bins (lanes 20-31 skip the mel phase).
template <int NMEL>
struct MelLayout {
    static_assert(NMEL == 128 || NMEL == 80, "log-mel kernels are built for 128 or 80 mel bins");
    static constexpr int TAPS = NMEL == 128 ? 12 : 14;
    static constexpr int LANES = NMEL / 4;
};

template <int NMEL>
struct MelTables {
    static constexpr int TAPS = MelLayout<NMEL>::TAPS;
    float2 tw200[NC];       // exp(-2 pi i m / 200)
    float2 tw400[N_BINS];   // exp(-2 pi i k / 400)
    float window[N_FFT];    // periodic Hann
    int mel_start[NMEL];
    int mel_cnt[NMEL];
    float mel_w[NMEL][TAPS];
};

template <int NMEL>
struct MelSmem {
    static constexpr int TAPS = MelLayout<NMEL>::TAPS;
    float x[SX];
    float2 a[NWARP][NCP];     // per-warp FFT ping (padded, see padi)
    float2 b[NWARP][NCP];     // per-warp FFT pong, then the power spectrum (N_BINS floats)
    float2 tw200[NC];
    float2 tw400[N_BINS];
    float window[N_FFT];
    float4 mel_w4[TAPS][32];           // [tap][lane] = the tap's weight for mel bins 4*lane .. 4*lane+3 (one LDS.128, no conflicts)
    int4 mel_start4[32];               // [lane] = first FFT bin of those four filters
    float red[2][NWARP];
};

#define HD __host__ __device__ __forceinline__

HD float2 cmul(float2 a, float2 b) { return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }
HD float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
HD float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
HD float2 cmul_mi(float2 a) { return make_float2(a.y, -a.x); }  // a * (-i)
HD float2 cmul_pi(float2 a) { return make_float2(-a.y, a.x); }  // a * (+i)

HD void dft4(float2 a, float2 b, float2 c, float2 d, float2& o0, float2& o1, float2& o2, float2& o3) {
    float2 s0 = cadd(a, c), s1 = csub(a, c), s2 = cadd(b, d), s3 = csub(b, d);
    o0 = cadd(s0, s2);
    o1 = cadd(s1, cmul_mi(s3));
    o2 = csub(s0, s2);
    o3 = cadd(s1, cmul_pi(s3));
}
HD void dft8(float2* v) {
    const float h = 0.70710678118654752f;
    float2 e0, e1, e2, e3, o0, o1, o2, o3;
    dft4(v[0], v[2], v[4], v[6], e0, e1, e2, e3);
    dft4(v[1], v[3], v[5], v[7], o0, o1, o2, o3);
    // w8^1 = (1 - i)/sqrt2, w8^2 = -i, w8^3 = (-1 - i)/sqrt2
    float2 t1 = make_float2(h * (o1.x + o1.y), h * (o1.y - o1.x));
    float2 t2 = cmul_mi(o2);
    float2 t3 = make_float2(h * (o3.y - o3.x), -h * (o3.x + o3.y));
    v[0] = cadd(e0, o0); v[4] = csub(e0, o0);
    v[1] = cadd(e1, t1); v[5] = csub(e1, t1);
    v[2] = cadd(e2, t2); v[6] = csub(e2, t2);
    v[3] = cadd(e3, t3); v[7] = csub(e3, t3);
}
HD void dft5(float2* v) {
    const float c1 = 0.30901699437494742f, c2 = -0.80901699437494742f;
    const float s1 = 0.95105651629515357f, s2 = 0.58778525229247313f;
    float2 a1 = cadd(v[1], v[4]), a2 = cadd(v[2], v[3]);
    float2 b1 = csub(v[1], v[4]), b2 = csub(v[2], v[3]);
    float2 r0 = cadd(v[0], cadd(a1, a2));
    float2 p1 = make_float2(v[0].x + c1 * a1.x + c2 * a2.x, v[0].y + c1 * a1.y + c2 * a2.y);
    float2 p2 = make_float2(v[0].x + c2 * a1.x + c1 * a2.x, v[0].y + c2 * a1.y + c1 * a2.y);
    float2 q1 = make_float2(s1 * b1.x + s2 * b2.x, s1 * b1.y + s2 * b2.y);
    float2 q2 = make_float2(s2 * b1.x - s1 * b2.x, s2 * b1.y - s1 * b2.y);
    v[0] = r0;
    v[1] = cadd(p1, cmul_mi(q1));
    v[4] = cadd(p1, cmul_pi(q1));
    v[2] = cadd(p2, cmul_mi(q2));
    v[3] = cadd(p2, cmul_pi(q2));
}

// phase 0: stage samples [160*f0 - 200, 160*f0 - 200 + SX) with reflect padding on the 480000-
// sample (zero-padded) clip; samples at or beyond n_valid read as 0 (HF pads with zeros first,
// then torch.stft(center=True) reflects the padded clip).
HD void phase_load(int tid, int nt, const float* pcm, int n_valid, int f0, float* sx) {
    const int base = HOP * f0 - N_FFT / 2;
    for (int i = tid; i < SX; i += nt) {
        int g = base + i;
        if (g < 0) g = -g;
        if (g >= N_SAMPLES) g = 2 * (N_SAMPLES - 1) - g;
        sx[i] = (g < n_valid) ? pcm[g] : 0.0f;
    }
}
// FFT workspaces are padded by one complex slot per 16 (the radix-8 stage writes with a stride of 8 complex values =
// 64 bytes: without padding 13 of its 25 lanes hit the same two banks)
HD int padi(int i) { return i + (i >> 4); }
// The FFT phases below work on ONE frame (a warp's current frame): xf = its 400 staged samples.
// phase 1: window + pack to complex + radix-8 stage (Ns = 1, no twiddles).  25 items.
HD void phase_fft_r8(int tid, int nt, const float* xf, const float* window, float2* out) {
    constexpr int T = NC / 8;  // 25
    for (int j = tid; j < T; j += nt) {
        float2 v[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            const int n = j + t * T;
            v[t] = make_float2(xf[2 * n] * window[2 * n], xf[2 * n + 1] * window[2 * n + 1]);
        }
        dft8(v);
#pragma unroll
        for (int u = 0; u < 8; ++u) out[padi(j * 8 + u)] = v[u];
    }
}
// phases 2/3: radix-5 Stockham stage with sub-transform length Ns (8, then 40).  40 items.
HD void phase_fft_r5(int tid, int nt, int Ns, const float2* tw200, const float2* in, float2* out) {
    constexpr int T = NC / 5;  // 40
    const int twstep = NC / (Ns * 5);
    for (int j = tid; j < T; j += nt) {
        const int k = j % Ns;
        float2 v[5];
        v[0] = in[padi(j)];
#pragma unroll
        for (int t = 1; t < 5; ++t) v[t] = cmul(in[padi(j + t * T)], tw200[t * k * twstep]);
        dft5(v);
        const int j0 = (j / Ns) * Ns * 5 + k;
#pragma unroll
        for (int u = 0; u < 5; ++u) out[padi(j0 + u * Ns)] = v[u];
    }
}
// phase 4: real-FFT post-process + power.  X[k] = E[k] + W400^k O[k], k = 0..200.
HD void phase_power(int tid, int nt, const float2* tw400, const float2* Z, float* pw) {
    for (int k = tid; k < N_BINS; k += nt) {
        const float2 zk = Z[padi(k == NC ? 0 : k)];
        const float2 zr = Z[padi((k == 0 || k == NC) ? 0 : NC - k)];
        const float2 zc = make_float2(zr.x, -zr.y);
        const float2 e = make_float2(0.5f * (zk.x + zc.x), 0.5f * (zk.y + zc.y));
        const float2 d = make_float2(0.5f * (zk.x - zc.x), 0.5f * (zk.y - zc.y));
        const float2 o = cmul_mi(d);
        const float2 x = cadd(e, cmul(tw400[k], o));
        pw[k] = x.x * x.x + x.y * x.y;
    }
}
// phase 5: one mel bin of one frame: sparse projection + log10 clamp
template <int TAPS>
HD float mel_log10(int m, const int* mel_start, const int* mel_cnt, const float (*mel_w)[TAPS], const float* pw) {
    const int s = mel_start[m], c = mel_cnt[m];
    float acc = 0.0f;
    for (int i = 0; i < c; ++i) acc = fmaf(mel_w[m][i], pw[s + i], acc);
    return log10f(fmaxf(acc, 1e-10f));
}
// the value stored before the per-clip floor is known, and the floor in the same scale (see the header: monotone)
HD float scaled(float log10_value) { return (log10_value + 4.0f) * 0.25f; }
HD float scaled_floor(float clip_max_log10) { return ((clip_max_log10 - 8.0f) + 4.0f) * 0.25f; }

#ifndef TW_HOST_TEST
// monotone map float -> unsigned whose ZERO is below every float: zero-filled scratch is a valid "no maximum yet"
TW_DEVINL unsigned int float_to_umono(float f) { return (unsigned int)float_to_ordered(f) ^ 0x80000000u; }
TW_DEVINL float umono_to_float(unsigned int u) { return ordered_to_float((int)(u ^ 0x80000000u)); }

struct Scratch {            // per clip; zero-filled once by the owner, re-armed by the kernel
    unsigned int clip_max;  // float_to_umono(max log10 value of the clip)
    unsigned int arrived;   // CTAs of this clip that have stored their tile
    float tile_min[N_TILES];
    float tile_max[N_TILES];
};

// Fills the table part of the shared memory: twiddles, window, and the filterbank transposed to [tap][lane] float4s.
template <int NMEL>
TW_DEVINL void load_tables(int tid, const MelTables<NMEL>* __restrict__ tab, MelSmem<NMEL>& s) {
    constexpr int TAPS = MelLayout<NMEL>::TAPS, LANES = MelLayout<NMEL>::LANES;
    for (int i = tid; i < NC; i += NT) s.tw200[i] = tab->tw200[i];
    for (int i = tid; i < N_BINS; i += NT) s.tw400[i] = tab->tw400[i];
    for (int i = tid; i < N_FFT; i += NT) s.window[i] = tab->window[i];
    for (int i = tid; i < TAPS * 32; i += NT) {
        const int tap = i >> 5, l = i & 31;
        if (l < LANES)
            s.mel_w4[tap][l] = make_float4(tab->mel_w[4 * l][tap], tab->mel_w[4 * l + 1][tap], tab->mel_w[4 * l + 2][tap],
                                           tab->mel_w[4 * l + 3][tap]);
    }
    if (tid < LANES) s.mel_start4[tid] = make_int4(tab->mel_start[4 * tid], tab->mel_start[4 * tid + 1], tab->mel_start[4 * tid + 2],
                                                   tab->mel_start[4 * tid + 3]);
}

// Sparse mel projection of the four bins 4*lane .. 4*lane+3 of the frame whose power spectrum is pw: taps beyond a
// filter's length carry weight 0 (same fmaf order as mel_log10, so the sums are identical to the host emulation's).
template <int NMEL>
TW_DEVINL void mel_project(int lane, const MelSmem<NMEL>& s, const float* pw, float (&acc)[4]) {
    const int4 st4 = s.mel_start4[lane];
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[q] = 0.f;
#pragma unroll
    for (int tp = 0; tp < MelLayout<NMEL>::TAPS; ++tp) {
        const float4 w = s.mel_w4[tp][lane];
        acc[0] = fmaf(w.x, pw[min(st4.x + tp, N_BINS - 1)], acc[0]);
        acc[1] = fmaf(w.y, pw[min(st4.y + tp, N_BINS - 1)], acc[1]);
        acc[2] = fmaf(w.z, pw[min(st4.z + tp, N_BINS - 1)], acc[2]);
        acc[3] = fmaf(w.w, pw[min(st4.w + tp, N_BINS - 1)], acc[3]);
    }
}
// log10 through the hardware log2 (abs. error < 2e-7 here, the stated tolerance is 1e-4)
TW_DEVINL float fast_log10(float acc) { return __log2f(fmaxf(acc, 1e-10f)) * 0.30102999566398120f; }

template <int NMEL>
__global__ void __launch_bounds__(NT) logmel_kernel(const float* __restrict__ pcm, long long pcm_stride,
                                                   const int* __restrict__ n_valid, const MelTables<NMEL>* __restrict__ tab,
                                                   Scratch* __restrict__ scratch, float* __restrict__ out_f32,
                                                   __nv_bfloat16* __restrict__ out_t, long long out_t_bstride,
                                                   int row_off) {
    constexpr int LANES = MelLayout<NMEL>::LANES;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    MelSmem<NMEL>& s = *reinterpret_cast<MelSmem<NMEL>*>(smem_raw);
    __shared__ int s_last;
    const int b = blockIdx.y, tile = blockIdx.x;
    const int f0 = tile * FR;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nv = n_valid ? min(n_valid[b], N_SAMPLES) : N_SAMPLES;

    load_tables<NMEL>(tid, tab, s);
    phase_load(tid, NT, pcm + (size_t)b * pcm_stride, nv, f0, s.x);
    __syncthreads();

    // every warp: its FPW frames, one at a time, in its own workspace
    float2* wa = s.a[warp];
    float2* wb = s.b[warp];
    float* pw = reinterpret_cast<float*>(wb);
    float vmax = -INFINITY, vmin = INFINITY;
    float keep[FPW][4];                       // reference-layout output: 4 mel rows x FPW consecutive frames per lane
    float* of = (out_f32 && lane < LANES) ? out_f32 + ((size_t)b * NMEL + 4 * lane) * N_FRAMES : nullptr;
    __nv_bfloat16* ot = out_t ? out_t + (size_t)b * out_t_bstride : nullptr;
#pragma unroll
    for (int i = 0; i < FPW; ++i) {
        const int fl = warp * FPW + i;        // frame within the tile
        const int f = f0 + fl;
        if (f < N_FRAMES) {                   // warp-uniform
            phase_fft_r8(lane, 32, s.x + fl * HOP, s.window, wa);
            __syncwarp();
            phase_fft_r5(lane, 32, 8, s.tw200, wa, wb);
            __syncwarp();
            phase_fft_r5(lane, 32, 40, s.tw200, wb, wa);
            __syncwarp();
            phase_power(lane, 32, s.tw400, wa, pw);
            __syncwarp();
            if (lane < LANES) {               // all lanes at 128 bins
                float acc[4], y[4];
                mel_project<NMEL>(lane, s, pw, acc);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float l = fast_log10(acc[q]);
                    vmax = fmaxf(vmax, l);
                    vmin = fminf(vmin, l);
                    y[q] = scaled(l);
                    keep[i][q] = y[q];
                }
                if (ot) {
                    uint2 pk;
                    pk.x = pack_bf16x2(y[0], y[1]);
                    pk.y = pack_bf16x2(y[2], y[3]);
                    reinterpret_cast<uint2*>(ot + (size_t)(row_off + f) * NMEL)[lane] = pk;
                }
            }
            __syncwarp();                     // pw (= wb) and wa are reused by the next frame
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) keep[i][q] = 0.f;
        }
    }
    if (of) {
        const int fw = f0 + warp * FPW;       // first frame of this warp: a multiple of 4, so float4 stores are aligned
        if (fw + FPW <= N_FRAMES) {
#pragma unroll
            for (int q = 0; q < 4; ++q)
                *reinterpret_cast<float4*>(of + (size_t)q * N_FRAMES + fw) = make_float4(keep[0][q], keep[1][q], keep[2][q], keep[3][q]);
        } else {
            for (int i = 0; i < FPW; ++i)
                if (fw + i < N_FRAMES)
                    for (int q = 0; q < 4; ++q) of[(size_t)q * N_FRAMES + fw + i] = keep[i][q];
        }
    }
    // tile statistics -> clip maximum (atomic), per-tile min / max for the floor pass
    vmax = warp_max(vmax);
    vmin = -warp_max(-vmin);
    if (lane == 0) { s.red[0][warp] = vmax; s.red[1][warp] = vmin; }
    __threadfence();                          // this CTA's output is visible before it counts as arrived
    __syncthreads();
    Scratch& sc = scratch[b];
    if (tid == 0) {
        float mx = s.red[0][0], mn = s.red[1][0];
#pragma unroll
        for (int i = 1; i < NWARP; ++i) { mx = fmaxf(mx, s.red[0][i]); mn = fminf(mn, s.red[1][i]); }
        sc.tile_min[tile] = mn;
        sc.tile_max[tile] = mx;
        atomicMax(&sc.clip_max, float_to_umono(mx));
        __threadfence();
        const unsigned int prev = atomicAdd(&sc.arrived, 1u);
        s_last = (prev == gridDim.x - 1);
    }
    __syncthreads();
    if (!s_last) return;
    // ---- last CTA of the clip: raise everything below the floor (only tiles that have such values)
    __threadfence();
    const float clip_max = umono_to_float(__ldcg(&sc.clip_max));
    const float floor_l = clip_max - 8.0f, floor_y = scaled_floor(clip_max);
    const uint32_t floor_bf = pack_bf16x2(floor_y, floor_y);
    const float floor_bf_f = __uint_as_float(floor_bf << 16);
    for (int t = 0; t < (int)gridDim.x; ++t) {
        if (!(__ldcg(&sc.tile_min[t]) < floor_l)) continue;      // block-uniform
        const int tf0 = t * FR, nfr = min(FR, N_FRAMES - tf0);
        if (ot) {   // nfr rows of NMEL bf16, contiguous: NMEL / 8 uint4 per row
            uint4* base = reinterpret_cast<uint4*>(ot + (size_t)(row_off + tf0) * NMEL);
            for (int i = tid; i < nfr * (NMEL / 8); i += NT) {
                uint4 v = __ldcg(base + i);
                uint32_t* w = reinterpret_cast<uint32_t*>(&v);
                bool changed = false;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    float lo = __uint_as_float(w[k] << 16), hi = __uint_as_float(w[k] & 0xffff0000u);
                    if (lo < floor_bf_f) { lo = floor_bf_f; changed = true; }
                    if (hi < floor_bf_f) { hi = floor_bf_f; changed = true; }
                    w[k] = (__float_as_uint(lo) >> 16) | (__float_as_uint(hi) & 0xffff0000u);
                }
                if (changed) base[i] = v;
            }
        }
        if (out_f32) {
            float* fb = out_f32 + (size_t)b * NMEL * N_FRAMES + tf0;
            for (int i = tid; i < NMEL * nfr; i += NT) {
                const int m = i / nfr, fr = i - m * nfr;
                float* p = fb + (size_t)m * N_FRAMES + fr;
                if (__ldcg(p) < floor_y) *p = floor_y;
            }
        }
    }
    __syncthreads();
    if (tid == 0) { sc.clip_max = 0u; sc.arrived = 0u; }      // re-arm for the next call on this stream
}

// ---- whole-clip features for un-chunked long-form input (WhisperFeatureExtractor with truncation=False,
// $TF/models/whisper/feature_extraction_whisper.py:135-164 over the full waveform; the ASR pipeline's path for inputs
// longer than 30 s without chunk_length_s, $TF/pipelines/automatic_speech_recognition.py:446-454).  The clip is covered by
// OVERLAPPING 30 s windows that start `hop_samples` apart: a frame only depends on 400 samples, so every frame of a
// window that does not touch the window's own reflect padding equals the clip's frame; window b contributes its frames
// [frame_lo[b], frame_hi[b]) to rows out_row0[b].. of the clip's time-major output.  The clamp uses the maximum of the
// WHOLE clip: this kernel stores un-floored values and raises the clip's maximum, logmel_floor_kernel applies the floor.
// Several clips in one launch: window b reads pcm + win_off[b] and raises long_max[win_clip[b]] (NULL arrays: window b
// starts at b * hop_samples and every window belongs to clip 0).
template <int NMEL>
__global__ void __launch_bounds__(NT) logmel_long_kernel(const float* __restrict__ pcm, long long hop_samples,
                                                        const long long* __restrict__ win_off,
                                                        const int* __restrict__ win_clip,
                                                        const MelTables<NMEL>* __restrict__ tab, const int* __restrict__ frame_lo,
                                                        const int* __restrict__ frame_hi, const int* __restrict__ out_row0,
                                                        unsigned int* __restrict__ long_max,
                                                        __nv_bfloat16* __restrict__ out_t, int row_off) {
    constexpr int LANES = MelLayout<NMEL>::LANES;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    MelSmem<NMEL>& s = *reinterpret_cast<MelSmem<NMEL>*>(smem_raw);
    const int b = blockIdx.y, tile = blockIdx.x;
    const int f0 = tile * FR;
    const int lo = frame_lo[b], hi = frame_hi[b];
    if (f0 + FR <= lo || f0 >= hi) return;       // block-uniform: no frame of this tile belongs to the window's share
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    load_tables<NMEL>(tid, tab, s);
    phase_load(tid, NT, pcm + (win_off ? win_off[b] : (long long)b * hop_samples), N_SAMPLES, f0, s.x);
    __syncthreads();

    float2* wa = s.a[warp];
    float2* wb = s.b[warp];
    float* pw = reinterpret_cast<float*>(wb);
    float vmax = -INFINITY;
    __nv_bfloat16* ot = out_t + (size_t)(row_off + out_row0[b] - lo) * NMEL;     // row of window frame 0 (may lie before row 0)
#pragma unroll
    for (int i = 0; i < FPW; ++i) {
        const int fl = warp * FPW + i;
        const int f = f0 + fl;
        if (f >= lo && f < hi) {                  // warp-uniform
            phase_fft_r8(lane, 32, s.x + fl * HOP, s.window, wa);
            __syncwarp();
            phase_fft_r5(lane, 32, 8, s.tw200, wa, wb);
            __syncwarp();
            phase_fft_r5(lane, 32, 40, s.tw200, wb, wa);
            __syncwarp();
            phase_power(lane, 32, s.tw400, wa, pw);
            __syncwarp();
            if (lane < LANES) {               // all lanes at 128 bins
                float acc[4], y[4];
                mel_project<NMEL>(lane, s, pw, acc);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float l = fast_log10(acc[q]);
                    vmax = fmaxf(vmax, l);
                    y[q] = scaled(l);
                }
                uint2 pk;
                pk.x = pack_bf16x2(y[0], y[1]);
                pk.y = pack_bf16x2(y[2], y[3]);
                reinterpret_cast<uint2*>(ot + (size_t)f * NMEL)[lane] = pk;
            }
            __syncwarp();
        }
    }
    vmax = warp_max(vmax);
    if (lane == 0) s.red[0][warp] = vmax;
    __syncthreads();
    if (tid == 0) {
        float mx = s.red[0][0];
#pragma unroll
        for (int i = 1; i < NWARP; ++i) mx = fmaxf(mx, s.red[0][i]);
        if (mx > -INFINITY) atomicMax(long_max + (win_clip ? win_clip[b] : 0), float_to_umono(mx));
    }
}

// raise every value below the clip's floor (max - 8 in log10 units, compared after the bf16 rounding of the output, like
// the floor pass of logmel_kernel).  It sees the output as a flat run of uint4, so one kernel serves both bin counts.
// blockIdx.y = clip c, which owns the rows [clip_row[c], clip_row[c + 1]) (vec_per_row uint4 each) and the maximum
// long_max[c] (clip_row NULL: one clip owning the whole run [0, n_vec)).
__global__ void __launch_bounds__(256) logmel_floor_kernel(uint4* __restrict__ mel, long long n_vec,
                                                          const long long* __restrict__ clip_row, int vec_per_row,
                                                          const unsigned int* __restrict__ long_max) {
    const int c = blockIdx.y;
    const float floor_y = scaled_floor(umono_to_float(long_max[c]));
    const uint32_t floor_bf = pack_bf16x2(floor_y, floor_y);
    const float floor_bf_f = __uint_as_float(floor_bf << 16);
    const long long v0 = clip_row ? clip_row[c] * vec_per_row : 0, v1 = clip_row ? clip_row[c + 1] * vec_per_row : n_vec;
    for (long long i = v0 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < v1; i += (long long)gridDim.x * blockDim.x) {
        uint4 v = mel[i];
        uint32_t* w = reinterpret_cast<uint32_t*>(&v);
        bool changed = false;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float lo = __uint_as_float(w[k] << 16), hi = __uint_as_float(w[k] & 0xffff0000u);
            if (lo < floor_bf_f) { lo = floor_bf_f; changed = true; }
            if (hi < floor_bf_f) { hi = floor_bf_f; changed = true; }
            w[k] = (__float_as_uint(lo) >> 16) | (__float_as_uint(hi) & 0xffff0000u);
        }
        if (changed) mel[i] = v;
    }
}
#endif  // TW_HOST_TEST

// Host: build the constant tables from the dense [201, NMEL] fp32 filterbank (HF mel_filters).
template <int NMEL>
int build_tables(const float* mel_filters, MelTables<NMEL>* t) {
    constexpr int TAPS = MelLayout<NMEL>::TAPS;
    const double PI = 3.14159265358979323846;
    for (int m = 0; m < NC; ++m)
        t->tw200[m] = make_float2((float)cos(2.0 * PI * m / NC), (float)-sin(2.0 * PI * m / NC));
    for (int k = 0; k < N_BINS; ++k)
        t->tw400[k] = make_float2((float)cos(2.0 * PI * k / N_FFT), (float)-sin(2.0 * PI * k / N_FFT));
    for (int n = 0; n < N_FFT; ++n) t->window[n] = (float)(0.5 - 0.5 * cos(2.0 * PI * n / N_FFT));
    for (int m = 0; m < NMEL; ++m) {
        int first = -1, last = -1;
        for (int k = 0; k < N_BINS; ++k)
            if (mel_filters[k * NMEL + m] != 0.0f) {
                if (first < 0) first = k;
                last = k;
            }
        if (first < 0) { first = 0; last = -1; }
        const int cnt = last - first + 1;
        if (cnt > TAPS) {
            set_error("mel filter %d has %d taps (max %d)", m, cnt, TAPS);
            return 2;
        }
        t->mel_start[m] = first;
        t->mel_cnt[m] = cnt;
        for (int i = 0; i < TAPS; ++i)
            t->mel_w[m][i] = (i < cnt) ? mel_filters[(first + i) * NMEL + m] : 0.0f;
    }
    return 0;
}

#ifdef TW_HOST_TEST
// The names tests/csrc/logmel_host_test.cu is written against: the 128-bin layout.
constexpr int N_MEL = 128;
constexpr int MEL_MAX_TAPS = MelLayout<N_MEL>::TAPS;
using Tables = MelTables<N_MEL>;
using Smem = MelSmem<N_MEL>;
#endif

}  // namespace logmel
}  // namespace tw

#ifndef TW_HOST_TEST
using namespace tw;
using namespace tw::logmel;

extern "C" size_t tw_logmel_tables_bytes(void) { return std::max(sizeof(MelTables<128>), sizeof(MelTables<80>)); }
extern "C" size_t tw_logmel_scratch_bytes(int batch) { return (size_t)batch * sizeof(Scratch); }

#define TW_REQUIRE_N_MELS(fn, n)                                                                        \
    TW_REQUIRE((n) == 128 || (n) == 80, fn ": n_mels %d is not supported (the kernels are built for 80 and 128)", (int)(n))

namespace {
template <int NMEL>
int logmel_init(void* tables_dev, const float* mel_filters) {
    MelTables<NMEL>* h = new MelTables<NMEL>;
    int rc = build_tables<NMEL>(mel_filters, h);
    if (rc == 0) {
        cudaError_t e = cudaMemcpy(tables_dev, h, sizeof(MelTables<NMEL>), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) {
            set_error("tw_logmel_init: cudaMemcpy failed: %s", cudaGetErrorString(e));
            rc = 1;
        }
    }
    delete h;
    return rc;
}

template <int NMEL>
int logmel_launch(const void* tables_dev, const float* pcm, int64_t pcm_stride, const int32_t* n_valid, int batch,
                  void* scratch, float* out_f32, void* out_bf16_t, int64_t out_t_bstride, int32_t out_t_row_off,
                  cudaStream_t stream) {
    static std::atomic<unsigned long long> attr_done{0};
    if (device_needs_setup(attr_done)) {
        TW_CUDA_CHECK(cudaFuncSetAttribute(logmel_kernel<NMEL>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)sizeof(MelSmem<NMEL>)));
        mark_device_done(attr_done);
    }
    logmel_kernel<NMEL><<<dim3(N_TILES, batch), NT, sizeof(MelSmem<NMEL>), stream>>>(
        pcm, (long long)pcm_stride, n_valid, (const MelTables<NMEL>*)tables_dev, (Scratch*)scratch, out_f32,
        (__nv_bfloat16*)out_bf16_t, (long long)out_t_bstride, out_t_row_off);
    TW_CUDA_CHECK(cudaGetLastError());
    return 0;
}

template <int NMEL>
int logmel_long_launch(const void* tables_dev, const float* pcm_long, int64_t hop_samples, const int64_t* win_off,
                       const int32_t* win_clip, int32_t n_windows, const int32_t* frame_lo, const int32_t* frame_hi,
                       const int32_t* out_row0, int32_t n_clips, const int64_t* clip_row, uint32_t* max_scratch,
                       void* out_bf16_t, int64_t total_frames, int32_t out_t_row_off, cudaStream_t st) {
    static std::atomic<unsigned long long> attr_done{0};
    if (device_needs_setup(attr_done)) {
        TW_CUDA_CHECK(cudaFuncSetAttribute(logmel_long_kernel<NMEL>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)sizeof(MelSmem<NMEL>)));
        mark_device_done(attr_done);
    }
    // zero is below every real value in the ordered map
    TW_CUDA_CHECK(cudaMemsetAsync(max_scratch, 0, sizeof(uint32_t) * n_clips, st));
    logmel_long_kernel<NMEL><<<dim3(N_TILES, n_windows), NT, sizeof(MelSmem<NMEL>), st>>>(
        pcm_long, (long long)hop_samples, (const long long*)win_off, win_clip, (const MelTables<NMEL>*)tables_dev,
        frame_lo, frame_hi, out_row0, max_scratch, (__nv_bfloat16*)out_bf16_t, out_t_row_off);
    TW_CUDA_CHECK(cudaGetLastError());
    const long long n_vec = (long long)total_frames * NMEL / 8;
    uint4* first = reinterpret_cast<uint4*>((__nv_bfloat16*)out_bf16_t + (size_t)out_t_row_off * NMEL);
    const int blocks = (int)std::max<long long>(1, std::min<long long>((n_vec / n_clips + 255) / 256, 148 * 8));
    logmel_floor_kernel<<<dim3(blocks, n_clips), 256, 0, st>>>(first, n_vec, (const long long*)clip_row, NMEL / 8,
                                                                max_scratch);
    TW_CUDA_CHECK(cudaGetLastError());
    return 0;
}
}  // namespace

extern "C" int tw_logmel_init_n(void* tables_dev, const float* mel_filters_host, int32_t n_mels) {
    TW_REQUIRE(tables_dev && mel_filters_host, "tw_logmel_init: null argument");
    TW_REQUIRE_N_MELS("tw_logmel_init", n_mels);
    return n_mels == 128 ? logmel_init<128>(tables_dev, mel_filters_host) : logmel_init<80>(tables_dev, mel_filters_host);
}

extern "C" int tw_logmel_init(void* tables_dev, const float* mel_filters_host_201x128) {
    return tw_logmel_init_n(tables_dev, mel_filters_host_201x128, 128);
}

extern "C" int tw_logmel_n(const void* tables_dev, const float* pcm, int64_t pcm_stride,
                           const int32_t* n_valid, int batch, void* scratch, float* out_f32,
                           void* out_bf16_t, int64_t out_t_bstride, int32_t out_t_row_off,
                           int32_t n_mels, void* stream) {
    TW_REQUIRE(tables_dev && pcm && scratch, "tw_logmel: null argument");
    TW_REQUIRE_N_MELS("tw_logmel", n_mels);
    if (tw::ensure_device(pcm)) return 1;
    TW_REQUIRE(batch >= 0 && batch <= 65535, "tw_logmel: batch %d out of range", batch);
    TW_REQUIRE(pcm_stride >= N_SAMPLES, "tw_logmel: pcm_stride %lld < %d", (long long)pcm_stride,
               N_SAMPLES);
    TW_REQUIRE(!out_bf16_t || (((uintptr_t)out_bf16_t & 15) == 0 && out_t_bstride % 8 == 0),
               "tw_logmel: the time-major output must be 16-byte aligned");
    TW_REQUIRE(!out_f32 || ((uintptr_t)out_f32 & 15) == 0, "tw_logmel: out_f32 must be 16-byte aligned");
    if (batch == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    return n_mels == 128
        ? logmel_launch<128>(tables_dev, pcm, pcm_stride, n_valid, batch, scratch, out_f32, out_bf16_t, out_t_bstride,
                             out_t_row_off, st)
        : logmel_launch<80>(tables_dev, pcm, pcm_stride, n_valid, batch, scratch, out_f32, out_bf16_t, out_t_bstride,
                            out_t_row_off, st);
}

extern "C" int tw_logmel(const void* tables_dev, const float* pcm, int64_t pcm_stride,
                         const int32_t* n_valid, int batch, void* scratch, float* out_f32,
                         void* out_bf16_t, int64_t out_t_bstride, int32_t out_t_row_off,
                         void* stream) {
    return tw_logmel_n(tables_dev, pcm, pcm_stride, n_valid, batch, scratch, out_f32, out_bf16_t, out_t_bstride,
                       out_t_row_off, 128, stream);
}

extern "C" int tw_logmel_long_n(const void* tables_dev, const float* pcm_long, int64_t hop_samples, int32_t n_windows,
                                const int32_t* frame_lo, const int32_t* frame_hi, const int32_t* out_row0,
                                uint32_t* max_scratch, void* out_bf16_t, int64_t total_frames, int32_t out_t_row_off,
                                int32_t n_mels, void* stream) {
    TW_REQUIRE(tables_dev && pcm_long && frame_lo && frame_hi && out_row0 && max_scratch && out_bf16_t,
               "tw_logmel_long: null argument");
    TW_REQUIRE_N_MELS("tw_logmel_long", n_mels);
    if (tw::ensure_device(pcm_long)) return 1;
    TW_REQUIRE(n_windows >= 0 && n_windows <= 65535, "tw_logmel_long: %d windows out of range", n_windows);
    TW_REQUIRE(hop_samples > 0 && hop_samples % HOP == 0, "tw_logmel_long: hop_samples must be a positive multiple of %d", HOP);
    TW_REQUIRE(((uintptr_t)out_bf16_t & 15) == 0 && total_frames >= 0, "tw_logmel_long: the output must be 16-byte aligned");
    if (n_windows == 0 || total_frames == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    return n_mels == 128
        ? logmel_long_launch<128>(tables_dev, pcm_long, hop_samples, nullptr, nullptr, n_windows, frame_lo, frame_hi,
                                  out_row0, 1, nullptr, max_scratch, out_bf16_t, total_frames, out_t_row_off, st)
        : logmel_long_launch<80>(tables_dev, pcm_long, hop_samples, nullptr, nullptr, n_windows, frame_lo, frame_hi,
                                 out_row0, 1, nullptr, max_scratch, out_bf16_t, total_frames, out_t_row_off, st);
}

extern "C" int tw_logmel_long_multi(const void* tables_dev, const float* pcm, const int64_t* win_offset,
                                    const int32_t* win_clip, int32_t n_windows, const int32_t* frame_lo,
                                    const int32_t* frame_hi, const int32_t* out_row0, int32_t n_clips,
                                    const int64_t* clip_row0, uint32_t* max_scratch, void* out_bf16_t,
                                    int64_t total_frames, int32_t n_mels, void* stream) {
    TW_REQUIRE(tables_dev && pcm && win_offset && win_clip && frame_lo && frame_hi && out_row0 && clip_row0 &&
               max_scratch && out_bf16_t, "tw_logmel_long_multi: null argument");
    TW_REQUIRE_N_MELS("tw_logmel_long_multi", n_mels);
    if (tw::ensure_device(pcm)) return 1;
    TW_REQUIRE(n_windows >= 0 && n_windows <= 65535, "tw_logmel_long_multi: %d windows out of range", n_windows);
    TW_REQUIRE(n_clips >= 1 && n_clips <= 65535, "tw_logmel_long_multi: %d clips out of range", n_clips);
    TW_REQUIRE(((uintptr_t)out_bf16_t & 15) == 0 && total_frames >= 0,
               "tw_logmel_long_multi: the output must be 16-byte aligned");
    if (n_windows == 0 || total_frames == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    return n_mels == 128
        ? logmel_long_launch<128>(tables_dev, pcm, 1, win_offset, win_clip, n_windows, frame_lo, frame_hi, out_row0,
                                  n_clips, clip_row0, max_scratch, out_bf16_t, total_frames, 0, st)
        : logmel_long_launch<80>(tables_dev, pcm, 1, win_offset, win_clip, n_windows, frame_lo, frame_hi, out_row0,
                                 n_clips, clip_row0, max_scratch, out_bf16_t, total_frames, 0, st);
}

extern "C" int tw_logmel_long(const void* tables_dev, const float* pcm_long, int64_t hop_samples, int32_t n_windows,
                              const int32_t* frame_lo, const int32_t* frame_hi, const int32_t* out_row0,
                              uint32_t* max_scratch, void* out_bf16_t, int64_t total_frames, int32_t out_t_row_off,
                              void* stream) {
    return tw_logmel_long_n(tables_dev, pcm_long, hop_samples, n_windows, frame_lo, frame_hi, out_row0, max_scratch,
                            out_bf16_t, total_frames, out_t_row_off, 128, stream);
}
#endif
