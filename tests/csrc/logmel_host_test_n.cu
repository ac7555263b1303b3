// CPU emulation of the log-mel CUDA kernel's phases for a given mel-bin count (-DLOGMEL_NMEL=80 or 128; default 80), the
// same __host__ __device__ code as logmel_host_test.cu run serially.  Usage: logmel_host_test_n pcm.f32 n_valid
// melfilters.f32 out.f32, with melfilters fp32 [201, NMEL] and out fp32 [NMEL, 3000].  Lanes 0 .. NMEL/4 - 1 own bins
// 4l..4l+3 as in the kernel; the remaining lanes of a warp skip the mel phase.
#define TW_HOST_TEST 1
#include "../../turbo-whisper-workspace_b200/csrc/logmel.cu"
#include <stdio.h>
#include <stdlib.h>
#include <stdarg.h>
#include <vector>
namespace tw { void set_error(const char* fmt, ...) { va_list ap; va_start(ap, fmt); vfprintf(stderr, fmt, ap); va_end(ap); } }
using namespace tw::logmel;

#ifndef LOGMEL_NMEL
#define LOGMEL_NMEL 80
#endif
constexpr int NMEL = LOGMEL_NMEL;

static std::vector<float> read_f32(const char* path) {
    FILE* f = fopen(path, "rb"); if (!f) { perror(path); exit(1); }
    fseek(f, 0, SEEK_END); long n = ftell(f); fseek(f, 0, SEEK_SET);
    std::vector<float> v(n / 4); if (fread(v.data(), 4, v.size(), f) != v.size()) exit(1); fclose(f); return v;
}
int main(int argc, char** argv) {
    if (argc != 5) return 2;
    std::vector<float> pcm = read_f32(argv[1]);
    int n_valid = atoi(argv[2]);
    std::vector<float> fb = read_f32(argv[3]);
    if (fb.size() != (size_t)N_BINS * NMEL) { fprintf(stderr, "filterbank must be [201, %d]\n", NMEL); return 2; }
    pcm.resize(N_SAMPLES, 0.f);
    MelTables<NMEL>* tab = new MelTables<NMEL>;
    if (build_tables<NMEL>(fb.data(), tab)) return 1;
    std::vector<float> out((size_t)NMEL * N_FRAMES);
    MelSmem<NMEL>* s = new MelSmem<NMEL>;
    float vmax = -1e30f;
    for (int f0 = 0; f0 < N_FRAMES; f0 += FR) {
        for (int tid = 0; tid < NT; ++tid) phase_load(tid, NT, pcm.data(), n_valid, f0, s->x);
        for (int warp = 0; warp < NWARP; ++warp)
            for (int i = 0; i < FPW; ++i) {
                const int fl = warp * FPW + i, f = f0 + fl;
                if (f >= N_FRAMES) continue;
                float2* wa = s->a[warp];
                float2* wb = s->b[warp];
                float* pw = reinterpret_cast<float*>(wb);
                for (int lane = 0; lane < 32; ++lane) phase_fft_r8(lane, 32, s->x + fl * HOP, tab->window, wa);
                for (int lane = 0; lane < 32; ++lane) phase_fft_r5(lane, 32, 8, tab->tw200, wa, wb);
                for (int lane = 0; lane < 32; ++lane) phase_fft_r5(lane, 32, 40, tab->tw200, wb, wa);
                for (int lane = 0; lane < 32; ++lane) phase_power(lane, 32, tab->tw400, wa, pw);
                for (int lane = 0; lane < MelLayout<NMEL>::LANES; ++lane)
                    for (int q = 0; q < 4; ++q) {
                        const int m = 4 * lane + q;
                        const float l = mel_log10(m, tab->mel_start, tab->mel_cnt, tab->mel_w, pw);
                        vmax = fmaxf(vmax, l);
                        out[(size_t)m * N_FRAMES + f] = scaled(l);
                    }
            }
    }
    const float floor_y = scaled_floor(vmax);
    for (size_t i = 0; i < out.size(); ++i) out[i] = fmaxf(out[i], floor_y);
    FILE* f = fopen(argv[4], "wb"); fwrite(out.data(), 4, out.size(), f); fclose(f);
    return 0;
}
