// K5 — persistent, warp-specialised, TMA-fed tcgen05/TMEM bf16 GEMM with fused epilogue.
//
//   out[b, r, n] = act( sum_k A[b, a_row_off[b] + r, k] * W[n, k] + bias[n] ) + resid[b, r, n]
//
// A (activations) and W (nn.Linear weight [N,K]) are both K-major, which is exactly the operand
// layout tcgen05.mma wants, so no transposes exist anywhere.  A is addressed through a rank-3 TMA
// tensor map (k, row, batch) whose row stride is a free parameter: nn.Linear uses stride K, the two
// Conv1d layers of the Whisper stem use overlapping rows (stride C resp. 2C, length 3C) over
// time-major activations, so im2col is never materialised
// ($TF/models/whisper/modeling_whisper.py:619-620 conv1/conv2 + gelu).
//
// CTA = 320 threads: warp 0 TMA producer, warp 1 MMA issuer (+TMEM owner), warps 2-9 epilogue.  CTA pairs
// (cta_group::2) own a 256 x 256 x 64 tile, 6-stage ring of 32 KB per CTA.
// Two 256-column fp32 accumulators in TMEM per CTA so the epilogue of tile i overlaps the MMAs of tile i+1.
// Grid = #SMs, static tile striding.
#include "common.cuh"
#include "twb200_internal.h"

namespace tw {
namespace gemm {

constexpr int BM = 128;
constexpr int BN = 256;
constexpr int BK = 64;
constexpr int UMMA_K = 16;
constexpr int A_STAGE_BYTES = BM * BK * 2;  // 16 KB
constexpr int NUM_THREADS = 320;   // warp 0 TMA, warp 1 MMA, warps 2-9 epilogue (two warps per TMEM lane quarter)
constexpr int TMEM_COLS = 512;
constexpr int EPI_WARPS = 8;
constexpr int EPI_STAGE_BYTES = EPI_WARPS * 32 * 32 * 4;  // one 32x32 fp32 tile per epilogue warp

struct Params {
    int rows, batches, N, K;
    int m_tiles_per_batch, n_tiles, num_tiles, num_k_blocks;   // a tile is 2 * BM rows (one CTA pair) x BN columns
    const int* a_row_off;
    const float* bias;
    const float* resid;
    long long resid_ld, resid_batch_rows;
    void* out;
    int out_f32;
    long long out_ld, out_batch_rows;
    int out_row_off;
    int act;
    int out_mode;  // 0: row-major [.., out_ld]; 1: head-major [N/64][batches][rows][64]
};

struct TileCoord {
    int b, m0, n0;
};
TW_DEVINL TileCoord decode_tile(const Params& p, int tile) {
    TileCoord t;
    const int nt = tile % p.n_tiles;
    const int mt_all = tile / p.n_tiles;
    t.b = mt_all / p.m_tiles_per_batch;
    t.m0 = (mt_all - t.b * p.m_tiles_per_batch) * (2 * BM);
    t.n0 = nt * BN;
    return t;
}

// ================================================================================================
// A CLUSTER of two CTAs (one SM pair) owns a 256 x 256 output tile.
//
// One CTA per 128 x 256 tile would move (128 + 256) * K * 2 bytes into shared memory per 2 * 128 * 256 * K FLOP =
// 85 FLOP/B, and at ~64 B/clk per SM of shared-memory fill that caps the chip near 1500 TFLOP/s (measured 1210-1330 on
// the K = 1280 encoder shapes).  Here each CTA loads its own 128 rows of A and only HALF of the B tile (128 of the 256
// output columns); tcgen05.mma.cta_group::2 (issued by the leader CTA only, M = 256) reads A and B from both CTAs'
// shared memory: 128 FLOP/B.  Each CTA keeps the accumulator rows of its own 128 rows in its own TMEM and runs the
// epilogue for them.
//   * TMA loads of both CTAs complete on the LEADER's full barrier (shared::cluster address with the peer bit cleared);
//   * tcgen05.commit multicasts to the empty / accumulator-full barriers of both CTAs;
//   * the epilogue threads of both CTAs arrive on the leader's accumulator-empty barrier (remote mbarrier arrive).
// ================================================================================================
#ifndef GEMM_STAGES2
#define GEMM_STAGES2 6
#endif
constexpr int STAGES2 = GEMM_STAGES2;
constexpr int B2_STAGE_BYTES = 128 * BK * 2;  // half of the B tile: 16 KB
constexpr int SMEM2_BYTES = STAGES2 * (A_STAGE_BYTES + B2_STAGE_BYTES) + 1024 + 256 + EPI_STAGE_BYTES;
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;   // shared::cluster address of the same offset in the even CTA of the pair

TW_DEVINL uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
TW_DEVINL uint32_t cluster_id_x() { uint32_t r; asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r)); return r; }
TW_DEVINL uint32_t num_clusters_x() { uint32_t r; asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r)); return r; }
TW_DEVINL void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
TW_DEVINL void tmem_alloc_2cta(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
}
TW_DEVINL void tmem_relinquish_2cta() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory"); }
TW_DEVINL void tmem_dealloc_2cta(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
TW_DEVINL void tcgen05_mma_f16_2cta(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n"
        :
        : "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives (once all prior MMAs of this thread retired) on the barrier at this offset in BOTH CTAs of the pair
TW_DEVINL void tcgen05_commit_2cta(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::
                     "r"(smem_u32(bar)), "h"((uint16_t)3)
                 : "memory");
}
TW_DEVINL void tma_load_2d_2cta(const CUtensorMap* m, uint64_t* leader_bar, void* dst, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        :
        : "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(leader_bar) & PEER_BIT_MASK), "r"(c0), "r"(c1)
        : "memory");
}
TW_DEVINL void tma_load_3d_2cta(const CUtensorMap* m, uint64_t* leader_bar, void* dst, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        :
        : "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(leader_bar) & PEER_BIT_MASK), "r"(c0), "r"(c1),
          "r"(c2)
        : "memory");
}
TW_DEVINL void mbar_arrive_leader(uint64_t* bar) {   // arrive on the even CTA's copy of this barrier
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & PEER_BIT_MASK) : "memory");
}

// OUT_F32 / HAS_RESID / ACT are compile-time so the epilogue carries no per-element flag tests
template <bool OUT_F32, bool HAS_RESID, int ACT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
gemm_bf16_2cta_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                      const Params p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sA = smem;
    uint8_t* sB = smem + STAGES2 * A_STAGE_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES2 * (A_STAGE_BYTES + B2_STAGE_BYTES));
    uint64_t* full_bar = bars;                           // [STAGES2]  used in the leader only
    uint64_t* empty_bar = bars + STAGES2;                // [STAGES2]  one per CTA (commit multicast)
    uint64_t* tmem_full_bar = bars + 2 * STAGES2;        // [2]        one per CTA (commit multicast)
    uint64_t* tmem_empty_bar = bars + 2 * STAGES2 + 2;   // [2]        leader only, arrivals from both CTAs
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * STAGES2 + 4);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int cluster = (int)cluster_id_x(), n_clusters = (int)num_clusters_x();

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        for (int s = 0; s < STAGES2; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(&tmem_full_bar[s], 1);
            mbar_init(&tmem_empty_bar[s], 2 * EPI_WARPS * 32);
        }
        fence_barrier_init();
    }
    if (warp == 1) {
        tmem_alloc_2cta(tmem_ptr_smem, TMEM_COLS);
        tmem_relinquish_2cta();
    }
    tcgen05_fence_before();
    cluster_sync_all();          // barriers of both CTAs are initialised before any remote arrive / TMA completion
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    if (warp == 0) {
        if (lane == 0) {
            // ===================== TMA producer (both CTAs: own 128 rows of A, own half of B) =====================
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = cluster; tile < p.num_tiles; tile += n_clusters) {
                const TileCoord t = decode_tile(p, tile);
                const int row0 = t.m0 + (int)rank * BM + (p.a_row_off ? p.a_row_off[t.b] : 0);
                for (int kb = 0; kb < p.num_k_blocks; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * (A_STAGE_BYTES + B2_STAGE_BYTES));
                    tma_load_3d_2cta(&tmA, &full_bar[stage], sA + stage * A_STAGE_BYTES, kb * BK, row0, t.b);
                    tma_load_2d_2cta(&tmB, &full_bar[stage], sB + stage * B2_STAGE_BYTES, kb * BK, t.n0 + (int)rank * 128);
                    if (++stage == STAGES2) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && leader) {
            // ===================== MMA issuer (leader CTA only) =====================
            constexpr uint32_t idesc = umma_idesc_bf16(2 * BM, BN, 0, 0);
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int tile = cluster; tile < p.num_tiles; tile += n_clusters) {
                mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1);
                tcgen05_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                for (int kb = 0; kb < p.num_k_blocks; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tcgen05_fence_after();
                    const uint32_t a_addr = smem_u32(sA + stage * A_STAGE_BYTES);
                    const uint32_t b_addr = smem_u32(sB + stage * B2_STAGE_BYTES);
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) {
                        const uint64_t adesc = umma_desc_sw128(a_addr + k * UMMA_K * 2, 16, 1024);
                        const uint64_t bdesc = umma_desc_sw128(b_addr + k * UMMA_K * 2, 16, 1024);
                        tcgen05_mma_f16_2cta(d_tmem, adesc, bdesc, idesc, (kb | k) != 0 ? 1u : 0u);
                    }
                    tcgen05_commit_2cta(&empty_bar[stage]);   // frees the slot in BOTH CTAs when the MMAs retire
                    if (++stage == STAGES2) { stage = 0; phase ^= 1; }
                }
                tcgen05_commit_2cta(&tmem_full_bar[acc]);     // accumulator complete -> epilogue of both CTAs
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ===================== epilogue (warps 2..9 of both CTAs) =====================
        // Two phases per 32-column chunk so that every global access is coalesced:
        //   A  thread = accumulator row: tcgen05.ld 32 fp32 -> its 128-byte row of the warp's smem tile
        //      (16-byte chunks XOR-swizzled by row, conflict-free)
        //   B  8 lanes = one 128-byte row segment: bias, activation, fp32 residual (coalesced 128 B
        //      loads), store (128 B fp32 / 64 B bf16 per row per instruction)
        const int quarter = warp & 3;       // TMEM lane quarter this warp may access
        const int chalf = (warp - 2) >> 2;  // warps 2-5 take column chunks 0-3, warps 6-9 chunks 4-7 of the tile
        float* stage = reinterpret_cast<float*>(smem + STAGES2 * (A_STAGE_BYTES + B2_STAGE_BYTES) + 256) + (warp - 2) * (32 * 32);
        const int sub = lane & 7;    // phase B: 16-byte column chunk within the 32-column chunk
        const int rgrp = lane >> 3;  // phase B: row = rgrp + 4*i
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int tile = cluster; tile < p.num_tiles; tile += n_clusters) {
            const TileCoord t = decode_tile(p, tile);
            mbar_wait(&tmem_full_bar[acc], acc_phase);
            tcgen05_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * BN;
            const int row_base = t.m0 + (int)rank * BM + quarter * 32;
#pragma unroll 1
            for (int c = chalf * (BN / 64); c < (chalf + 1) * (BN / 64); ++c) {
                const int n_base = t.n0 + c * 32;
                if (n_base >= p.N) break;
                uint32_t v[32];
                tmem_ld_32x32b_x32(taddr + c * 32, v);
                tmem_ld_wait();
                {
                    float4* dst = reinterpret_cast<float4*>(stage + lane * 32);
                    const int sw = lane & 7;
#pragma unroll
                    for (int g = 0; g < 8; ++g)
                        dst[g ^ sw] = make_float4(__uint_as_float(v[4 * g]), __uint_as_float(v[4 * g + 1]),
                                                  __uint_as_float(v[4 * g + 2]), __uint_as_float(v[4 * g + 3]));
                }
                __syncwarp();
                const int n = n_base + sub * 4;
                if (n < p.N) {
                    float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (p.bias) bias4 = __ldg(reinterpret_cast<const float4*>(p.bias + n));
                    const int r0 = row_base + rgrp;
                    const float* rp = nullptr;
                    if (HAS_RESID) rp = p.resid + ((size_t)t.b * p.resid_batch_rows + r0) * p.resid_ld + n;
                    size_t o0 = ((size_t)t.b * p.out_batch_rows + p.out_row_off + r0) * p.out_ld + n;
                    size_t out_ld = (size_t)p.out_ld;
                    if (p.out_mode == 1) {
                        o0 = (((size_t)(n >> 6) * p.batches + t.b) * p.rows + r0) * 64 + (n & 63);
                        out_ld = 64;
                    }
                    float* of = reinterpret_cast<float*>(p.out) + o0;
                    __nv_bfloat16* ob = reinterpret_cast<__nv_bfloat16*>(p.out) + o0;
                    const int nrows = p.rows - r0;
                    float4 val[8];
                    float4 res[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int rl = rgrp + 4 * i;
                        val[i] = reinterpret_cast<const float4*>(stage + rl * 32)[sub ^ (rl & 7)];
                        if (HAS_RESID) {
                            res[i] = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (4 * i < nrows) res[i] = *reinterpret_cast<const float4*>(rp + (size_t)(4 * i) * p.resid_ld);
                        }
                    }
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        float4 f = val[i];
                        f.x += bias4.x; f.y += bias4.y; f.z += bias4.z; f.w += bias4.w;
                        if (ACT == 1) {
                            gelu_erf_fast_x2(f.x, f.y);
                            gelu_erf_fast_x2(f.z, f.w);
                        }
                        if (HAS_RESID) { f.x += res[i].x; f.y += res[i].y; f.z += res[i].z; f.w += res[i].w; }
                        if (4 * i < nrows) {
                            if (OUT_F32) {
                                *reinterpret_cast<float4*>(of + (size_t)(4 * i) * out_ld) = f;
                            } else {
                                uint2 pk;
                                pk.x = pack_bf16x2(f.x, f.y);
                                pk.y = pack_bf16x2(f.z, f.w);
                                *reinterpret_cast<uint2*>(ob + (size_t)(4 * i) * out_ld) = pk;
                            }
                        }
                    }
                }
                __syncwarp();
            }
            tcgen05_fence_before();
            mbar_arrive_leader(&tmem_empty_bar[acc]);   // the leader's MMA warp waits for both CTAs' epilogues
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }

    tcgen05_fence_before();
    cluster_sync_all();          // no CTA of the pair may exit (or free TMEM) while the other still uses its smem / TMEM
    if (warp == 1) {
        tcgen05_fence_after();
        tmem_dealloc_2cta(tmem_base, TMEM_COLS);
    }
}

}  // namespace gemm
}  // namespace tw

using namespace tw;
using namespace tw::gemm;

extern "C" int tw_gemm_bf16(const tw_gemm_args* a, void* stream) {
    TW_REQUIRE(a != nullptr, "tw_gemm_bf16: null args");
    TW_REQUIRE(a->a && a->w && a->out, "tw_gemm_bf16: null tensor pointer");
    if (tw::ensure_device(a->a)) return 1;
    TW_REQUIRE(a->batches >= 0 && a->rows >= 0 && a->n > 0 && a->k > 0, "tw_gemm_bf16: bad shape");
    TW_REQUIRE(a->n % 8 == 0 && a->k % 8 == 0, "tw_gemm_bf16: N (%d) and K (%d) must be multiples of 8",
               a->n, a->k);
    TW_REQUIRE(a->a_row_stride % 8 == 0 && a->a_batch_stride % 8 == 0,
               "tw_gemm_bf16: A strides must be multiples of 8 elements (16 B)");
    TW_REQUIRE(((uintptr_t)a->a & 15) == 0 && ((uintptr_t)a->w & 15) == 0 && ((uintptr_t)a->out & 15) == 0,
               "tw_gemm_bf16: pointers must be 16-byte aligned");
    TW_REQUIRE(a->out_ld % 8 == 0, "tw_gemm_bf16: out_ld must be a multiple of 8");
    TW_REQUIRE(!a->resid || (a->resid_ld % 4 == 0 && ((uintptr_t)a->resid & 15) == 0),
               "tw_gemm_bf16: resid must be 16-byte aligned with ld %% 4 == 0");
    TW_REQUIRE(a->act == 0 || a->act == 1, "tw_gemm_bf16: unknown activation %d", a->act);
    TW_REQUIRE(a->out_mode == 0 || (a->out_mode == 1 && a->n % 64 == 0 && a->out_row_off == 0),
               "tw_gemm_bf16: out_mode %d needs N %% 64 == 0 and out_row_off == 0", a->out_mode);
    if (a->batches == 0 || a->rows == 0) return 0;

    CUtensorMap tmA, tmB;
    {
        const int batches = a->batches;
        const uint64_t dims[3] = {(uint64_t)a->k, (uint64_t)a->a_rows, (uint64_t)batches};
        // a size-1 batch dimension still needs a legal (16 B multiple, non-zero) stride
        const uint64_t bstride = (batches > 1 ? (uint64_t)a->a_batch_stride
                                              : (uint64_t)a->a_rows * (uint64_t)a->a_row_stride) * 2;
        const uint64_t strides[2] = {(uint64_t)a->a_row_stride * 2, bstride};
        const uint32_t box[3] = {BK, BM, 1};
        if (encode_tensor_map(&tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, a->a, dims, strides, box,
                              CU_TENSOR_MAP_SWIZZLE_128B))
            return 1;
    }
    {   // each CTA of the pair loads 128 of the tile's 256 output columns
        const uint64_t dims[2] = {(uint64_t)a->k, (uint64_t)a->n};
        const uint64_t strides[1] = {(uint64_t)a->k * 2};
        const uint32_t box[2] = {BK, 128};
        if (encode_tensor_map(&tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, a->w, dims, strides, box,
                              CU_TENSOR_MAP_SWIZZLE_128B))
            return 1;
    }
    Params p;
    p.rows = a->rows;
    p.batches = a->batches;
    p.N = a->n;
    p.K = a->k;
    p.m_tiles_per_batch = (a->rows + 2 * BM - 1) / (2 * BM);
    p.n_tiles = (a->n + BN - 1) / BN;
    p.num_tiles = p.m_tiles_per_batch * p.batches * p.n_tiles;
    p.num_k_blocks = (a->k + BK - 1) / BK;
    p.a_row_off = a->a_row_off;
    p.bias = a->bias;
    p.resid = a->resid;
    p.resid_ld = a->resid_ld;
    p.resid_batch_rows = a->resid_batch_rows;
    p.out = a->out;
    p.out_f32 = a->out_f32;
    p.out_ld = a->out_ld;
    p.out_batch_rows = a->out_batch_rows;
    p.out_row_off = a->out_row_off;
    p.act = a->act;
    p.out_mode = a->out_mode;

    const int sms = num_sms();
    TW_REQUIRE(sms > 0, "tw_gemm_bf16: no CUDA device");
    typedef void (*kern_t)(const CUtensorMap, const CUtensorMap, const Params);
    static const kern_t kernels[8] = {
        gemm_bf16_2cta_kernel<false, false, 0>, gemm_bf16_2cta_kernel<false, false, 1>, gemm_bf16_2cta_kernel<false, true, 0>,
        gemm_bf16_2cta_kernel<false, true, 1>,  gemm_bf16_2cta_kernel<true, false, 0>,  gemm_bf16_2cta_kernel<true, false, 1>,
        gemm_bf16_2cta_kernel<true, true, 0>,   gemm_bf16_2cta_kernel<true, true, 1>};
    static std::atomic<unsigned long long> attr_done{0};
    if (device_needs_setup(attr_done)) {
        for (int i = 0; i < 8; ++i)
            TW_CUDA_CHECK(cudaFuncSetAttribute(kernels[i], cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM2_BYTES));
        mark_device_done(attr_done);
    }
    const int clusters = p.num_tiles < sms / 2 ? p.num_tiles : sms / 2;
    const kern_t k = kernels[(p.out_f32 ? 4 : 0) + (p.resid ? 2 : 0) + (p.act ? 1 : 0)];
    k<<<2 * clusters, NUM_THREADS, SMEM2_BYTES, (cudaStream_t)stream>>>(tmA, tmB, p);
    TW_CUDA_CHECK(cudaGetLastError());
    return 0;
}
