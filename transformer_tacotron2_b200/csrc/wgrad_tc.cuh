// Weight-gradient GEMM on tcgen05 / TMEM / TMA (training path, SURVEY.md 8(a) a12):
//     dW[n][k * taps + tap] += sum_{b, t} dY[b, t, n] * X[b, t + tap - pad, k]          (the reduction runs over TOKENS)
// Both operands are read straight from the row-major activations [tokens][features] as MN-major UMMA operands (the feature
// dimension is contiguous, the reduction dimension is the row index): TMA boxes {64 features, 64 tokens} with 128B swizzle,
// two boxes per 128-wide operand tile (LBO = 8 KB between them) -- no transposed copies of dY or X are ever made.  The
// conv taps shift the token coordinate of X inside the utterance's own 3-D slice (TMA zero-fills outside), as in gemm_tc.cuh.
// The output is tiny (<= 6144 x 512) while the reduction is long (25.6k-51.2k tokens), so every output tile is split along
// the token axis (split-K) to fill the 148 SMs; partial tiles are added with red.global.add.f32 into the zeroed gradient
// buffer.  Persistent CTAs, 192 threads (TMA warp / MMA warp / 4 epilogue warps), double-buffered TMEM accumulator.
// The bias gradient (column sums of dY) rides along: the items of the first n-tile / tap issue one extra N = 16 MMA per
// k-step against a tile of ones, so db = dY^T . 1 comes out of the tensor pipe into 16 spare TMEM columns.
#pragma once
#include <cuda.h>
#include "common.cuh"
#include "gemm_tc.cuh"
#include "attention_bwd_tc.cuh"     // fb_desc_mn

namespace tts {

struct WgradParams {
    const bf16* dY; int ldy; int Cout;
    const bf16* X; int ldx; int Cin;
    int taps, T, nb;                  // rows per utterance, utterances (M = nb * T)
    float* dW;                        // [Cout][Cin * taps] fp32, accumulated
    float* dbias;                     // optional [Cout]: += column sums of dY (by the n-tile 0 / tap 0 items, via a ones-tile MMA)
};

struct WgradTcParams {
    alignas(64) CUtensorMap tm_dy, tm_x;     // bf16 {C, T, nb}, box {64, 64, 1}, SWIZZLE_128B
    alignas(64) CUtensorMap tm_dw;           // fp32 {Cin, Cout}, box {32, 32}, SWIZZLE_128B: TMA reduce-add of the partial tiles (taps == 1)
    int tma_red;
    WgradParams g;
    int tiles_m, tiles_n, n_tiles;           // output tiles: Cout/128 x Cin/128 x taps
    int kb_per_utt, n_kb, splits, kb_per_split, n_items;
};

constexpr int WG_STAGES = 4, WG_STAGE_BYTES = 32768, WG_THREADS = 192;
constexpr int WG_SMEM_BYTES = WG_STAGES * WG_STAGE_BYTES + 2048 + 4 * 4096 + 256;    // ring + ones tile + output staging + barriers
constexpr uint32_t WG_IDESC_ONES = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(16 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
constexpr uint32_t WG_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);

__global__ void __launch_bounds__(WG_THREADS, 1) wgrad_tc_kernel(const __grid_constant__ WgradTcParams p) {
    extern __shared__ __align__(1024) unsigned char wg_smem[];
    unsigned char* ones = wg_smem + WG_STAGES * WG_STAGE_BYTES;         // [16 tokens][64 features] of bf16 1.0
    unsigned char* ostage = ones + 2048;                                // [4 epilogue warps][32 rows x 128 B], 128B-swizzled
    uint64_t* full = reinterpret_cast<uint64_t*>(ostage + 4 * 4096);
    uint64_t* empty = full + WG_STAGES;
    uint64_t* tmem_full = empty + WG_STAGES;
    uint64_t* tmem_empty = tmem_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const WgradParams& g = p.g;
    const int pad = g.taps >> 1;

    for (int i = threadIdx.x; i < 512; i += WG_THREADS) reinterpret_cast<uint32_t*>(ones)[i] = 0x3F803F80u;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (threadIdx.x == 0) {
        if (tc_smem_u32(wg_smem) & 1023) __trap();
        for (int s = 0; s < WG_STAGES; ++s) { tc_mbar_init(&full[s], 1); tc_mbar_init(&empty[s], 1); }
        for (int a = 0; a < 2; ++a) { tc_mbar_init(&tmem_full[a], 1); tc_mbar_init(&tmem_empty[a], 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem_u32(tmem_slot)), "r"(512) : "memory");   // 2 x 128 dW + 2 x 16 db columns
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    // item -> (split, tile) with the TILE index fastest: the CTAs running at the same time work on the same token range, so a
    // block of dY / X rows is fetched from HBM once and the other tiles' CTAs hit it in L2 (tile-major order re-read every
    // operand tiles_n / tiles_m times from HBM: 840 MB for the 2048 x 512 FFN gradient).  tile -> (mt, nt, tap); split -> [kb0, kb1)
    if (warp == 0) {
        if (lane == 0) {                                 // ---------------- TMA producer
            uint32_t it = 0;
            for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
                const int sp = item / p.n_tiles, tile = item - sp * p.n_tiles;
                const int tap = tile % g.taps, nt = (tile / g.taps) % p.tiles_n, mt = tile / (g.taps * p.tiles_n);
                const int kb0 = sp * p.kb_per_split, kb1 = min(p.n_kb, kb0 + p.kb_per_split);
                for (int kb = kb0; kb < kb1; ++kb, ++it) {
                    const int s = it % WG_STAGES; const uint32_t use = it / WG_STAGES;
                    if (use > 0) tc_mbar_wait(&empty[s], (use & 1) ^ 1);
                    const int b = kb / p.kb_per_utt, t0 = (kb - b * p.kb_per_utt) * 64;
                    unsigned char* dst = wg_smem + s * WG_STAGE_BYTES;
                    tc_mbar_expect_tx(&full[s], WG_STAGE_BYTES);
                    tc_tma_3d(dst, &p.tm_dy, mt * 128, t0, b, &full[s]);
                    tc_tma_3d(dst + 8192, &p.tm_dy, mt * 128 + 64, t0, b, &full[s]);
                    tc_tma_3d(dst + 16384, &p.tm_x, nt * 128, t0 + tap - pad, b, &full[s]);
                    tc_tma_3d(dst + 24576, &p.tm_x, nt * 128 + 64, t0 + tap - pad, b, &full[s]);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {                                 // ---------------- MMA issuer
            uint32_t it = 0, j = 0;
            for (int item = blockIdx.x; item < p.n_items; item += gridDim.x, ++j) {
                const int sp = item / p.n_tiles, tile = item - sp * p.n_tiles;
                const bool do_bias = g.dbias && (tile % (g.taps * p.tiles_n)) == 0;      // first n-tile, tap 0
                const int kb0 = sp * p.kb_per_split, kb1 = min(p.n_kb, kb0 + p.kb_per_split);
                const uint32_t acc = j & 1, ause = j >> 1;
                const uint32_t ones_addr = tc_smem_u32(ones);
                if (ause > 0) tc_mbar_wait(&tmem_empty[acc], (ause & 1) ^ 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t d_tmem = tmem_base + acc * 128;
                for (int kb = kb0; kb < kb1; ++kb, ++it) {
                    const int s = it % WG_STAGES; const uint32_t use = it / WG_STAGES;
                    tc_mbar_wait(&full[s], use & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t a_addr = tc_smem_u32(wg_smem + s * WG_STAGE_BYTES), b_addr = a_addr + 16384;
#pragma unroll
                    for (int k = 0; k < 4; ++k)          // 16 tokens per MMA = 16 rows x 128 B inside each box
                        ft_mma(d_tmem, fb_desc_mn(a_addr + k * 2048, 8192), fb_desc_mn(b_addr + k * 2048, 8192), WG_IDESC, (kb > kb0) || k != 0);
                    if (do_bias) {
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            ft_mma(tmem_base + 256 + acc * 16, fb_desc_mn(a_addr + k * 2048, 8192), fb_desc_mn(ones_addr, 16), WG_IDESC_ONES, (kb > kb0) || k != 0);
                    }
                    ft_commit(&empty[s]);
                }
                ft_commit(&tmem_full[acc]);
            }
        }
    } else {                                             // ---------------- epilogue: thread = output row n (a dY feature)
        const int lg = warp & 3;
        uint32_t j = 0;
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x, ++j) {
            const int sp = item / p.n_tiles, tile = item - sp * p.n_tiles;
            const int tap = tile % g.taps, nt = (tile / g.taps) % p.tiles_n, mt = tile / (g.taps * p.tiles_n);
            const int kb0 = sp * p.kb_per_split;
            const uint32_t acc = j & 1;
            const bool nonempty = kb0 < p.n_kb;
            if (nonempty) {
                tc_mbar_wait(&tmem_full[acc], (j >> 1) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            }
            const int n = mt * 128 + lg * 32 + lane;
            const int ldo = g.Cin * g.taps;
            if (nonempty && g.dbias && nt == 0 && tap == 0) {                            // db[n] += sum_tokens dY[token][n]
                uint32_t bv[16];
                asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                             : "=r"(bv[0]), "=r"(bv[1]), "=r"(bv[2]), "=r"(bv[3]), "=r"(bv[4]), "=r"(bv[5]), "=r"(bv[6]), "=r"(bv[7]),
                               "=r"(bv[8]), "=r"(bv[9]), "=r"(bv[10]), "=r"(bv[11]), "=r"(bv[12]), "=r"(bv[13]), "=r"(bv[14]), "=r"(bv[15])
                             : "r"(tmem_base + 256 + acc * 16 + ((uint32_t)(lg * 32) << 16)));
                ft_ld_wait();
                if (n < g.Cout) atomicAdd(g.dbias + n, __uint_as_float(bv[0]));
            }
#pragma unroll 1
            for (int c0 = 0; c0 < 128; c0 += 32) {
                uint32_t v[32];
                if (nonempty) {
                    ft_ld32_nowait(tmem_base + acc * 128 + ((uint32_t)(lg * 32) << 16) + (uint32_t)c0, v);
                    ft_ld_wait();
                    if (n < g.Cout) {
                        const int kcol = nt * 128 + c0;
                        float* o = g.dW + (size_t)n * ldo;
                        if (p.tma_red) {
                            // handled below by the whole warp (rows past Cout / columns past Cin are clipped by the tensor map)
                        } else {                     // any layout or alignment of dW (Cin % 4 != 0, taps > 1, dW not 16-byte aligned)
#pragma unroll
                            for (int i = 0; i < 32; ++i)
                                if (kcol + i < g.Cin) atomicAdd(o + (size_t)(kcol + i) * g.taps + tap, __uint_as_float(v[i]));
                        }
                    }
                    if (p.tma_red && nt * 128 + c0 < g.Cin) {
                        // one TMA reduce-add per 32 x 32 chunk instead of 32 per-row red instructions (32 request lines each)
                        unsigned char* st = ostage + (warp - 2) * 4096;
                        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
                        __syncwarp();
#pragma unroll
                        for (int q = 0; q < 8; ++q)
                            *reinterpret_cast<uint4*>(st + lane * 128 + ((q ^ (lane & 7)) << 4)) = make_uint4(v[q * 4], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        __syncwarp();
                        if (lane == 0) {
                            asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%1, %2}], [%3];"
                                         ::"l"(&p.tm_dw), "r"(nt * 128 + c0), "r"(mt * 128 + lg * 32), "r"(tc_smem_u32(st)) : "memory");
                            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                        }
                    }
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0 && nonempty) ft_arrive(&tmem_empty[acc]);
        }
    }
    if (warp >= 2 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
    }
}

inline cudaError_t launch_wgrad_tc(const WgradParams& g, cudaStream_t stream) {
    static PerDevice pd;
    int num_sms = 0;
    {
        const cudaError_t e = per_device_once(pd, &num_sms, [] {
            return cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, WG_SMEM_BYTES);
        });
        if (e != cudaSuccess) return e;
    }
    TcEncodeFn enc = tc_encode_fn();
    if (!enc || (g.ldy & 7) || (g.ldx & 7)) return cudaErrorInvalidValue;
    WgradTcParams p;
    p.g = g;
    auto make = [&](CUtensorMap* tm, const bf16* base, int C, int ld) -> bool {
        const cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)g.T, (cuuint64_t)g.nb};
        const cuuint64_t strides[2] = {(cuuint64_t)ld * 2, (cuuint64_t)ld * 2 * g.T};
        const cuuint32_t box[3] = {64, 64, 1};
        const cuuint32_t estr[3] = {1, 1, 1};
        return enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<bf16*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
    };
    if (!make(&p.tm_dy, g.dY, g.Cout, g.ldy) || !make(&p.tm_x, g.X, g.Cin, g.ldx)) return cudaErrorInvalidValue;
    p.tma_red = 0;
    if (g.taps == 1 && (g.Cin & 3) == 0 && (reinterpret_cast<uintptr_t>(g.dW) & 15) == 0) {
        const cuuint64_t dims[2] = {(cuuint64_t)g.Cin, (cuuint64_t)g.Cout};
        const cuuint64_t strides[1] = {(cuuint64_t)g.Cin * 4};
        const cuuint32_t box[2] = {32, 32};
        const cuuint32_t estr[2] = {1, 1};
        if (enc(&p.tm_dw, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, g.dW, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS)
            p.tma_red = 1;
    }
    p.tiles_m = (g.Cout + 127) / 128; p.tiles_n = (g.Cin + 127) / 128;
    p.n_tiles = p.tiles_m * p.tiles_n * g.taps;
    p.kb_per_utt = (g.T + 63) / 64; p.n_kb = p.kb_per_utt * g.nb;
    // split-K factor: enough items to fill the SMs (>= ~2 per SM), at least 4 token blocks per item, and a total that
    // lands just under a whole number of waves (a 2.2-wave launch wastes a quarter of the machine)
    const int max_splits = std::max(1, (p.n_kb + 3) / 4);
    int splits = 1; double best = -1.0;
    for (int sp = 1; sp <= max_splits && sp <= 64; ++sp) {
        const int kbs = (p.n_kb + sp - 1) / sp, real = (p.n_kb + kbs - 1) / kbs;
        const long items = (long)p.n_tiles * real;
        const long waves = (items + num_sms - 1) / num_sms;
        double eff = (double)items / (double)(waves * num_sms);
        if (items < 2L * num_sms) eff *= (double)items / (2.0 * num_sms);   // too few items: pipeline prologue / epilogue exposed
        eff -= 0.004 * real;                                                // every split adds one round of atomics
        if (eff > best) { best = eff; splits = real; }
    }
    p.kb_per_split = (p.n_kb + splits - 1) / splits;
    p.splits = (p.n_kb + p.kb_per_split - 1) / p.kb_per_split;
    p.n_items = p.n_tiles * p.splits;
    const int grid = std::min(p.n_items, num_sms);
    wgrad_tc_kernel<<<grid, WG_THREADS, WG_SMEM_BYTES, stream>>>(p);
    ++launch_counter();
    return cudaGetLastError();
}

}  // namespace tts
