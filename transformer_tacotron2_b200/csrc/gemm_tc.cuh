// tcgen05 / TMEM / TMA GEMM for the sequence-parallel path (SURVEY.md 8(a) rows a3, a4, a10; component C12):
//     C[m, n] = epi( sum_tap sum_k A[b, t + tap - pad, k] * W[tap][n, k] ),   m = b * T + t
// i.e. plain GEMMs (taps = 1, T = M) and conv1d(k = 5, pad = 2) as 5 row-shifted GEMMs accumulated into ONE
// TMEM accumulator; rows outside [0, T) of their own utterance are zero-filled by TMA's out-of-bounds handling
// (the A operand is a 3-D tensor map {channels, frames, utterances}), so no padded copies exist.
// Structure (persistent: one CTA per SM walks 128 x 128 output tiles; 320 threads; the TMEM accumulator is double-buffered
// so the epilogue of tile i overlaps the mainloop of tile i+1):
//   warp 0  : TMA producer      cp.async.bulk.tensor -> 4-stage shared-memory ring (128B swizzle), mbarrier full/empty
//   warp 1  : MMA issuer        one elected lane issues tcgen05.mma.cta_group::1.kind::f16 (M128 N128 K16), accumulator
//                               in TMEM (128 fp32 columns); tcgen05.commit releases ring slots / signals the epilogue
//   warps 2-9: epilogue         tcgen05.ld 32x32b (thread = output row) -> fused epilogue of gemm_epilogue.cuh (bias, BN fold,
//                               ReLU / tanh, residual, alpha*PE, length mask, Philox dropout, KV scatter, head split)
#pragma once
#include <cuda.h>
#include "common.cuh"
#include "gemm_epilogue.cuh"
#include "philox.cuh"

namespace tts {

constexpr int TC_BM = 128, TC_BK = 64, TC_STAGES = 4;     // N tile: 256 (default) or 128 (template parameter BN)
constexpr int TC_EPI_WARPS = 8;                                           // two warps per TMEM lane quarter, half of the columns each
__host__ __device__ constexpr int tc_stage_bytes(int BN) { return (TC_BM + BN) * TC_BK * 2; }      // 48 KB / 32 KB
__host__ __device__ constexpr int tc_smem_bytes(int BN) { return TC_STAGES * tc_stage_bytes(BN) + TC_EPI_WARPS * 4096 + 1024 + 256; }   // ring + output staging + alignment slack + barriers
constexpr int TC_THREADS = 64 + 32 * TC_EPI_WARPS;

struct GemmTcParams {
    alignas(64) CUtensorMap tm_a;     // bf16 {K (inner), T, B}, box {64, 128, 1}, SWIZZLE_128B
    alignas(64) CUtensorMap tm_w;     // bf16 {K (inner), taps * Nw}, box {64, 128}, SWIZZLE_128B
    alignas(64) CUtensorMap tm_out;   // output {N (inner), T, B}: fp32 box {32, 32, 1} / bf16 box {64, 32, 1}, SWIZZLE_128B (TMA store)
    int tma_out;                      // 0 = direct stores, 1 = fp32 via TMA store, 2 = bf16 via TMA store
    GemmParams g;                     // shapes + epilogue (A / W pointers unused here)
    int Tl;                           // rows per A-tensor slab: T for convs (taps > 1), M for plain GEMMs
    int tiles_per_utt;                // ceil(Tl / 128)
    int n_tiles_n, n_tiles;           // tiles along N; total tiles (persistent CTAs walk tile = blockIdx.x + i * gridDim.x)
};

TTS_D uint32_t tc_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
TTS_D void tc_mbar_init(uint64_t* bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tc_smem_u32(bar)), "r"(count) : "memory"); }
TTS_D void tc_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tc_smem_u32(bar)), "r"(bytes) : "memory");
}
TTS_D void tc_mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok = 0;
    while (!ok)
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(tc_smem_u32(bar)), "r"(parity) : "memory");
}
TTS_D void tc_tma_3d(void* dst, const CUtensorMap* tm, int c0, int c1, int c2, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"(tc_smem_u32(dst)), "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(tc_smem_u32(bar)) : "memory");
}
TTS_D void tc_tma_2d(void* dst, const CUtensorMap* tm, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(tc_smem_u32(dst)), "l"(tm), "r"(c0), "r"(c1), "r"(tc_smem_u32(bar)) : "memory");
}
// K-major operand tile [rows][64 bf16] written by TMA with 128-byte swizzle: 8-row atoms of 1024 B (SBO = 1024 B),
// LBO unused (1), descriptor version 1 (sm_100), layout type 2 (SWIZZLE_128B)  -- cute::UMMA::SmemDescriptor
TTS_D uint64_t tc_smem_desc(uint32_t smem_addr) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFF) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// kind::f16 instruction descriptor: D = f32 (bits 4-5 = 1), A = B = bf16 (bits 7-9 = 1, 10-12 = 1), both K-major,
// N >> 3 at bits 17-22, M >> 4 at bits 24-28  -- cute::UMMA::InstrDescriptor
__host__ __device__ constexpr uint32_t tc_idesc(int BN) { return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24); }

template <int BN>
__global__ void __launch_bounds__(TC_THREADS, 1) gemm_tc_kernel(const __grid_constant__ GemmTcParams p) {
    constexpr int TC_BN = BN, TC_STAGE_BYTES = tc_stage_bytes(BN);
    constexpr uint32_t TC_IDESC = tc_idesc(BN);
    extern __shared__ unsigned char tc_smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(tc_smem_raw) + 1023) & ~(uintptr_t)1023);
    unsigned char* ostage = smem + TC_STAGES * TC_STAGE_BYTES;          // [TC_EPI_WARPS][4 KB] output staging for the TMA stores
    uint64_t* full = reinterpret_cast<uint64_t*>(ostage + TC_EPI_WARPS * 4096);
    uint64_t* empty = full + TC_STAGES;
    uint64_t* tmem_full = empty + TC_STAGES;             // [2]
    uint64_t* tmem_empty = tmem_full + 2;                // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const GemmParams& g = p.g;
    const int kblocks = (g.K + TC_BK - 1) / TC_BK, nk = kblocks * g.taps, pad = g.taps >> 1;

    if (threadIdx.x == 0) {
        for (int s = 0; s < TC_STAGES; ++s) { tc_mbar_init(&full[s], 1); tc_mbar_init(&empty[s], 1); }
        for (int a = 0; a < 2; ++a) { tc_mbar_init(&tmem_full[a], 1); tc_mbar_init(&tmem_empty[a], TC_EPI_WARPS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&p.tm_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&p.tm_w) : "memory");
    }
    if (warp == 1) {                                     // TMEM: 2 x 128 columns x 128 lanes fp32 (double-buffered accumulator)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem_u32(tmem_slot)), "r"(2 * TC_BN) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {                                 // ---------------- TMA producer
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
                const int mt = tile / p.n_tiles_n, n0 = (tile - mt * p.n_tiles_n) * TC_BN;
                const int b = mt / p.tiles_per_utt, t0 = (mt - b * p.tiles_per_utt) * TC_BM;
                for (int i = 0; i < nk; ++i, ++it) {
                    const int s = it % TC_STAGES; const uint32_t use = it / TC_STAGES;
                    if (use > 0) tc_mbar_wait(&empty[s], (use & 1) ^ 1);
                    const int tap = i / kblocks, kc = (i - tap * kblocks) * TC_BK;
                    unsigned char* a_dst = smem + s * TC_STAGE_BYTES;
                    tc_mbar_expect_tx(&full[s], TC_STAGE_BYTES);
                    tc_tma_3d(a_dst, &p.tm_a, kc, t0 + tap - pad, b, &full[s]);        // rows outside [0, T): zero fill
                    tc_tma_2d(a_dst + TC_BM * TC_BK * 2, &p.tm_w, kc, tap * g.Nw + n0, &full[s]);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {                                 // ---------------- MMA issuer
            uint32_t it = 0, j = 0;
            for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++j) {
                const uint32_t acc = j & 1, ause = j >> 1;
                if (ause > 0) tc_mbar_wait(&tmem_empty[acc], (ause & 1) ^ 1);           // epilogue drained this accumulator
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t d_tmem = tmem_base + acc * TC_BN;
                for (int i = 0; i < nk; ++i, ++it) {
                    const int s = it % TC_STAGES; const uint32_t use = it / TC_STAGES;
                    tc_mbar_wait(&full[s], use & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t a_addr = tc_smem_u32(smem + s * TC_STAGE_BYTES), b_addr = a_addr + TC_BM * TC_BK * 2;
#pragma unroll
                    for (int k = 0; k < TC_BK / 16; ++k) {   // advance 32 bytes (16 bf16) inside the 128-byte swizzle atom
                        const uint64_t da = tc_smem_desc(a_addr + k * 32), db = tc_smem_desc(b_addr + k * 32);
                        const uint32_t accum = (i | k) != 0;
                        asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                                     ::"r"(d_tmem), "l"(da), "l"(db), "r"(TC_IDESC), "r"(accum) : "memory");
                    }
                    // commit: the slot is free again once these MMAs have read it (implies fence::before_thread_sync)
                    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem_u32(&empty[s])) : "memory");
                }
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem_u32(&tmem_full[acc])) : "memory");
            }
        }
    } else {                                             // ---------------- epilogue warps 2..9
        const int lg = warp & 3;                         // TMEM lane group this warp may access: lanes 32*lg .. 32*lg+31
        const int chalf = (warp - 2) >> 2;               // which half of the tile's columns (the epilogue is latency-bound: 8 warps halve it)
        uint32_t j = 0;
        for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++j) {
        const int mt = tile / p.n_tiles_n, n0 = (tile - mt * p.n_tiles_n) * TC_BN;
        const int b = mt / p.tiles_per_utt, t0 = (mt - b * p.tiles_per_utt) * TC_BM;
        const uint32_t acc = j & 1;
        // bias of this warp's 128 columns: 4 per lane, fetched once per tile while the MMAs run (a per-chunk __ldg put an L2
        // round trip into every chunk's dependency chain); the chunks pick their values up by shuffle
        float4 bq = make_float4(0.f, 0.f, 0.f, 0.f);
        if (g.bias) {
            const int bc = n0 + chalf * (TC_BN / 2) + lane * 4;
            if (lane * 4 >= TC_BN / 2) { /* this lane's columns belong to the other warp */ }
            else if (bc + 3 < g.N) bq = __ldg(reinterpret_cast<const float4*>(g.bias + bc));
            else { if (bc < g.N) bq.x = g.bias[bc]; if (bc + 1 < g.N) bq.y = g.bias[bc + 1]; if (bc + 2 < g.N) bq.z = g.bias[bc + 2]; }
        }
        tc_mbar_wait(&tmem_full[acc], (j >> 1) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int t = t0 + lg * 32 + lane;
        const int m = b * p.Tl + t;
#pragma unroll 1
        for (int c0 = chalf * (TC_BN / 2); c0 < (chalf + 1) * (TC_BN / 2); c0 += 32) {
            uint32_t v[32];
            const uint32_t taddr = tmem_base + acc * TC_BN + ((uint32_t)(lg * 32) << 16) + (uint32_t)c0;
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
                         "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                         : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                           "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                           "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                           "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                         : "r"(taddr));
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            {
                const int nb0 = n0 + c0;
                const bool rvalid = t < p.Tl && m < g.M;
                const bool vec = g.scatter == SC_NONE && nb0 + 32 <= g.N && (g.ldo & 7) == 0 && (g.ldr & 7) == 0;      // warp-uniform
                if (!vec) {
                    if (rvalid) {
#pragma unroll
                        for (int j = 0; j < 32; j += 2)
                            gemm_store(g, m, nb0 + j, __uint_as_float(v[j]), __uint_as_float(v[j + 1]));
                    }
                } else {                                 // thread = one output row: 32 consecutive columns
                    float f[32];
                    {
                        const int src0 = (c0 - chalf * (TC_BN / 2)) >> 2;      // lane holding the bias of this chunk's first 4 columns
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            f[j] = __uint_as_float(v[j]) + __shfl_sync(0xffffffffu, bq.x, src0 + (j >> 2));
                            f[j + 1] = __uint_as_float(v[j + 1]) + __shfl_sync(0xffffffffu, bq.y, src0 + (j >> 2));
                            f[j + 2] = __uint_as_float(v[j + 2]) + __shfl_sync(0xffffffffu, bq.z, src0 + (j >> 2));
                            f[j + 3] = __uint_as_float(v[j + 3]) + __shfl_sync(0xffffffffu, bq.w, src0 + (j >> 2));
                        }
                    }
                    if (rvalid) {
                        const int bb = m / g.T, tt = m - bb * g.T;
                        const uint64_t seed = g.seed_ptr ? *g.seed_ptr : g.seed;
                        if (g.pe) {
                            const float alpha = g.alpha_ptr ? *g.alpha_ptr : g.alpha;
#pragma unroll
                            for (int j = 0; j < 32; j += 4) {
                                const float4 pv = __ldg(reinterpret_cast<const float4*>(g.pe + (size_t)tt * kDModel + nb0 + j));
                                f[j] += alpha * pv.x; f[j + 1] += alpha * pv.y; f[j + 2] += alpha * pv.z; f[j + 3] += alpha * pv.w;
                            }
                        }
                        if (g.dropw_site >= 0) {             // word dropout (P12): 4 consecutive columns = one Philox call
#pragma unroll
                            for (int j = 0; j < 32; j += 4) {
                                const uint4 w4 = philox4x32_10(make_uint4((uint32_t)g.dropw_site, (uint32_t)tt, (uint32_t)(g.utt_offset + bb), (uint32_t)((nb0 + j) >> 2)),
                                                               (uint32_t)seed, (uint32_t)(seed >> 32));
                                f[j] = w4.x >= g.dropw_thresh ? f[j] * g.dropw_scale : 0.f;
                                f[j + 1] = w4.y >= g.dropw_thresh ? f[j + 1] * g.dropw_scale : 0.f;
                                f[j + 2] = w4.z >= g.dropw_thresh ? f[j + 2] * g.dropw_scale : 0.f;
                                f[j + 3] = w4.w >= g.dropw_thresh ? f[j + 3] * g.dropw_scale : 0.f;
                            }
                        }
                        if (g.resid_bf16) {
#pragma unroll
                            for (int j = 0; j < 32; j += 8) {
                                const uint4 rv = *reinterpret_cast<const uint4*>(g.resid_bf16 + (size_t)m * g.ldr + nb0 + j);
                                const float2 r0 = unpack_bf16x2(rv.x), r1 = unpack_bf16x2(rv.y), r2 = unpack_bf16x2(rv.z), r3 = unpack_bf16x2(rv.w);
                                f[j] += r0.x; f[j + 1] += r0.y; f[j + 2] += r1.x; f[j + 3] += r1.y;
                                f[j + 4] += r2.x; f[j + 5] += r2.y; f[j + 6] += r3.x; f[j + 7] += r3.y;
                            }
                        }
                        if (g.resid_f32) {
#pragma unroll
                            for (int j = 0; j < 32; j += 4) {
                                const float4 rv = *reinterpret_cast<const float4*>(g.resid_f32 + (size_t)m * g.ldr + nb0 + j);
                                f[j] += rv.x; f[j + 1] += rv.y; f[j + 2] += rv.z; f[j + 3] += rv.w;
                            }
                        }
                        if (g.act == ACT_RELU) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) f[j] = fmaxf(f[j], 0.f);
                        } else if (g.act == ACT_TANH) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) f[j] = tanhf(f[j]);
                        }
                        if (g.drop_site >= 0) {              // 32 aligned columns = one Philox word (P16)
                            const uint4 w4 = philox4x32_10(make_uint4((uint32_t)g.drop_site, (uint32_t)tt, (uint32_t)(g.utt_offset + bb), (uint32_t)(nb0 >> 7)),
                                                           (uint32_t)seed, (uint32_t)(seed >> 32));
                            const uint32_t wi = (nb0 >> 5) & 3u;
                            const uint32_t bits = wi == 0 ? w4.x : wi == 1 ? w4.y : wi == 2 ? w4.z : w4.w;
#pragma unroll
                            for (int j = 0; j < 32; ++j) f[j] = ((bits >> j) & 1u) ? 2.f * f[j] : 0.f;
                        }
                        if (g.lens && tt >= g.lens[bb]) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) f[j] = 0.f;
                        }
                    }
                    // Output: a thread-per-row store instruction touches 32 different lines (32 L1->XBAR requests); instead the
                    // warp writes its 32 x 128-byte chunk into 128B-swizzled staging and one lane issues a TMA tensor store
                    // (rows past T / M are clipped by the tensor map).  bf16: two 32-column chunks share one 128-byte-wide box.
                    const int half = (c0 >> 5) & 1;
                    const bool use_tma = p.tma_out == 1 || (p.tma_out == 2 && n0 + (c0 & ~63) + 64 <= g.N);
                    if (use_tma) {
                        unsigned char* st = ostage + (warp - 2) * 4096 + lane * 128;
                        if (p.tma_out == 1 || half == 0) {
                            if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");       // previous store has read the staging
                            __syncwarp();
                        }
                        if (p.tma_out == 1) {
#pragma unroll
                            for (int q = 0; q < 8; ++q)
                                *reinterpret_cast<float4*>(st + ((q ^ (lane & 7)) << 4)) = make_float4(f[q * 4], f[q * 4 + 1], f[q * 4 + 2], f[q * 4 + 3]);
                        } else {
#pragma unroll
                            for (int q = 0; q < 4; ++q)
                                *reinterpret_cast<uint4*>(st + (((half * 4 + q) ^ (lane & 7)) << 4)) =
                                    make_uint4(pack_bf16x2(f[q * 8], f[q * 8 + 1]), pack_bf16x2(f[q * 8 + 2], f[q * 8 + 3]), pack_bf16x2(f[q * 8 + 4], f[q * 8 + 5]), pack_bf16x2(f[q * 8 + 6], f[q * 8 + 7]));
                        }
                        if (p.tma_out == 1 || half == 1) {
                            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                            __syncwarp();
                            if (lane == 0) {
                                asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%1, %2, %3}], [%4];"
                                             ::"l"(&p.tm_out), "r"(p.tma_out == 1 ? nb0 : nb0 - 32), "r"(t0 + lg * 32), "r"(b), "r"(tc_smem_u32(ostage + (warp - 2) * 4096)) : "memory");
                                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                            }
                        }
                    } else if (rvalid) {
                        if (g.out_f32) {
#pragma unroll
                            for (int j = 0; j < 32; j += 4)
                                *reinterpret_cast<float4*>(g.out_f32 + (size_t)m * g.ldo + nb0 + j) = make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
                        }
                        if (g.out_bf16) {
#pragma unroll
                            for (int j = 0; j < 32; j += 8)
                                *reinterpret_cast<uint4*>(g.out_bf16 + (size_t)m * g.ldo + nb0 + j) =
                                    make_uint4(pack_bf16x2(f[j], f[j + 1]), pack_bf16x2(f[j + 2], f[j + 3]), pack_bf16x2(f[j + 4], f[j + 5]), pack_bf16x2(f[j + 6], f[j + 7]));
                        }
                    }
                }
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc_smem_u32(&tmem_empty[acc])) : "memory");   // accumulator free
        }
    }
    if (warp >= 2 && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");      // this warp's TMA stores are complete
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(2 * TC_BN) : "memory");
    }
}

// host side ---------------------------------------------------------------------------------------------------------
typedef CUresult (*TcEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline TcEncodeFn tc_encode_fn() {
    static TcEncodeFn fn = nullptr;
    if (!fn) {
        void* f = nullptr; cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<TcEncodeFn>(f);
    }
    return fn;
}

// Same contract as launch_gemm (gemm_epilogue.cuh): g.A / g.W are bf16 row-major, lda / ldw in elements (multiples of 8),
// W has taps * Nw rows (Nw = N rounded up to 128).  Returns cudaErrorInvalidValue for shapes it cannot describe.
inline cudaError_t launch_gemm_tc(const GemmParams& g, cudaStream_t stream) {
    static PerDevice pd;
    int num_sms = 0;
    {
        const cudaError_t e = per_device_once(pd, &num_sms, [] {
            cudaError_t e2 = cudaFuncSetAttribute(gemm_tc_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem_bytes(256));
            if (e2 == cudaSuccess) e2 = cudaFuncSetAttribute(gemm_tc_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc_smem_bytes(128));
            return e2;
        });
        if (e != cudaSuccess) return e;
    }
    TcEncodeFn enc = tc_encode_fn();
    if (!enc || (g.lda & 7) || (g.ldw & 7) || (g.M % g.T) != 0) return cudaErrorInvalidValue;
    GemmTcParams p;
    p.g = g;
    p.Tl = g.taps > 1 ? g.T : g.M;                       // plain GEMMs ignore the utterance structure when loading A
    const int nb = g.M / p.Tl;
    p.tiles_per_utt = (p.Tl + TC_BM - 1) / TC_BM;
    // N tile: 256 columns halve the operand traffic per FLOP; 128 when that would leave SMs idle (small M: the encoder) or
    // when N itself is narrow (80 / 81 / 128-wide outputs)
    const int m_tiles = nb * p.tiles_per_utt;
    const int TC_BN = (g.N <= 128 || (long)m_tiles * ((g.N + 255) / 256) < num_sms) ? 128 : 256;
    const cuuint32_t estr[3] = {1, 1, 1};
    {
        const cuuint64_t dims[3] = {(cuuint64_t)g.K, (cuuint64_t)p.Tl, (cuuint64_t)nb};
        const cuuint64_t strides[2] = {(cuuint64_t)g.lda * 2, (cuuint64_t)g.lda * 2 * p.Tl};
        const cuuint32_t box[3] = {TC_BK, TC_BM, 1};
        if (enc(&p.tm_a, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<bf16*>(g.A), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return cudaErrorInvalidValue;
    }
    {
        const cuuint64_t dims[2] = {(cuuint64_t)g.K, (cuuint64_t)g.taps * g.Nw};
        const cuuint64_t strides[1] = {(cuuint64_t)g.ldw * 2};
        const cuuint32_t box[2] = {TC_BK, (cuuint32_t)TC_BN};
        if (enc(&p.tm_w, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<bf16*>(g.W), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            return cudaErrorInvalidValue;
    }
    p.tma_out = 0;
    if (g.scatter == SC_NONE && (g.out_f32 != nullptr) != (g.out_bf16 != nullptr)) {
        const bool f32 = g.out_f32 != nullptr;
        const size_t es = f32 ? 4 : 2;
        void* base = f32 ? (void*)g.out_f32 : (void*)g.out_bf16;
        if (((size_t)g.ldo * es) % 16 == 0 && (reinterpret_cast<uintptr_t>(base) & 15) == 0 && (g.ldo & 7) == 0 && (g.ldr & 7) == 0) {
            const cuuint64_t dims[3] = {(cuuint64_t)g.N, (cuuint64_t)p.Tl, (cuuint64_t)nb};
            const cuuint64_t strides[2] = {(cuuint64_t)g.ldo * es, (cuuint64_t)g.ldo * es * p.Tl};
            const cuuint32_t box[3] = {f32 ? 32u : 64u, 32, 1};
            if (enc(&p.tm_out, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS)
                p.tma_out = f32 ? 1 : 2;
        }
    }
    p.n_tiles_n = (g.N + TC_BN - 1) / TC_BN;
    p.n_tiles = p.n_tiles_n * nb * p.tiles_per_utt;
    int grid = p.n_tiles < num_sms ? p.n_tiles : num_sms;                // persistent: one CTA per SM, static round-robin tiles
    // capped beside a running kernel: a CTA that finds no free SM would hold its round-robin tiles until that kernel ends
    if (g.max_ctas > 0 && grid > g.max_ctas) grid = g.max_ctas;
    if (TC_BN == 256) gemm_tc_kernel<256><<<grid, TC_THREADS, tc_smem_bytes(256), stream>>>(p);
    else gemm_tc_kernel<128><<<grid, TC_THREADS, tc_smem_bytes(128), stream>>>(p);
    ++launch_counter();
    return cudaGetLastError();
}

}  // namespace tts
