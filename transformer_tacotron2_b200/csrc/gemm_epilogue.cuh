// Parameters and fused epilogue of the sequence-parallel GEMM / conv kernel (gemm_tc.cuh):
//     C[M,N] = epi( sum_tap A[m + tap - pad, :] . W[tap][n, :] )
// epi order: + bias, + alpha * pe, word dropout, + residual, activation, bit dropout, length mask
// used by the encoder, the cross-K/V projection, the teacher-forced decoder and the postnet
// (SURVEY.md 8(a) rows a3, a4, a10).  gemm_store is the scalar (pair-wise) form of the epilogue; the kernel uses
// a 16-byte vectorised form of the same arithmetic where the output is a plain matrix with 16-byte aligned rows.  The two
// forms give bit-identical results (tests/test_gpu_seq_kernels.py); the scalar form handles any layout, so it also takes the
// scatters, the columns past the last full 32-column chunk and every misaligned operand.
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace tts {

enum GemmAct { ACT_NONE = 0, ACT_RELU = 1, ACT_TANH = 2 };
enum GemmScatter { SC_NONE = 0, SC_CROSS_KV = 1, SC_HEAD = 2, SC_CROSS_KV_VT = 3 };

struct GemmParams {
    // operands
    const bf16* A; int lda;          // [M][lda] bf16, K valid columns (K % 32 == 0)
    const bf16* W; int ldw;          // [taps][Nw][ldw] bf16, Nw = N rounded up to 128 (zero rows)
    int M, N, K, taps, Nw;
    int T;                           // rows per utterance (row m -> b = m / T, t = m % T); T = M if unused
    // epilogue
    const float* bias;               // [N] or null
    int act;
    const bf16* resid_bf16; const float* resid_f32; int ldr;
    const float* pe; float alpha;    // + alpha * pe[t][n]   (pe row stride 512)
    const float* alpha_ptr;          // if set, alpha is read from device memory (trainable scalar)
    const int* lens;                 // zero rows with t >= lens[b]
    int drop_site; uint64_t seed; int utt_offset;   // p = 0.5 bit dropout after the activation (site < 0: off)
    const uint64_t* seed_ptr;        // if set, the seed is read from device memory (training steps replayed from a CUDA graph)
    int dropw_site; uint32_t dropw_thresh; float dropw_scale;   // word dropout (training, P12) of (acc + bias + alpha * pe), BEFORE the residual
    float* out_f32; bf16* out_bf16; int ldo;
    int scatter;                     // GemmScatter
    // SC_CROSS_KV: out_bf16 = cache [layers][2][B][H][Lpad][64], N = layers * 1024, T = S; SC_CROSS_KV_VT: the decode kernel's blocks
    // SC_HEAD    : out_f32 = mel_before [M][80], out2_f32 = stop_logits [M]
    float* out2_f32; int B;
    int Lpad;                        // SC_CROSS_KV*: row capacity of the cache per (layer, b, h): multiple of 16 (row-major) / 64 (blocks)
    int max_ctas;                    // launch_gemm_tc: at most this many persistent CTAs (0 = one per SM); leaves SMs to a concurrent kernel
};

TTS_D void gemm_store(const GemmParams& p, int m, int n, float v0, float v1) {
    // (m, n) and (m, n+1); n is even
    if (m >= p.M || n >= p.N) return;
    const bool has1 = (n + 1) < p.N;
    const int b = m / p.T, t = m - b * p.T;
    const uint64_t seed = p.seed_ptr ? *p.seed_ptr : p.seed;
    // + 0 without a bias, as the vector form adds (a -0 accumulator leaves both forms as +0)
    v0 += p.bias ? p.bias[n] : 0.f; v1 += p.bias && has1 ? p.bias[n + 1] : 0.f;
    if (p.pe) {                                      // explicit FMA / multiply below: both forms round alike whatever nvcc contracts
        const float alpha = p.alpha_ptr ? *p.alpha_ptr : p.alpha;
        v0 = __fmaf_rn(alpha, p.pe[(size_t)t * kDModel + n], v0);
        if (has1) v1 = __fmaf_rn(alpha, p.pe[(size_t)t * kDModel + n + 1], v1);
    }
    if (p.dropw_site >= 0) {                         // n even: words n % 4 and n % 4 + 1 of chunk n / 4
        const uint4 w = philox4x32_10(make_uint4((uint32_t)p.dropw_site, (uint32_t)t, (uint32_t)(p.utt_offset + b), (uint32_t)(n >> 2)),
                                      (uint32_t)seed, (uint32_t)(seed >> 32));
        const uint32_t w0 = (n & 2) ? w.z : w.x, w1 = (n & 2) ? w.w : w.y;
        v0 = w0 >= p.dropw_thresh ? __fmul_rn(v0, p.dropw_scale) : 0.f;
        v1 = w1 >= p.dropw_thresh ? __fmul_rn(v1, p.dropw_scale) : 0.f;
    }
    if (p.resid_bf16) {
        v0 += __bfloat162float(p.resid_bf16[(size_t)m * p.ldr + n]);
        if (has1) v1 += __bfloat162float(p.resid_bf16[(size_t)m * p.ldr + n + 1]);
    }
    if (p.resid_f32) {
        v0 += p.resid_f32[(size_t)m * p.ldr + n];
        if (has1) v1 += p.resid_f32[(size_t)m * p.ldr + n + 1];
    }
    if (p.act == ACT_RELU) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); }
    else if (p.act == ACT_TANH) { v0 = tanhf(v0); v1 = tanhf(v1); }
    if (p.drop_site >= 0) {
        v0 = keep_bit(seed, p.drop_site, t, p.utt_offset + b, n) ? 2.f * v0 : 0.f;
        if (has1) v1 = keep_bit(seed, p.drop_site, t, p.utt_offset + b, n + 1) ? 2.f * v1 : 0.f;
    }
    if (p.lens && t >= p.lens[b]) { v0 = 0.f; v1 = 0.f; }
    if (p.scatter == SC_CROSS_KV) {
        // teacher-forced flash attention: n = layer * 1024 + kv * 512 + h * 64 + d  ->  cache [layer][kv][B][H][Lpad][64], row-major
        const int lkv = n >> 9, h = (n >> 6) & 7, d = n & 63;
        const size_t base = (((size_t)lkv * p.B + b) * kHeads + h) * (size_t)p.Lpad * kDHead;
        *reinterpret_cast<uint32_t*>(p.out_bf16 + base + (size_t)t * kDHead + d) = pack_bf16x2(v0, v1);
        return;
    }
    if (p.scatter == SC_CROSS_KV_VT) {
        // decode kernel (decode_cluster.cuh): per (layer, b, h) 64-row blocks of 8192 elements,
        // four 16-row sub-chunks [K rows | V in MMA A-fragment order] (kv_k_elem / kv_v_elem, common.cuh); Lpad = 64 * blocks
        const int layer = n >> 10, kv = (n >> 9) & 1, h = (n >> 6) & 7, d = n & 63, r = t & 63;
        bf16* blk = p.out_bf16 + ((((size_t)layer * p.B + b) * kHeads + h) * (size_t)(p.Lpad >> 6) + (t >> 6)) * 8192;
        if (kv) {
            blk[kv_v_elem(r, d)] = __float2bfloat16(v0);
            blk[kv_v_elem(r, d + 1)] = __float2bfloat16(v1);
        } else {
            *reinterpret_cast<uint32_t*>(blk + kv_k_elem(r, d)) = pack_bf16x2(v0, v1);
        }
        return;
    }
    if (p.scatter == SC_HEAD) {
        if (n < 80) { p.out_f32[(size_t)m * 80 + n] = v0; if (n + 1 < 80) p.out_f32[(size_t)m * 80 + n + 1] = v1; }
        if (n == 80) p.out2_f32[m] = v0;
        return;
    }
    if (p.out_f32) {
        p.out_f32[(size_t)m * p.ldo + n] = v0;
        if (has1) p.out_f32[(size_t)m * p.ldo + n + 1] = v1;
    }
    if (p.out_bf16) {
        bf16* o = p.out_bf16 + (size_t)m * p.ldo + n;
        if (has1 && (reinterpret_cast<uintptr_t>(o) & 3) == 0) *reinterpret_cast<uint32_t*>(o) = pack_bf16x2(v0, v1);
        else {
            o[0] = __float2bfloat16(v0);
            if (has1) o[1] = __float2bfloat16(v1);
        }
    }
}

}  // namespace tts
