// Encoder-decoder attention alignments of the teacher-forced forward, and FastSpeech-style phoneme durations from them
// (Ren et al., 2019, section 3.3; the procedure of ESPnet's DurationCalculator).
//
//   cross_align_kernel   P[b][h][t][s] = softmax_s(q_t . k_s / 8) of one decoder layer, from the bf16 operands the flash
//                        kernel just used (Q = x2 [B*T][512], K = that layer's row-major cross-K [B][H][Spad][64]), plus per
//                        row rowmax = max_s P and argmax = the first s with the largest score.  The kernel computes its own
//                        softmax statistics (the flash kernel's log-sum-exp takes part of its exponentials from a polynomial,
//                        so a P rebuilt from it would not sum to 1 within fp32 rounding): pass 1 over the key tiles keeps the
//                        running max, argmax and sum; pass 2 (only when P is wanted) recomputes the scores and writes
//                        2^((s - m) * scale) / sum.  rowmax = 1 / sum comes from pass 1 at no cost: the maximal element is
//                        2^0 / sum.
//   focus_kernel         F[l][b][h] = mean over t < mel_len[b] of rowmax (the focus rate), summed in a fixed order.
//   durations_kernel     per utterance the (layer, head) with the largest F (ties: lowest layer * 8 + h) or a fixed one;
//                        durations[b][s] = number of frames t < mel_len[b] whose argmax is s.
//
// Layout of cross_align_kernel: one CTA = 64 query rows of one (b, h), four warps of 16 rows each.  A key tile of 64 rows is
// staged in shared memory (rows padded to 72 bf16, so the B-fragment loads of the eight row groups hit distinct banks); the
// scores of a warp's 16 x 64 block come from mma.sync m16n8k16 (bf16, fp32 accumulation).  The P write stream (164 MB per
// layer at B 64, T 800, S 100) is the cost, not the math: each warp stages its 16 x 64 block of P in shared memory and writes
// it back row by row, 32 consecutive floats per store instruction, with streaming (evict-first) stores.
// Every reduction runs in a fixed order and there are no floating-point atomics: the output is bit-identical run to run.
#pragma once
#include "common.cuh"

namespace tts {

constexpr int AL_BM = 64, AL_BN = 64, AL_THREADS = 128;
constexpr int AL_KPAD = 72;                 // bf16 per staged key row
constexpr int AL_PPAD = 72;                 // fp32 per staged P row
constexpr int AL_MIN_CTAS = 4;              // resident CTAs per SM (37 KB of shared memory each): the kernel is latency-bound

struct AlignParams {
    const bf16* Q; long q_bs, q_rs;         // Q[b][t][64 h + d]: element strides of batch and row
    const bf16* K; long k_bs, k_hs;         // K[b][h][s][64] (row stride 64)
    const int* qlens; const int* klens;     // rows t >= qlens[b] and keys s >= klens[b] are masked (null: all valid)
    int B, H, Lq, Lk;
    float scale_log2;                       // (1/8) * log2(e)
    float* P;                               // optional [B][H][Lq][Lk]
    float* rowmax;                          // optional [B][H][Lq]
    int16_t* argmax;                        // optional [B][H][Lq]
};

// combine two (max, argmax, sum) triples; ties of the max go to the lower index
TTS_D void al_combine(float& m, int& i, float& l, float m2, int i2, float l2, float c) {
    const float mn = fmaxf(m, m2);
    if (mn == -INFINITY) return;
    const float a = m == -INFINITY ? 0.f : l * fast_exp2((m - mn) * c);
    const float b = m2 == -INFINITY ? 0.f : l2 * fast_exp2((m2 - mn) * c);
    if (m2 > m || (m2 == m && i2 < i)) i = i2;
    m = mn; l = a + b;
}

__global__ void __launch_bounds__(AL_THREADS, AL_MIN_CTAS) cross_align_kernel(AlignParams p) {
    __shared__ __align__(16) bf16 ks[2][AL_BN * AL_KPAD];
    __shared__ __align__(16) float ps[AL_THREADS / 32][16 * AL_PPAD];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t4 = lane & 3;
    const int h = blockIdx.y, b = blockIdx.z;
    const int r0 = blockIdx.x * AL_BM + warp * 16;                 // first query row of this warp
    const int qlen = p.qlens ? min(max(p.qlens[b], 0), p.Lq) : p.Lq;
    const int klen = p.klens ? min(max(p.klens[b], 0), p.Lk) : p.Lk;
    const float c = p.scale_log2;
    const bf16* kbase = p.K + (long)b * p.k_bs + (long)h * p.k_hs;

    // Key tiles are consumed in the sequence 0 .. n1-1 (pass 1), then 0 .. n1-1 again (pass 2, if P is wanted); tile i + 1 of
    // the sequence is fetched with cp.async into the other buffer while tile i is used.
    const int n1 = (klen + AL_BN - 1) / AL_BN;
    const int nseq = p.P ? 2 * n1 : n1;
    auto fetch = [&](int i) {
        const int k0 = (i % n1) * AL_BN;
        bf16* dst = ks[i & 1];
        for (int e = threadIdx.x; e < AL_BN * 8; e += AL_THREADS) {
            const int r = e >> 3, ch = e & 7;
            const bool v = k0 + r < p.Lk;
            cp_async_16(&dst[r * AL_KPAD + ch * 8], kbase + (v ? (long)(k0 + r) * 64 + ch * 8 : 0), v);
        }
        cp_async_commit();
    };
    if (nseq > 0) fetch(0);

    // Q fragments of the warp's 16 rows x 64 dims (rows past Lq read as zero)
    uint32_t qa[4][4];
    {
        const bf16* q = p.Q + (long)b * p.q_bs + (long)h * 64;
        const int ra = r0 + g, rb = r0 + g + 8;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            const int d = kk * 16 + 2 * t4;
            qa[kk][0] = ra < p.Lq ? *reinterpret_cast<const uint32_t*>(q + (long)ra * p.q_rs + d) : 0u;
            qa[kk][1] = rb < p.Lq ? *reinterpret_cast<const uint32_t*>(q + (long)rb * p.q_rs + d) : 0u;
            qa[kk][2] = ra < p.Lq ? *reinterpret_cast<const uint32_t*>(q + (long)ra * p.q_rs + d + 8) : 0u;
            qa[kk][3] = rb < p.Lq ? *reinterpret_cast<const uint32_t*>(q + (long)rb * p.q_rs + d + 8) : 0u;
        }
    }

    // scores of the warp's 16 x 64 block against tile i of the sequence (block-uniform call: it synchronises)
    auto scores = [&](int i, float (&acc)[8][4]) {
        if (i + 1 < nseq) { fetch(i + 1); cp_async_wait<1>(); }
        else cp_async_wait<0>();
        __syncthreads();                                           // tile i visible to every warp
        const bf16* kt = ks[i & 1];
#pragma unroll
        for (int n = 0; n < 8; ++n) {
            acc[n][0] = acc[n][1] = acc[n][2] = acc[n][3] = 0.f;
            const bf16* kr = &kt[(n * 8 + g) * AL_KPAD + 2 * t4];
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
                mma_bf16_16816(acc[n], qa[kk], *reinterpret_cast<const uint32_t*>(kr + kk * 16),
                               *reinterpret_cast<const uint32_t*>(kr + kk * 16 + 8));
        }
        __syncthreads();                                           // every warp is done with buffer i & 1 before fetch(i + 2)
    };

    // ---- pass 1: running max / first argmax / sum of 2^((s - m) c) for rows g (j = 0) and g + 8 (j = 1)
    float m[2] = {-INFINITY, -INFINITY}, l[2] = {0.f, 0.f};
    int am[2] = {-1, -1};
    for (int kt = 0; kt < n1; ++kt) {
        const int k0 = kt * AL_BN;
        float acc[8][4];
        scores(kt, acc);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            float tm = -INFINITY; int ti = -1;
#pragma unroll
            for (int n = 0; n < 8; ++n)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int s = k0 + n * 8 + 2 * t4 + e;
                    const float v = acc[n][2 * j + e];
                    if (s < klen && v > tm) { tm = v; ti = s; }    // columns ascend: strict > keeps the first maximum
                }
            if (tm == -INFINITY) continue;
            float ts = 0.f;
#pragma unroll
            for (int n = 0; n < 8; ++n)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int s = k0 + n * 8 + 2 * t4 + e;
                    if (s < klen) ts += fast_exp2((acc[n][2 * j + e] - tm) * c);
                }
            al_combine(m[j], am[j], l[j], tm, ti, ts, c);           // earlier tiles hold lower indices
        }
    }
    // the four lanes of a row group hold interleaved columns: combine them in a fixed butterfly order
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int o = 1; o < 4; o <<= 1) {
            const float m2 = __shfl_xor_sync(0xffffffffu, m[j], o), l2 = __shfl_xor_sync(0xffffffffu, l[j], o);
            const int i2 = __shfl_xor_sync(0xffffffffu, am[j], o);
            al_combine(m[j], am[j], l[j], m2, i2, l2, c);
        }
    float inv[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const int r = r0 + g + 8 * j;
        const bool ok = r < qlen && m[j] != -INFINITY;
        inv[j] = ok ? 1.f / l[j] : 0.f;
        if (!ok) am[j] = -1;
        if (t4 == 0 && r < p.Lq) {
            const long o = ((long)b * p.H + h) * p.Lq + r;
            if (p.rowmax) p.rowmax[o] = inv[j];
            if (p.argmax) p.argmax[o] = (int16_t)am[j];
        }
    }
    if (!p.P) return;

    // ---- pass 2: P = 2^((s - m) c) / sum, zero at masked keys and rows; staged per warp, written row by row
    float* stage = ps[warp];
    const int ntile2 = (p.Lk + AL_BN - 1) / AL_BN;
    for (int kt = 0; kt < ntile2; ++kt) {
        const int k0 = kt * AL_BN;
        float acc[8][4];
        if (kt < n1) scores(n1 + kt, acc);
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int n = 0; n < 8; ++n) {
                float v[2];
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int s = k0 + n * 8 + 2 * t4 + e;
                    v[e] = (kt < n1 && s < klen && inv[j] != 0.f) ? fast_exp2((acc[n][2 * j + e] - m[j]) * c) * inv[j] : 0.f;
                }
                *reinterpret_cast<float2*>(&stage[(g + 8 * j) * AL_PPAD + n * 8 + 2 * t4]) = make_float2(v[0], v[1]);
            }
        __syncwarp();
        const int ncol = min(AL_BN, p.Lk - k0);
        for (int rr = 0; rr < 16; ++rr) {
            const int r = r0 + rr;
            if (r >= p.Lq) break;
            float* dst = p.P + (((long)b * p.H + h) * p.Lq + r) * p.Lk + k0;
            if (lane < ncol) __stcs(dst + lane, stage[rr * AL_PPAD + lane]);
            if (lane + 32 < ncol) __stcs(dst + lane + 32, stage[rr * AL_PPAD + lane + 32]);
        }
        __syncwarp();
    }
}

// focus[l][b][h] = (1 / qlen[b]) sum_{t < qlen[b]} rowmax[l][b][h][t] for the layers in layer_mask, -1 for the others.
// One warp per (l, b, h); lane-strided partial sums, then a fixed butterfly.
__global__ void focus_kernel(const float* __restrict__ rowmax, const int* __restrict__ qlens, int B, int H, int T, uint32_t layer_mask,
                             float* __restrict__ focus) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= 6 * B * H) return;
    const int l = w / (B * H), b = (w / H) % B;
    float f = -1.f;
    if ((layer_mask >> l) & 1u) {
        const int n = min(max(qlens[b], 0), T);
        const float* r = rowmax + (long)w * T;
        float s = 0.f;
        for (int t = lane; t < n; t += 32) s += r[t];
        s = warp_sum(s);
        f = n > 0 ? s / (float)n : 0.f;
    }
    if (lane == 0) focus[w] = f;
}

// One block per utterance: pick the (layer, head), then count the frames whose argmax is each phoneme (integer shared-memory
// atomics: the counts do not depend on their order).  durations [B][S] int32 (0 past klens[b]), head [B] = layer * H + h.
__global__ void durations_kernel(const float* __restrict__ focus, const int16_t* __restrict__ argmax, const int* __restrict__ qlens,
                                 const int* __restrict__ klens, int B, int H, int S, int T, uint32_t layer_mask, int fixed_head,
                                 int32_t* __restrict__ durations, int32_t* __restrict__ head) {
    extern __shared__ int cnt[];                                   // [S]
    __shared__ int sel;
    const int b = blockIdx.x;
    if (threadIdx.x == 0) {
        int best = fixed_head;
        if (best < 0) {
            float bf = -INFINITY;
            for (int l = 0; l < 6; ++l) {
                if (!((layer_mask >> l) & 1u)) continue;
                for (int hh = 0; hh < H; ++hh) {
                    const float f = focus[((long)l * B + b) * H + hh];
                    if (best < 0 || f > bf) { bf = f; best = l * H + hh; }
                }
            }
        }
        sel = best;
        if (head) head[b] = best;
    }
    for (int s = threadIdx.x; s < S; s += blockDim.x) cnt[s] = 0;
    __syncthreads();
    const int l = sel / H, hh = sel % H;
    const int n = min(max(qlens[b], 0), T), kl = min(max(klens[b], 0), S);
    const int16_t* a = argmax + (((long)l * B + b) * H + hh) * T;
    for (int t = threadIdx.x; t < n; t += blockDim.x) {
        const int s = a[t];
        if (s >= 0 && s < kl) atomicAdd(&cnt[s], 1);
    }
    __syncthreads();
    if (durations)
        for (int s = threadIdx.x; s < S; s += blockDim.x) durations[(long)b * S + s] = cnt[s];
}

inline cudaError_t launch_cross_align(const AlignParams& p, cudaStream_t st) {
    dim3 grid((p.Lq + AL_BM - 1) / AL_BM, p.H, p.B);
    cross_align_kernel<<<grid, AL_THREADS, 0, st>>>(p);
    ++launch_counter();
    return cudaGetLastError();
}

}  // namespace tts
