// Speaker conditioning of the encoder memory (ESPnet Transformer-TTS, spk_embed_integration_type "add"):
//     cond[b] = E[sids[b]] + W . normalize(spembs[b]) + bias,      memory[b, s] = encoder_out[b, s] + cond[b]  (every s < S)
// E [n_speakers][512] is the speaker-ID table, W [512][D] / bias [512] the x-vector projection; either part may be absent.
// The addition itself is fused into the last encoder LayerNorm (layernorm512_kernel<true>), so memory costs no extra pass:
// the decode kernel, the alignment kernels and the postnet see conditioning through the cross-K/V projection of memory.
// Every reduction here runs in a fixed order without atomics, so results (and gradients) are bit-identical from run to run.
#pragma once
#include "common.cuh"
#include "misc_kernels.cuh"

namespace tts {

constexpr int kSpkMaxDim = 1024;            // largest x-vector dimension D (the normalised vector is staged in shared memory)
constexpr int kSpkThreads = 512;
constexpr int kSpkMaxSpeakers = 65536;      // speaker-ID table rows (fp32: 128 MB at most)

// One CTA per utterance.  nhat[b] = spembs[b] / max(||spembs[b]||, 1e-12) (F.normalize), cond[b][n] = E[sids[b]][n] (zero row for
// an id outside [0, n_speakers)) + bias[n] + sum_k W[n][k] nhat[b][k].  E null: no speaker-ID term; W null (D = 0): no x-vector term.
__global__ void __launch_bounds__(kSpkThreads) speaker_cond_kernel(const int* __restrict__ sids, const float* __restrict__ spembs,
                                                                  int n_speakers, int D, const float* __restrict__ E,
                                                                  const float* __restrict__ W, const float* __restrict__ bias,
                                                                  float* __restrict__ cond, float* __restrict__ nhat) {
    __shared__ float xs[kSpkMaxDim];
    __shared__ float red[kSpkThreads / 32];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (W) {
        float ss = 0.f;
        for (int k = tid; k < D; k += kSpkThreads) { const float v = spembs[(size_t)b * D + k]; xs[k] = v; ss += v * v; }
        ss = warp_sum(ss);
        if (lane == 0) red[warp] = ss;
        __syncthreads();
        float tot = 0.f;
#pragma unroll
        for (int i = 0; i < kSpkThreads / 32; ++i) tot += red[i];
        const float den = fmaxf(sqrtf(tot), 1e-12f);
        __syncthreads();
        for (int k = tid; k < D; k += kSpkThreads) { const float v = xs[k] / den; xs[k] = v; nhat[(size_t)b * D + k] = v; }
        __syncthreads();
    }
    float* out = cond + (size_t)b * kDModel;
    if (E) {
        const int sid = sids[b];
        out[tid] = (sid >= 0 && sid < n_speakers) ? E[(size_t)sid * kDModel + tid] : 0.f;
    } else {
        out[tid] = 0.f;
    }
    if (!W) return;
    __syncthreads();
    // the projection: warp w owns output rows w, w + 16, ...; lanes stride the row (coalesced), one warp_sum per row
    for (int n = warp; n < kDModel; n += kSpkThreads / 32) {
        const float* wr = W + (size_t)n * D;
        float acc = 0.f;
        for (int k = lane; k < D; k += 32) acc += wr[k] * xs[k];
        acc = warp_sum(acc);
        if (lane == 0) out[n] += bias[n] + acc;
    }
}

// dcond[b][n] = sum_{s < plens[b]} dmem[b * S + s][n]: one thread per (b, n), rows summed in ascending s.
__global__ void speaker_dcond_kernel(const float* __restrict__ dmem, const int* __restrict__ plens, int B, int S, float* __restrict__ dcond) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * kDModel) return;
    const int b = i / kDModel, n = i - b * kDModel;
    const int L = min(max(plens[b], 0), S);
    const float* p = dmem + (size_t)b * S * kDModel + n;
    float acc = 0.f;
    for (int s = 0; s < L; ++s) acc += p[(size_t)s * kDModel];
    dcond[i] = acc;
}

// Parameter gradients from dcond, each output element owned by one thread and summed over b in ascending order:
//   dE[j][n] += sum_{b: sids[b] = j} dcond[b][n]   (rows of speakers not in the batch are not touched)
//   dW[n][k] += sum_b dcond[b][n] nhat[b][k],   dbias[n] += sum_b dcond[b][n]
// Threads [0, n_speakers * 512) cover dE, the next 512 * D dW, the last 512 dbias.
__global__ void speaker_param_grad_kernel(const float* __restrict__ dcond, const int* __restrict__ sids, const float* __restrict__ nhat, int B,
                                          int n_speakers, int D, float* __restrict__ dE, float* __restrict__ dW, float* __restrict__ dbias) {
    long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    const long nE = dE ? (long)n_speakers * kDModel : 0, nW = dW ? (long)kDModel * D : 0;
    if (i < nE) {
        const int j = (int)(i / kDModel), n = (int)(i - (long)j * kDModel);
        float acc = 0.f;
        bool any = false;
        for (int b = 0; b < B; ++b)
            if (sids[b] == j) { acc += dcond[(size_t)b * kDModel + n]; any = true; }
        if (any) dE[i] += acc;
        return;
    }
    i -= nE;
    if (i < nW) {
        const int n = (int)(i / D), k = (int)(i - (long)n * D);
        float acc = 0.f;
        for (int b = 0; b < B; ++b) acc += dcond[(size_t)b * kDModel + n] * nhat[(size_t)b * D + k];
        dW[i] += acc;
        return;
    }
    i -= nW;
    if (dW && i < kDModel) {
        float acc = 0.f;
        for (int b = 0; b < B; ++b) acc += dcond[(size_t)b * kDModel + i];
        dbias[i] += acc;
    }
}

// ---- launches (shared by the library's forward / training step and the per-kernel test entry points)
inline cudaError_t launch_speaker_cond(const int* sids, const float* spembs, int B, int n_speakers, int D, const float* E, const float* W,
                                       const float* bias, float* cond, float* nhat, cudaStream_t st) {
    speaker_cond_kernel<<<B, kSpkThreads, 0, st>>>(sids, spembs, n_speakers, D, E, W, bias, cond, nhat);
    ++launch_counter();
    return cudaGetLastError();
}
inline cudaError_t launch_layernorm_cond(const float* x, const float* g, const float* b, bf16* o16, float* o32, int M, float eps, const float* cond,
                                         int S, cudaStream_t st) {
    layernorm512_kernel<true><<<(M + 7) / 8, 256, 0, st>>>(x, g, b, o16, o32, M, eps, cond, S);
    ++launch_counter();
    return cudaGetLastError();
}
// two launches: the segmented column sum, then the parameter gradients
inline cudaError_t launch_speaker_cond_bwd(const float* dmem, const int* plens, const int* sids, const float* nhat, int B, int S, int n_speakers,
                                           int D, float* dcond, float* dE, float* dW, float* dbias, cudaStream_t st) {
    speaker_dcond_kernel<<<(B * kDModel + 255) / 256, 256, 0, st>>>(dmem, plens, B, S, dcond);
    const long n = (dE ? (long)n_speakers * kDModel : 0) + (dW ? (long)kDModel * D + kDModel : 0);
    speaker_param_grad_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dcond, sids, nhat, B, n_speakers, D, dE, dW, dbias);
    launch_counter() += 2;
    return cudaGetLastError();
}

}  // namespace tts
