// Small memory-bound kernels around the GEMM / attention kernels of the sequence-parallel path.
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace tts {

// x[b][s][:] = (s < len[b]) ? embed[phoneme] : 0      (bf16 [B*S][512]); P6 + P9
__global__ void embed_kernel(const int64_t* __restrict__ ph, const int* __restrict__ lens, const bf16* __restrict__ table,
                             bf16* __restrict__ out, int B, int S, int n_vocab) {
    const int row = blockIdx.x * (blockDim.x >> 6) + (threadIdx.x >> 6);   // 64 threads (x 16 B) per row
    if (row >= B * S) return;
    const int b = row / S, s = row - b * S, c = threadIdx.x & 63;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (s < lens[b]) {
        long id = ph[row];
        if (id >= 0 && id < n_vocab) v = *reinterpret_cast<const uint4*>(table + id * kDModel + c * 8);
    }
    *reinterpret_cast<uint4*>(out + (size_t)row * kDModel + c * 8) = v;
}

// LayerNorm over rows of 512 (fp32 in, bf16 and/or fp32 out); one warp per row, two-pass statistics.
// kCond: the row of utterance m / S of cond fp32 [B][512] is added to the affine output in fp32, before the rounding
// (speaker conditioning of the encoder memory, speaker.cuh); the <false> instantiation never reads cond.
template <bool kCond>
__global__ void layernorm512_kernel(const float* __restrict__ x, const float* __restrict__ g, const float* __restrict__ bta,
                                    bf16* __restrict__ out_bf16, float* __restrict__ out_f32, int M, float eps,
                                    const float* __restrict__ cond, int S) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= M) return;
    float v[16];
    const float* src = x + (size_t)row * kDModel;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float4 t = *reinterpret_cast<const float4*>(src + i * 128 + lane * 4);
        v[i * 4] = t.x; v[i * 4 + 1] = t.y; v[i * 4 + 2] = t.z; v[i * 4 + 3] = t.w;
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += v[i];
    const float mean = warp_sum(s) * (1.f / 512.f);
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) { const float d = v[i] - mean; ss += d * d; }
    const float rstd = rsqrtf(warp_sum(ss) * (1.f / 512.f) + eps);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int c = i * 128 + lane * 4;
        const float4 g4 = *reinterpret_cast<const float4*>(g + c), b4 = *reinterpret_cast<const float4*>(bta + c);
        float o0 = (v[i * 4] - mean) * rstd * g4.x + b4.x, o1 = (v[i * 4 + 1] - mean) * rstd * g4.y + b4.y;
        float o2 = (v[i * 4 + 2] - mean) * rstd * g4.z + b4.z, o3 = (v[i * 4 + 3] - mean) * rstd * g4.w + b4.w;
        if constexpr (kCond) {
            const float4 c4 = *reinterpret_cast<const float4*>(cond + (size_t)(row / S) * kDModel + c);
            o0 += c4.x; o1 += c4.y; o2 += c4.z; o3 += c4.w;
        }
        if (out_bf16) *reinterpret_cast<uint2*>(out_bf16 + (size_t)row * kDModel + c) = make_uint2(pack_bf16x2(o0, o1), pack_bf16x2(o2, o3));
        if (out_f32) *reinterpret_cast<float4*>(out_f32 + (size_t)row * kDModel + c) = make_float4(o0, o1, o2, o3);
    }
}

// mel rows fp32 [B][T_src][80] -> bf16 [B][T][96] (zero channel padding), optionally shifted right by
// one frame (teacher forcing, P8: row t reads frame t-1, row 0 is the zero go-frame) and masked
// (rows t >= lens[b] -> 0).  Also optionally writes the masked fp32 rows compactly ([B][T][80]).
__global__ void mel_to_bf16_kernel(const float* __restrict__ mel, int T_src, const int* __restrict__ lens, int shift,
                                   bf16* __restrict__ out16, float* __restrict__ out32, int B, int T) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;            // one thread per (row, 4 channels); 24 groups/row
    if (idx >= B * T * 24) return;
    const int row = idx / 24, cg = idx - row * 24, b = row / T, t = row - b * T;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    const int ts = t - shift;
    const bool valid = (lens == nullptr) || (shift ? (ts < lens[b]) : (t < lens[b]));
    if (cg < 20 && ts >= 0 && valid) v = *reinterpret_cast<const float4*>(mel + ((size_t)b * T_src + ts) * 80 + cg * 4);
    if (out16) *reinterpret_cast<uint2*>(out16 + (size_t)row * 96 + cg * 4) = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
    if (out32 && cg < 20) *reinterpret_cast<float4*>(out32 + (size_t)row * 80 + cg * 4) = v;
}

// stop logits [B][T_src] -> compact masked [B][T]; lens copied out.
__global__ void finalize_stop_kernel(const float* __restrict__ stop, int T_src, const int* __restrict__ lens,
                                     float* __restrict__ out, int* __restrict__ lens_out, int B, int T) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < B * T) {
        const int b = idx / T, t = idx - b * T;
        out[idx] = (t < lens[b]) ? stop[(size_t)b * T_src + t] : 0.f;
    }
    if (idx < B && lens_out) lens_out[idx] = lens[idx];
}

// Postnet input of frames [a, a + W) of a running decode session (tts_decode_emit), the window counterpart of mel_to_bf16_kernel +
// finalize_stop_kernel: bf16 [B][W][96] (zero channel padding) and the fp32 residual [B][W][80], both zero at t >= len;
// wlens[b] = len - a clamped to [0, W] (the postnet's per-layer mask); stop [B][n] of frames [t_begin, t_begin + n), zero at
// t >= len; lens_out[b] (optional) = lens[b] if the utterance had stopped by t_status, else -1.  Here len = min(lens[b], t_status).
// lens[] may be written meanwhile by a decode launch from t_status on (an utterance stopping in it gets lens = t + 1 > t_status),
// so either value gives the same len and the same lens_out; the frames read (< t_status) are written by no such launch.
__global__ void stream_window_kernel(const float* __restrict__ mel, const float* __restrict__ stop, int T_src, const int* lens,
                                     int t_status, int a, int W, int t_begin, int n, bf16* __restrict__ out16,
                                     float* __restrict__ out32, int* __restrict__ wlens, float* __restrict__ stop_out,
                                     int* __restrict__ lens_out, int B) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;            // one thread per (row, 4 channels); 24 groups/row
    if (idx < B * W * 24) {
        const int row = idx / 24, cg = idx - row * 24, b = row / W, t = a + (row - b * W);
        const int len = min(*(volatile const int*)(lens + b), t_status);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (cg < 20 && t < len) v = *reinterpret_cast<const float4*>(mel + ((size_t)b * T_src + t) * 80 + cg * 4);
        *reinterpret_cast<uint2*>(out16 + (size_t)row * 96 + cg * 4) = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
        if (cg < 20) *reinterpret_cast<float4*>(out32 + (size_t)row * 80 + cg * 4) = v;
    }
    if (idx < B * n) {
        const int b = idx / n, t = t_begin + (idx - b * n);
        const int len = min(*(volatile const int*)(lens + b), t_status);
        stop_out[idx] = t < len ? stop[(size_t)b * T_src + t] : 0.f;
    }
    if (idx < B) {
        const int l = *(volatile const int*)(lens + idx);
        wlens[idx] = max(0, min(min(l, t_status) - a, W));
        if (lens_out) lens_out[idx] = l <= t_status ? l : -1;
    }
}

__global__ void bf16_to_f32_kernel(const bf16* __restrict__ in, float* __restrict__ out, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = __bfloat162float(in[i]);
}

__global__ void mask_rows_kernel(float* __restrict__ x, const int* __restrict__ lens, int B, int T, int C) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)B * T * C) return;
    const int row = (int)(i / C), b = row / T, t = row - b * T;
    if (t >= lens[b]) x[i] = 0.f;
}

__global__ void init_decode_state_kernel(int* lens, int* finished, int* scalars /*n_finished, ...*/, int B, int max_len) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < B) { lens[i] = max_len; finished[i] = 0; }
    if (i < 4) scalars[i] = 0;
}

__global__ void philox_bits_kernel(uint64_t seed, int site, int T, int B, int C, int utt_offset, uint8_t* out) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= T * B * C) return;
    const int c = idx % C, b = (idx / C) % B, t = idx / (C * B);
    out[idx] = keep_bit(seed, (uint32_t)site, (uint32_t)t, (uint32_t)(utt_offset + b), (uint32_t)c) ? 1 : 0;
}

}  // namespace tts
