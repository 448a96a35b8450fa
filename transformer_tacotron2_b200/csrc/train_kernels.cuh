// Memory-bound kernels of the training step (SURVEY.md 8(a) row a12 and the backward halves of a3, a6, a7, a10):
// weight repacking, operand transposes for the weight-gradient GEMMs, masked BatchNorm (batch statistics, P5),
// LayerNorm backward, activation / dropout backward, loss + its gradient (P13), Adam.
// Rows are m = b * T + t; a row is valid iff t < lens[b]; dropout masks come from the Philox contract (philox.cuh),
// so nothing is stored for them.
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace tts {

// ---------------------------------------------------------------------------------------------- weights
// fp32 master w[(n * K + k) * taps + tap]  ->  bf16 out[tap][n][k]  ([taps][Nw][Kp], zero padded)          (flip = 0)
//                                          ->  bf16 out[tap][k][n] = w[.. taps-1-tap]  ([taps][Kw][Np])      (flip = 1, dgrad)
// every matrix of the model in ONE launch: block -> descriptor (binary search over the first-block table), 2048 elements per block
struct PackDesc { long src_off, dst_off; int N, K, taps, R, Cc, flip; int blk0; int pad_; };
__global__ void __launch_bounds__(256) cast_pack_all_kernel(const PackDesc* __restrict__ descs, int nd, const float* __restrict__ P, bf16* __restrict__ wpack) {
    __shared__ float tile[64][33];
    int lo = 0, hi = nd - 1;
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (descs[mid].blk0 <= (int)blockIdx.x) lo = mid; else hi = mid - 1; }
    const PackDesc d = descs[lo];
    const float* w = P + d.src_off; bf16* out = wpack + d.dst_off;
    if (d.flip) {
        // transposed layout out[tap][k][n] (R = Kw rows, Cc = Np columns): a 32(k) x 64(n) tile through shared memory so that
        // both the fp32 reads (along k) and the bf16 writes (along n) are coalesced
        const int tiles_n = d.Cc >> 6, tiles_k = d.R >> 5, lb = blockIdx.x - d.blk0;
        const int tap = lb / (tiles_k * tiles_n), rem = lb - tap * tiles_k * tiles_n, kt = rem / tiles_n, nt = rem - kt * tiles_n;
        const int st = d.taps - 1 - tap;
        const int kl = threadIdx.x & 31, k = kt * 32 + kl;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int nl = (threadIdx.x >> 5) + 8 * i, n = nt * 64 + nl;
            tile[nl][kl] = (n < d.N && k < d.K) ? w[((long)n * d.K + k) * d.taps + st] : 0.f;
        }
        __syncthreads();
        const int nl = threadIdx.x & 63, n = nt * 64 + nl;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int kk = (threadIdx.x >> 6) + 4 * i;
            out[((long)tap * d.R + kt * 32 + kk) * d.Cc + n] = __float2bfloat16(tile[nl][kk]);
        }
        return;
    }
    const long total = (long)d.taps * d.R * d.Cc, base = (long)(blockIdx.x - d.blk0) * 2048;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const long i = base + j * 256 + threadIdx.x;
        if (i < total) {
            const int c = (int)(i % d.Cc), r = (int)((i / d.Cc) % d.R), tap = (int)(i / ((long)d.Cc * d.R));
            out[i] = __float2bfloat16((r < d.N && c < d.K) ? w[((long)r * d.K + c) * d.taps + tap] : 0.f);
        }
    }
}

// ---------------------------------------------------------------------------------------------- masked BatchNorm (P5)
// number of valid positions of the batch; computed once per block by its first warp (every thread of the block must call it)
TTS_D float n_valid(const int* lens, int B) {
    __shared__ float s_n;
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    if (tid < 32) {
        int n = 0;
        for (int b = tid; b < B; b += 32) n += lens[b];
        n = (int)warp_sum((float)n);
        if (tid == 0) s_n = (float)max(n, 1);
    }
    __syncthreads();
    return s_n;
}

// pass 0: stat[c] += sum_valid x;  pass 1: stat[C + c] += sum_valid (x - mean)^2      (stat zeroed by the caller)
__global__ void bn_stats_kernel(const float* __restrict__ x, int M, int C, int T, int B, const int* __restrict__ lens, float* __restrict__ stat, int pass) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const float n = n_valid(lens, B);
    if (c >= C) return;
    const float mean = pass ? stat[c] / n : 0.f;
    const int rows = (M + gridDim.y - 1) / gridDim.y, r0 = blockIdx.y * rows, r1 = min(M, r0 + rows);
    float acc = 0.f;
    for (int m = r0; m < r1; ++m) {
        if (m % T >= lens[m / T]) continue;
        const float v = x[(long)m * C + c] - mean;
        acc += pass ? v * v : v;
    }
    if (r1 > r0) atomicAdd(stat + pass * C + c, acc);
}

// y = mask * dropbits( act( (x - mean) * rstd * gamma + beta ) ); optional running-stat update by block 0.
// Thread = 4 consecutive channels (C % 4 == 0; blockDim.x = (C / 4) * row lanes, so a thread's channels never change and
// its statistics are hoisted); the 4 keep-bits come from one Philox call.
TTS_D uint32_t keep_bits4(uint64_t seed, uint32_t site, uint32_t t, uint32_t b, uint32_t c) {      // bits 0..3 = channels c..c+3 (c % 4 == 0)
    const uint4 w = philox4x32_10(make_uint4(site, t, b, c >> 7), (uint32_t)seed, (uint32_t)(seed >> 32));
    const uint32_t word = (c >> 5) & 3u;
    const uint32_t v = word == 0 ? w.x : word == 1 ? w.y : word == 2 ? w.z : w.w;
    return (v >> (c & 31u)) & 15u;
}
__global__ void bn_act_fwd_kernel(const float* __restrict__ x, int M, int C, int T, int B, const int* __restrict__ lens, const float* __restrict__ stat,
                                  const float* __restrict__ gamma, const float* __restrict__ beta, float eps, int act, int site, const uint64_t* seedp,
                                  int utt_offset, bf16* __restrict__ out16, int ldo, float* __restrict__ out32, float* run_mean, float* run_var,
                                  float momentum) {
    const uint64_t seed = *seedp;
    const float n = n_valid(lens, B);
    const int c4n = C >> 2, rl = blockDim.x / c4n, cg = threadIdx.x % c4n, rlane = threadIdx.x / c4n, c = cg * 4;
    if (rlane < rl) {
        float sc[4], sh[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float mean = stat[c + k] / n, rstd = rsqrtf(stat[C + c + k] / n + eps);
            sc[k] = rstd * gamma[c + k]; sh[k] = beta[c + k] - mean * sc[k];
        }
        for (int m = blockIdx.x * rl + rlane; m < M; m += gridDim.x * rl) {
            const int b = m / T, t = m - b * T;
            float v[4] = {0.f, 0.f, 0.f, 0.f};
            if (t < lens[b]) {
                const float4 xv = *reinterpret_cast<const float4*>(x + (long)m * C + c);
                const float xs[4] = {xv.x, xv.y, xv.z, xv.w};
                const uint32_t kb = site >= 0 ? keep_bits4(seed, site, t, utt_offset + b, c) : 15u;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    float y = xs[k] * sc[k] + sh[k];
                    if (act == 1) y = fmaxf(y, 0.f); else if (act == 2) y = tanhf(y);
                    v[k] = site >= 0 ? (((kb >> k) & 1u) ? 2.f * y : 0.f) : y;
                }
            }
            if (out16) *reinterpret_cast<uint2*>(out16 + (long)m * ldo + c) = make_uint2(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]));
            if (out32) *reinterpret_cast<float4*>(out32 + (long)m * C + c) = make_float4(v[0], v[1], v[2], v[3]);
        }
    }
    if (run_mean && blockIdx.x == 0)
        for (int cc = threadIdx.x; cc < C; cc += blockDim.x) {
            const float mean = stat[cc] / n, var = stat[C + cc] / n;
            run_mean[cc] = (1.f - momentum) * run_mean[cc] + momentum * mean;
            run_var[cc] = (1.f - momentum) * run_var[cc] + momentum * var * n / fmaxf(n - 1.f, 1.f);
        }
}

// gradient wrt the BN output of element (m, c): dout * mask * dropout * act'
TTS_D float bn_dact(float dout, float xhat_gb, int act, int site, uint64_t seed, int t, int bg, int c) {
    float d = dout;
    if (site >= 0) d = keep_bit(seed, site, t, bg, c) ? 2.f * d : 0.f;
    if (act == 1) d = xhat_gb > 0.f ? d : 0.f;
    else if (act == 2) { const float th = tanhf(xhat_gb); d *= 1.f - th * th; }
    return d;
}
// dbeta[c] += sum_valid g, dgamma[c] += sum_valid g * xhat, with g = d(loss)/d(BN output)
template <typename TD>
__global__ void bn_bwd_reduce_kernel(const TD* __restrict__ dout, int ldd, const float* __restrict__ x, int M, int C, int T, int B,
                                     const int* __restrict__ lens, const float* __restrict__ stat, const float* __restrict__ gamma,
                                     const float* __restrict__ beta, float eps, int act, int site, const uint64_t* seedp, int utt_offset, float* __restrict__ dbeta,
                                     float* __restrict__ dgamma) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const float n = n_valid(lens, B);
    if (c >= C) return;
    const uint64_t seed = *seedp;
    const float mean = stat[c] / n, rstd = rsqrtf(stat[C + c] / n + eps), ga = gamma[c], be = beta[c];
    const int rows = (M + gridDim.y - 1) / gridDim.y, r0 = blockIdx.y * rows, r1 = min(M, r0 + rows);
    float s0 = 0.f, s1 = 0.f;
    for (int m = r0; m < r1; ++m) {
        const int b = m / T, t = m - b * T;
        if (t >= lens[b]) continue;
        const float xh = (x[(long)m * C + c] - mean) * rstd;
        const float g = bn_dact(to_f32(dout[(long)m * ldd + c]), xh * ga + be, act, site, seed, t, utt_offset + b, c);
        s0 += g; s1 += g * xh;
    }
    if (r1 > r0) { atomicAdd(dbeta + c, s0); atomicAdd(dgamma + c, s1); }
}
// dx = gamma * rstd * (g - mean(g) - xhat * mean(g * xhat)) on valid rows, 0 elsewhere  -> bf16   (thread = 4 channels, as above)
TTS_D float load1(const float* p) { return *p; }
TTS_D float load1(const bf16* p) { return __bfloat162float(*p); }
template <typename TD>
__global__ void bn_bwd_apply_kernel(const TD* __restrict__ dout, int ldd, const float* __restrict__ x, int M, int C, int T, int B,
                                    const int* __restrict__ lens, const float* __restrict__ stat, const float* __restrict__ gamma,
                                    const float* __restrict__ beta, float eps, int act, int site, const uint64_t* seedp, int utt_offset,
                                    const float* __restrict__ dbeta, const float* __restrict__ dgamma, bf16* __restrict__ dx, int ldx) {
    const uint64_t seed = *seedp;
    const float n = n_valid(lens, B);
    const int c4n = C >> 2, rl = blockDim.x / c4n, cg = threadIdx.x % c4n, rlane = threadIdx.x / c4n, c = cg * 4;
    if (rlane >= rl) return;
    float mean[4], rstd[4], ga[4], be[4], mg[4], mgx[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        mean[k] = stat[c + k] / n; rstd[k] = rsqrtf(stat[C + c + k] / n + eps); ga[k] = gamma[c + k]; be[k] = beta[c + k];
        mg[k] = dbeta[c + k] / n; mgx[k] = dgamma[c + k] / n;
    }
    for (int m = blockIdx.x * rl + rlane; m < M; m += gridDim.x * rl) {
        const int b = m / T, t = m - b * T;
        float v[4] = {0.f, 0.f, 0.f, 0.f};
        if (t < lens[b]) {
            const float4 xv = *reinterpret_cast<const float4*>(x + (long)m * C + c);
            const float xs[4] = {xv.x, xv.y, xv.z, xv.w};
            const uint32_t kb = site >= 0 ? keep_bits4(seed, site, t, utt_offset + b, c) : 15u;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float xh = (xs[k] - mean[k]) * rstd[k];
                float g = load1(dout + (long)m * ldd + c + k);
                if (site >= 0) g = ((kb >> k) & 1u) ? 2.f * g : 0.f;
                const float yb = xh * ga[k] + be[k];
                if (act == 1) g = yb > 0.f ? g : 0.f;
                else if (act == 2) { const float th = tanhf(yb); g *= 1.f - th * th; }
                v[k] = ga[k] * rstd[k] * (g - mg[k] - xh * mgx[k]);
            }
        }
        *reinterpret_cast<uint2*>(dx + (long)m * ldx + c) = make_uint2(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]));
    }
}

// ---------------------------------------------------------------------------------------------- LayerNorm backward (512)
// warp per row.  dy = rstd * (g - mean(g) - xhat * mean(g * xhat)), g = dx * gamma;  dgamma += dx * xhat, dbeta += dx.
// Outputs: dy32 (the residual path) and dsub16 = dy * keep / (1 - p) of the sub-layer's residual-dropout site (site < 0: plain copy).
__global__ void __launch_bounds__(256) ln_bwd_kernel(const float* __restrict__ dx, const float* __restrict__ ypre, const float* __restrict__ gamma,
                                                     float eps, int M, int T, float* __restrict__ dy32, bf16* __restrict__ dsub16, int site,
                                                     const uint64_t* seedp, int utt_offset, uint32_t thresh, float dscale, float* __restrict__ dgamma,
                                                     float* __restrict__ dbeta) {
    __shared__ float sg[512], sb[512];
    const uint64_t seed = *seedp;
    for (int i = threadIdx.x; i < 512; i += 256) { sg[i] = 0.f; sb[i] = 0.f; }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float ag[16], ab[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) { ag[i] = 0.f; ab[i] = 0.f; }
    for (int m = blockIdx.x * 8 + warp; m < M; m += gridDim.x * 8) {
        float y[16], d[16];
#pragma unroll
        for (int q = 0; q < 4; ++q) {                    // columns lane * 4 + q * 128 + {0..3}
            const float4 a = *reinterpret_cast<const float4*>(ypre + (long)m * 512 + q * 128 + lane * 4);
            const float4 e = *reinterpret_cast<const float4*>(dx + (long)m * 512 + q * 128 + lane * 4);
            y[q * 4] = a.x; y[q * 4 + 1] = a.y; y[q * 4 + 2] = a.z; y[q * 4 + 3] = a.w;
            d[q * 4] = e.x; d[q * 4 + 1] = e.y; d[q * 4 + 2] = e.z; d[q * 4 + 3] = e.w;
        }
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i) s += y[i];
        const float mean = warp_sum(s) * (1.f / 512.f);
        float v = 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i) { y[i] -= mean; v += y[i] * y[i]; }
        const float rstd = rsqrtf(warp_sum(v) * (1.f / 512.f) + eps);
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int c = (i >> 2) * 128 + lane * 4 + (i & 3);
            y[i] *= rstd;                                // xhat
            ag[i] += d[i] * y[i]; ab[i] += d[i];
            d[i] *= gamma[c];                            // g
            s1 += d[i]; s2 += d[i] * y[i];
        }
        s1 = warp_sum(s1) * (1.f / 512.f); s2 = warp_sum(s2) * (1.f / 512.f);
        const int b = m / T, t = m - b * T;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            float o[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) o[i] = rstd * (d[q * 4 + i] - s1 - y[q * 4 + i] * s2);
            const int c = q * 128 + lane * 4;
            if (dy32) *reinterpret_cast<float4*>(dy32 + (long)m * 512 + c) = make_float4(o[0], o[1], o[2], o[3]);
            if (dsub16) {
                if (site >= 0) {
                    const uint4 w = philox4x32_10(make_uint4((uint32_t)site, (uint32_t)t, (uint32_t)(utt_offset + b), (uint32_t)(c >> 2)), (uint32_t)seed, (uint32_t)(seed >> 32));
                    o[0] = w.x >= thresh ? o[0] * dscale : 0.f; o[1] = w.y >= thresh ? o[1] * dscale : 0.f;
                    o[2] = w.z >= thresh ? o[2] * dscale : 0.f; o[3] = w.w >= thresh ? o[3] * dscale : 0.f;
                }
                *reinterpret_cast<uint2*>(dsub16 + (long)m * 512 + c) = make_uint2(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]));
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const int c = (i >> 2) * 128 + lane * 4 + (i & 3);
        atomicAdd(&sg[c], ag[i]); atomicAdd(&sb[c], ab[i]);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 512; i += 256) { atomicAdd(dgamma + i, sg[i]); atomicAdd(dbeta + i, sb[i]); }
}

// ---------------------------------------------------------------------------------------------- element-wise backward pieces
// d = saved > 0 ? d * scale : 0   (ReLU, or ReLU followed by p = 0.5 dropout with scale = 2), bf16 in place, 8 per thread
__global__ void relu_bwd_kernel(bf16* __restrict__ d, const bf16* __restrict__ saved, long n8, float scale) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n8) return;
    uint4 dv = reinterpret_cast<uint4*>(d)[i];
    const uint4 sv = reinterpret_cast<const uint4*>(saved)[i];
    uint32_t* dp = &dv.x; const uint32_t* sp = &sv.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float2 a = unpack_bf16x2(dp[j]), s = unpack_bf16x2(sp[j]);
        dp[j] = pack_bf16x2(s.x > 0.f ? a.x * scale : 0.f, s.y > 0.f ? a.y * scale : 0.f);
    }
    reinterpret_cast<uint4*>(d)[i] = dv;
}

// word-dropout backward of a [M][512] fp32 gradient -> bf16, plus dalpha += sum d * keep * scale * pe[t][c]
__global__ void dropw_bwd_kernel(const float* __restrict__ d, bf16* __restrict__ out, int M, int T, int site, const uint64_t* seedp, int utt_offset,
                                 uint32_t thresh, float dscale, const float* __restrict__ pe, float* __restrict__ dalpha) {
    const uint64_t seed = *seedp;
    float acc = 0.f;
    const long total4 = (long)M * 128;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (long)gridDim.x * blockDim.x) {
        const int m = (int)(i >> 7), c = (int)(i & 127) * 4, b = m / T, t = m - b * T;
        float4 v = reinterpret_cast<const float4*>(d)[i];
        if (site >= 0) {
            const uint4 w = philox4x32_10(make_uint4((uint32_t)site, (uint32_t)t, (uint32_t)(utt_offset + b), (uint32_t)(c >> 2)), (uint32_t)seed, (uint32_t)(seed >> 32));
            v.x = w.x >= thresh ? v.x * dscale : 0.f; v.y = w.y >= thresh ? v.y * dscale : 0.f;
            v.z = w.z >= thresh ? v.z * dscale : 0.f; v.w = w.w >= thresh ? v.w * dscale : 0.f;
        }
        reinterpret_cast<uint2*>(out)[i] = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
        const float4 pv = *reinterpret_cast<const float4*>(pe + (long)t * 512 + c);
        acc += v.x * pv.x + v.y * pv.y + v.z * pv.z + v.w * pv.w;
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) atomicAdd(dalpha, acc);
}

// dE[ph[m]][c] += d[m][c] over valid rows (padding index 0 gets no gradient)
__global__ void embed_bwd_kernel(const bf16* __restrict__ d, const int64_t* __restrict__ ph, const int* __restrict__ lens, int M, int S, int V,
                                 float* __restrict__ dE) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long)M * 512) return;
    const int m = (int)(i >> 9), c = (int)(i & 511), b = m / S, t = m - b * S;
    const int64_t id = ph[m];
    if (t < lens[b] && id > 0 && id < V) atomicAdd(dE + id * 512 + c, __bfloat162float(d[i]));
}

// ---------------------------------------------------------------------------------------------- loss (P13)
// acc[0..2] += sum (before - y)^2, sum (after - y)^2, sum bce over valid frames; gradients wrt the three outputs.
// dhead16 [M][128] = [d mel_before(direct) | d stop | 0...], dafter32 [M][80]
__global__ void loss_kernel(const float* __restrict__ before, const float* __restrict__ after, const float* __restrict__ stop,
                            const float* __restrict__ target, const int* __restrict__ lens, int B, int T, float pos_weight,
                            float* __restrict__ acc, float* __restrict__ dbefore32, float* __restrict__ dafter32, float* __restrict__ dstop32) {
    const float n = n_valid(lens, B);
    const float cm = 2.f / (n * 80.f);
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
    const long total = (long)B * T * 81;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const int m = (int)(i / 81), c = (int)(i % 81), b = m / T, t = m - b * T;
        const bool valid = t < lens[b];
        if (c < 80) {
            const long j = (long)m * 80 + c;
            const float eb = valid ? before[j] - target[j] : 0.f, ea = valid ? after[j] - target[j] : 0.f;
            a0 += eb * eb; a1 += ea * ea;
            dbefore32[j] = eb * cm; dafter32[j] = ea * cm;
        } else {
            float g = 0.f;
            if (valid) {
                const float x = stop[m], y = (t == lens[b] - 1) ? 1.f : 0.f;
                const float sp = fmaxf(-x, 0.f) + log1pf(expf(-fabsf(x)));       // softplus(-x) = -log sigmoid(x)
                a2 += pos_weight * y * sp + (1.f - y) * (x + sp);                // -log(1 - sigmoid(x)) = x + softplus(-x)
                const float sg = 1.f / (1.f + expf(-x));
                g = (sg * (1.f - y) - pos_weight * y * (1.f - sg)) / n;
            }
            dstop32[m] = g;
        }
    }
    a0 = warp_sum(a0); a1 = warp_sum(a1); a2 = warp_sum(a2);
    if ((threadIdx.x & 31) == 0) { atomicAdd(acc, a0); atomicAdd(acc + 1, a1); atomicAdd(acc + 2, a2); }
}
// loss = acc0 / (n * 80) + acc1 / (n * 80) + acc2 / n
__global__ void loss_finalize_kernel(const float* acc, const int* lens, int B, float* loss) {      // one warp
    const float n = n_valid(lens, B);
    if (threadIdx.x == 0) loss[0] = acc[0] / (n * 80.f) + acc[1] / (n * 80.f) + acc[2] / n;
}
// dhead16[m][0..79] = mask * (dbefore + dafter + dpost0), [80] = dstop, rest 0    (mel_after = (mel_before + postnet) * mask)
__global__ void head_grad_kernel(const float* __restrict__ dbefore32, const float* __restrict__ dafter32, const bf16* __restrict__ dpost0, int ldp,
                                 const float* __restrict__ dstop32, const int* __restrict__ lens, int M, int T, bf16* __restrict__ dhead16) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long)M * 128) return;
    const int m = (int)(i >> 7), c = (int)(i & 127), b = m / T, t = m - b * T;
    float v = 0.f;
    if (t < lens[b]) {
        if (c < 80) v = dbefore32[(long)m * 80 + c] + dafter32[(long)m * 80 + c] + __bfloat162float(dpost0[(long)m * ldp + c]);
        else if (c == 80) v = dstop32[m];
    }
    dhead16[i] = __float2bfloat16(v);
}

// ---------------------------------------------------------------------------------------------- launches
// Launch geometry of the kernels above, shared by the training step (train.cuh) and the per-kernel test entry points, so
// that the tests check the launches training runs.
// Masked BatchNorm: the statistics / reduce kernels run one thread per channel over BN_ROW_CHUNKS row chunks, the
// element-wise kernels (C / 4) channel groups x row lanes per block over BN_ELEM_BLOCKS blocks (grid-stride over rows).
constexpr int BN_ROW_CHUNKS = 592, BN_ELEM_BLOCKS = 1184;
constexpr int BN_STAT_FLOATS = 1024;             // stat buffer of one BN layer: [0, C) sums, [C, 2C) centred squares (C <= 512)
inline int bn_threads(int C) { return (C / 4) * std::max(1, 256 / (C / 4)); }

// stat <- batch statistics over the valid rows of x [B * T][C]; y = mask * dropout(act(BN(x))) -> out16 (row stride ldo) and / or
// out32 (row stride C); running statistics updated with momentum 0.1 (unbiased variance) when run_mean is given
inline cudaError_t launch_bn_train_fwd(const float* x, int M, int C, int T, int B, const int* lens, float* stat, const float* gamma,
                                       const float* beta, float eps, int act, int site, const uint64_t* seedp, int utt_offset, bf16* out16,
                                       int ldo, float* out32, float* run_mean, float* run_var, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(stat, 0, BN_STAT_FLOATS * 4, st);
    if (e != cudaSuccess) return e;
    const dim3 g((C + 127) / 128, BN_ROW_CHUNKS);
    bn_stats_kernel<<<g, 128, 0, st>>>(x, M, C, T, B, lens, stat, 0);
    bn_stats_kernel<<<g, 128, 0, st>>>(x, M, C, T, B, lens, stat, 1);
    bn_act_fwd_kernel<<<BN_ELEM_BLOCKS, bn_threads(C), 0, st>>>(x, M, C, T, B, lens, stat, gamma, beta, eps, act, site, seedp, utt_offset, out16, ldo,
                                                               out32, run_mean, run_var, 0.1f);
    launch_counter() += 3;
    return cudaGetLastError();
}
// backward of the same block from dout (row stride ldd): dbeta / dgamma (zero on entry) += their sums, dx (bf16, row stride ldx)
template <typename TD>
inline cudaError_t launch_bn_train_bwd(const TD* dout, int ldd, const float* x, int M, int C, int T, int B, const int* lens, const float* stat,
                                       const float* gamma, const float* beta, float eps, int act, int site, const uint64_t* seedp, int utt_offset,
                                       float* dbeta, float* dgamma, bf16* dx, int ldx, cudaStream_t st) {
    const dim3 g((C + 127) / 128, BN_ROW_CHUNKS);
    bn_bwd_reduce_kernel<TD><<<g, 128, 0, st>>>(dout, ldd, x, M, C, T, B, lens, stat, gamma, beta, eps, act, site, seedp, utt_offset, dbeta, dgamma);
    bn_bwd_apply_kernel<TD><<<BN_ELEM_BLOCKS, bn_threads(C), 0, st>>>(dout, ldd, x, M, C, T, B, lens, stat, gamma, beta, eps, act, site, seedp,
                                                                     utt_offset, dbeta, dgamma, dx, ldx);
    launch_counter() += 2;
    return cudaGetLastError();
}
inline cudaError_t launch_ln_bwd(const float* dx, const float* ypre, const float* gamma, float eps, int M, int T, float* dy32, bf16* dsub16, int site,
                                 const uint64_t* seedp, int utt_offset, uint32_t thresh, float dscale, float* dgamma, float* dbeta, cudaStream_t st) {
    ln_bwd_kernel<<<std::min((M + 7) / 8, 592), 256, 0, st>>>(dx, ypre, gamma, eps, M, T, dy32, dsub16, site, seedp, utt_offset, thresh, dscale,
                                                              dgamma, dbeta);
    ++launch_counter();
    return cudaGetLastError();
}
// acc (16 floats) zeroed, loss and its gradients, loss_out[0] = the scalar loss
inline cudaError_t launch_loss(const float* before, const float* after, const float* stop, const float* target, const int* lens, int B, int T,
                               float pos_weight, float* acc, float* dbefore32, float* dafter32, float* dstop32, float* loss_out, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(acc, 0, 64, st);
    if (e != cudaSuccess) return e;
    const long M = (long)B * T;
    loss_kernel<<<std::min<long>((M * 81 + 255) / 256, 2368), 256, 0, st>>>(before, after, stop, target, lens, B, T, pos_weight, acc, dbefore32,
                                                                            dafter32, dstop32);
    loss_finalize_kernel<<<1, 32, 0, st>>>(acc, lens, B, loss_out);
    launch_counter() += 2;
    return cudaGetLastError();
}
inline cudaError_t launch_head_grad(const float* dbefore32, const float* dafter32, const bf16* dpost0, int ldp, const float* dstop32, const int* lens,
                                    int M, int T, bf16* dhead16, cudaStream_t st) {
    head_grad_kernel<<<(unsigned)(((long)M * 128 + 255) / 256), 256, 0, st>>>(dbefore32, dafter32, dpost0, ldp, dstop32, lens, M, T, dhead16);
    ++launch_counter();
    return cudaGetLastError();
}
// the decoder's word-dropout backward runs on 1184 blocks, the encoder's (fewer rows) on 592
inline cudaError_t launch_dropw_bwd(bool decoder, const float* d, bf16* out, int M, int T, int site, const uint64_t* seedp, int utt_offset,
                                    uint32_t thresh, float dscale, const float* pe, float* dalpha, cudaStream_t st) {
    dropw_bwd_kernel<<<decoder ? 1184 : 592, 256, 0, st>>>(d, out, M, T, site, seedp, utt_offset, thresh, dscale, pe, dalpha);
    ++launch_counter();
    return cudaGetLastError();
}
inline cudaError_t launch_embed_bwd(const bf16* d, const int64_t* ph, const int* lens, int M, int S, int V, float* dE, cudaStream_t st) {
    embed_bwd_kernel<<<(unsigned)(((long)M * 512 + 255) / 256), 256, 0, st>>>(d, ph, lens, M, S, V, dE);
    ++launch_counter();
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------- Adam (Vaswani: beta (0.9, 0.98), eps 1e-9)
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long n, float lr,
                            float beta1, float beta2, float eps, float bc1, float bc2, float grad_scale) {
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
        const float gi = g[i] * grad_scale;
        const float mi = beta1 * m[i] + (1.f - beta1) * gi;
        const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
        m[i] = mi; v[i] = vi;
        p[i] -= lr * (mi / bc1) / (sqrtf(vi / bc2) + eps);
    }
}

// Data-parallel optimiser step as ONE kernel over NVLink peer memory (SURVEY.md 8(f)-1, ZeRO-1 style): this rank owns the
// shard [lo, hi) of the flat parameter buffer.  For every element of its shard it reads the gradient from EVERY rank's
// gradient buffer (reduce-scatter by peer loads), applies Adam with its shard-local moments, and stores the new parameter
// into EVERY rank's parameter buffer (all-gather by peer stores).  16-byte accesses; no staging buffers, no NCCL ring.
struct PeerPtrs { float* P[8]; const float* G[8]; };
__global__ void __launch_bounds__(256) adam_peer_kernel(PeerPtrs pp, int world, float* __restrict__ m, float* __restrict__ v, long lo4, long hi4,
                                                        float lr, float beta1, float beta2, float eps, float bc1, float bc2, float grad_scale) {
    const float4* P0 = reinterpret_cast<const float4*>(pp.P[0]);
    for (long i = lo4 + (long)blockIdx.x * blockDim.x + threadIdx.x; i < hi4; i += (long)gridDim.x * blockDim.x) {
        float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 8
        for (int r = 0; r < world; ++r) {
            const float4 x = __ldcg(reinterpret_cast<const float4*>(pp.G[r]) + i);
            g.x += x.x; g.y += x.y; g.z += x.z; g.w += x.w;
        }
        float4 mm = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i], p = P0[i];
        float* gp = &g.x; float* mp = &mm.x; float* vp = &vv.x; float* ppv = &p.x;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float gi = gp[k] * grad_scale;
            mp[k] = beta1 * mp[k] + (1.f - beta1) * gi;
            vp[k] = beta2 * vp[k] + (1.f - beta2) * gi * gi;
            ppv[k] -= lr * (mp[k] / bc1) / (sqrtf(vp[k] / bc2) + eps);
        }
        reinterpret_cast<float4*>(m)[i] = mm; reinterpret_cast<float4*>(v)[i] = vv;
        for (int r = 0; r < world; ++r) __stcg(reinterpret_cast<float4*>(pp.P[r]) + i, p);
    }
}

}  // namespace tts
