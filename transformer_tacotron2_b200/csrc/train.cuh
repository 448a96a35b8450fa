// Training step of the Transformer-TTS model (SURVEY.md 8(a) row a12, 8(e) "training"): train-mode forward (batch-statistics
// BatchNorm P5, Philox dropout at every site P7/P11/P12), loss P13, full backward, Adam.  Included by tts_b200.cu.
//
// Parameters live in ONE flat fp32 device buffer P (state_dict order rearranged so that tensors used concatenated are
// adjacent: wq|wk|wv, the 12 cross-attention K/V projections, mel|stop heads); gradients G, Adam moments M1 / V2 mirror it,
// so the data-parallel exchange is a single all-reduce over G and Adam is one launch.  bf16 operand copies of every
// matrix (forward layout [taps][N][K] and the transposed / tap-flipped layout the input-gradient GEMM wants) are
// re-derived from P after each optimiser step.
//
// All GEMM-shaped work (forward, input gradients, weight gradients, convolutions as shifted GEMMs) runs on
// gemm_tc_kernel; attention on flash_attn_tc_kernel / flash_attn_bwd_tc_kernel; the rest is train_kernels.cuh.
#pragma once

namespace {

struct TrMat { size_t off; int N, K, taps, Nw, Kp, Kw, Np; size_t fwd_off, bwd_off; bf16 *fwd, *bwd; };
struct TrLin { int mat; size_t b; };
struct TrConv { int mat; size_t b, g, be, rm, rv; int cin, cout; };
struct TrEnc { TrLin qkv, wo, w1, w2; size_t ln1g, ln1b, ln2g, ln2b; };
struct TrDec { TrLin qkv, wo, q2, wo2, w1, w2; size_t ln1g, ln1b, ln2g, ln2b, ln3g, ln3b; };
struct TrEntry { std::string name; size_t off, numel; };

// padded shapes of the two bf16 operand copies of an [N][K][taps] fp32 matrix: forward [taps][Nw][Kp], input gradient [taps][Kw][Np]
TrMat tr_mat_dims(int N, int K, int taps) {
    TrMat m; memset(&m, 0, sizeof(m));
    m.N = N; m.K = K; m.taps = taps;
    m.Nw = round_up(N, 128); m.Kp = round_up(K, 32); m.Kw = round_up(K, 128); m.Np = round_up(N, 64);
    return m;
}
// cast_pack_all_kernel descriptor of one copy (flip = 1: the transposed, tap-reversed input-gradient layout); *blocks = its grid share
PackDesc tr_pack_desc(const TrMat& m, int flip, long src_off, long dst_off, int blk0, int* blocks) {
    PackDesc d; memset(&d, 0, sizeof(d));
    d.src_off = src_off; d.dst_off = dst_off; d.N = m.N; d.K = m.K; d.taps = m.taps;
    d.R = flip ? m.Kw : m.Nw; d.Cc = flip ? m.Np : m.Kp; d.flip = flip; d.blk0 = blk0;
    *blocks = (int)(((long)d.taps * d.R * d.Cc + 2047) / 2048);
    return d;
}
// input-gradient GEMM dX[M][K] = sum_tap dY[m + tap - pad][:Kdy] . Wbwd[tap] over the packed layout [taps][Kw][Np] of m
GemmParams tr_dgrad_params(const TrMat& m, const bf16* wbwd, const bf16* dY, int ldy, int Kdy, int M, int Trows) {
    GemmParams p = gp(dY, ldy, wbwd, m.Np, M, m.K, Kdy);
    p.Nw = m.Kw; p.taps = m.taps; p.T = Trows; p.B = M / Trows;
    return p;
}

}  // namespace

struct TtsTrain {
    std::vector<TrEntry> params, buffers;
    size_t n = 0, nrs = 0, wpack_elems = 0;
    float *P = nullptr, *G = nullptr, *M1 = nullptr, *V2 = nullptr, *RS = nullptr;
    bf16* wpack = nullptr;
    std::vector<TrMat> mats;
    size_t enc_alpha = 0, dec_alpha = 0;
    int embed = 0;
    TrConv enc_conv[3], post_conv[5];
    TrLin enc_proj, fc1, fc2, dproj, ckv, head;
    TrEnc enc[6];
    TrDec dec[6];
    int step = 0;
    PackDesc* pack_descs = nullptr; int n_pack = 0, pack_blocks = 0;
    // data-parallel peers (tts_train_set_peers): every rank's P and G buffers mapped through CUDA IPC; P[rank] / G[rank] are local
    int rank = 0, world = 1;
    PeerPtrs peers{};
    void* ipc_opened[16] = {};
    // the whole forward + loss + backward of one shape as a CUDA graph (~640 launches, launch-bound otherwise): captured on the
    // second step with the same key, replayed afterwards
    struct GraphKey {
        void* ws; int B, S, T, utt0; double p_res; float pos_weight; float* loss_out; cudaStream_t st;
        bool operator==(const GraphKey& o) const {
            return ws == o.ws && B == o.B && S == o.S && T == o.T && utt0 == o.utt0 && p_res == o.p_res && pos_weight == o.pos_weight && loss_out == o.loss_out && st == o.st;
        }
    } graph_key{}, seen_key{};
    cudaGraphExec_t graph_exec = nullptr;
    cudaStream_t cap_stream = nullptr;
    unsigned long long graph_launches = 0;
};

namespace {

int train_free(TtsHandle* h) {
    if (!h->train) return 0;
    TtsTrain* t = h->train;
    for (void* q : t->ipc_opened) if (q) cudaIpcCloseMemHandle(q);
    if (t->graph_exec) cudaGraphExecDestroy(t->graph_exec);
    if (t->cap_stream) cudaStreamDestroy(t->cap_stream);
    for (void* p : {(void*)t->P, (void*)t->G, (void*)t->M1, (void*)t->V2, (void*)t->RS, (void*)t->wpack, (void*)t->pack_descs}) if (p) cudaFree(p);
    delete t;
    h->train = nullptr;
    return 0;
}

// ---- activations kept by the forward pass + scratch of the backward pass -------------------------------------------
struct TrWs {
    size_t total = 0;
    int Mep = 0, Mdp = 0;
    // encoder
    bf16* e[4]; float* ec[3]; bf16* xe[7];
    struct EL { bf16 *qkv, *ctx, *x1, *hdn; float *lse, *y1, *y2; } el[6];
    // decoder
    bf16 *din, *h1, *h2, *xd[7], *kvmem;
    struct DL { bf16 *qkv, *ctx, *x1, *q2, *ctx2, *x2, *hdn; float *lse1, *lse2, *y1, *y2, *y3; } dl[6];
    float *mel_before, *stop, *mel_after, *pc[5], *p5;
    bf16* pp[5];
    float* stat;                // [8][1024] BN batch statistics (3 encoder + 5 postnet convs)
    // loss
    float *acc, *dbefore, *dafter, *dstop;
    // backward scratch
    float *dx, *dxa, *dq32, *dsum;
    bf16 *dsub, *dwide, *dqkv, *dctx, *dkv, *dhead, *dcv, *dcv2;
    int *plens, *mlens;
    int64_t* ph_in; float* mels_in; uint64_t* seed_dev;     // staged inputs: a captured step only ever reads workspace memory
    static TrWs make(unsigned char* base, int B, int S, int T) {
        TrWs w; size_t o = 0;
        auto take = [&](size_t bytes) { size_t r = o; o = align_up(o + bytes, 1024); return base + r; };
        const size_t Me = (size_t)B * S, Md = (size_t)B * T, Mx = Me > Md ? Me : Md;
        w.Mep = (int)((Me + 63) / 64 * 64); w.Mdp = (int)((Md + 63) / 64 * 64);
        for (auto& p : w.e) p = (bf16*)take(Me * 512 * 2);
        for (auto& p : w.ec) p = (float*)take(Me * 512 * 4);
        for (auto& p : w.xe) p = (bf16*)take(Me * 512 * 2);
        for (auto& l : w.el) {
            l.qkv = (bf16*)take(Me * 1536 * 2); l.ctx = (bf16*)take(Me * 512 * 2); l.x1 = (bf16*)take(Me * 512 * 2); l.hdn = (bf16*)take(Me * 2048 * 2);
            l.lse = (float*)take(Me * 8 * 4); l.y1 = (float*)take(Me * 512 * 4); l.y2 = (float*)take(Me * 512 * 4);
        }
        w.din = (bf16*)take(Md * 96 * 2); w.h1 = (bf16*)take(Md * 256 * 2); w.h2 = (bf16*)take(Md * 256 * 2);
        for (auto& p : w.xd) p = (bf16*)take(Md * 512 * 2);
        w.kvmem = (bf16*)take(Me * 6144 * 2);
        for (auto& l : w.dl) {
            l.qkv = (bf16*)take(Md * 1536 * 2); l.ctx = (bf16*)take(Md * 512 * 2); l.x1 = (bf16*)take(Md * 512 * 2); l.q2 = (bf16*)take(Md * 512 * 2);
            l.ctx2 = (bf16*)take(Md * 512 * 2); l.x2 = (bf16*)take(Md * 512 * 2); l.hdn = (bf16*)take(Md * 2048 * 2);
            l.lse1 = (float*)take(Md * 8 * 4); l.lse2 = (float*)take(Md * 8 * 4);
            l.y1 = (float*)take(Md * 512 * 4); l.y2 = (float*)take(Md * 512 * 4); l.y3 = (float*)take(Md * 512 * 4);
        }
        w.mel_before = (float*)take(Md * 80 * 4); w.stop = (float*)take(Md * 4); w.mel_after = (float*)take(Md * 80 * 4);
        for (int i = 0; i < 5; ++i) w.pc[i] = (float*)take(Md * (i == 4 ? 80 : 512) * 4);
        w.p5 = (float*)take(Md * 80 * 4);
        w.pp[0] = (bf16*)take(Md * 96 * 2);
        for (int i = 1; i < 5; ++i) w.pp[i] = (bf16*)take(Md * 512 * 2);
        w.stat = (float*)take(8 * 1024 * 4);
        w.acc = (float*)take(64); w.dbefore = (float*)take(Md * 80 * 4); w.dafter = (float*)take(Md * 80 * 4); w.dstop = (float*)take(Md * 4);
        w.dx = (float*)take(Mx * 512 * 4); w.dxa = (float*)take(Mx * 512 * 4); w.dq32 = (float*)take(Mx * 512 * 4); w.dsum = (float*)take(Mx * 8 * 4);
        w.dsub = (bf16*)take(Mx * 512 * 2); w.dwide = (bf16*)take(Mx * 2048 * 2); w.dqkv = (bf16*)take(Mx * 1536 * 2); w.dctx = (bf16*)take(Mx * 512 * 2);
        w.dkv = (bf16*)take(Me * 6144 * 2); w.dhead = (bf16*)take(Md * 128 * 2);
        w.dcv = (bf16*)take(Mx * 512 * 2); w.dcv2 = (bf16*)take(Mx * 512 * 2);
        w.plens = (int*)take((size_t)B * 4); w.mlens = (int*)take((size_t)B * 4);
        w.ph_in = (int64_t*)take(Me * 8); w.mels_in = (float*)take(Md * 80 * 4); w.seed_dev = (uint64_t*)take(64);
        w.total = o;
        return w;
    }
};

// ---- parameter table --------------------------------------------------------------------------------------------------
int train_build(TtsHandle* h) {
    TtsTrain* t = new TtsTrain();
    h->train = t;
    const TtsConfig& c = h->cfg;
    const int D = 512, F = 2048;
    auto add = [&](const std::string& name, size_t numel) { size_t off = t->n; t->params.push_back({name, off, numel}); t->n += numel; return off; };
    auto pad4 = [&]() { t->n = (t->n + 3) / 4 * 4; };
    auto addbuf = [&](const std::string& name, size_t numel) { size_t off = t->nrs; t->buffers.push_back({name, off, numel}); t->nrs += numel; return off; };
    auto mat = [&](size_t off, int N, int K, int taps) {
        TrMat m = tr_mat_dims(N, K, taps); m.off = off;
        m.fwd_off = t->wpack_elems; t->wpack_elems += (size_t)taps * m.Nw * m.Kp;
        m.bwd_off = t->wpack_elems; t->wpack_elems += (size_t)taps * m.Kw * m.Np;
        m.fwd = m.bwd = nullptr;
        t->mats.push_back(m);
        return (int)t->mats.size() - 1;
    };
    auto lin = [&](const std::string& pre, int N, int K) { TrLin l; size_t w = add(pre + ".weight", (size_t)N * K); l.b = add(pre + ".bias", N); pad4(); l.mat = mat(w, N, K, 1); return l; };
    auto conv = [&](const std::string& pre, int cin, int cout) {
        TrConv cv; cv.cin = cin; cv.cout = cout;
        size_t w = add(pre + ".conv.weight", (size_t)cout * cin * 5); cv.b = add(pre + ".conv.bias", cout);
        cv.g = add(pre + ".bn.weight", cout); cv.be = add(pre + ".bn.bias", cout); pad4();
        cv.rm = addbuf(pre + ".bn.running_mean", cout); cv.rv = addbuf(pre + ".bn.running_var", cout);
        cv.mat = mat(w, cout, cin, 5);
        return cv;
    };
    auto qkv = [&](const std::string& pre) {
        TrLin l; size_t w = add(pre + ".wq.weight", (size_t)D * D); add(pre + ".wk.weight", (size_t)D * D); add(pre + ".wv.weight", (size_t)D * D);
        l.b = add(pre + ".wq.bias", D); add(pre + ".wk.bias", D); add(pre + ".wv.bias", D);
        l.mat = mat(w, 3 * D, D, 1);
        return l;
    };
    t->enc_alpha = add("enc_alpha", 1); pad4();
    t->dec_alpha = add("dec_alpha", 1); pad4();
    { size_t w = add("enc_prenet.embed.weight", (size_t)c.n_vocab * D); t->embed = mat(w, c.n_vocab, D, 1); }
    for (int i = 0; i < 3; ++i) t->enc_conv[i] = conv("enc_prenet.convs." + std::to_string(i), D, D);
    t->enc_proj = lin("enc_prenet.proj", D, D);
    for (int l = 0; l < 6; ++l) {
        const std::string p = "encoder.layers." + std::to_string(l);
        TrEnc& L = t->enc[l];
        L.qkv = qkv(p + ".self_attn"); L.wo = lin(p + ".self_attn.wo", D, D);
        L.ln1g = add(p + ".norm1.weight", D); L.ln1b = add(p + ".norm1.bias", D);
        L.w1 = lin(p + ".ffn.w1", F, D); L.w2 = lin(p + ".ffn.w2", D, F);
        L.ln2g = add(p + ".norm2.weight", D); L.ln2b = add(p + ".norm2.bias", D);
    }
    t->fc1 = lin("dec_prenet.fc1", 256, 80); t->fc2 = lin("dec_prenet.fc2", 256, 256); t->dproj = lin("dec_prenet.proj", D, 256);
    {   // the 12 cross-attention K/V projections as one [6 * 1024][512] matrix
        size_t w0 = 0;
        for (int l = 0; l < 6; ++l) {
            const std::string p = "decoder.layers." + std::to_string(l) + ".cross_attn";
            size_t w = add(p + ".wk.weight", (size_t)D * D); add(p + ".wv.weight", (size_t)D * D);
            if (l == 0) w0 = w;
        }
        for (int l = 0; l < 6; ++l) {
            const std::string p = "decoder.layers." + std::to_string(l) + ".cross_attn";
            size_t b = add(p + ".wk.bias", D); add(p + ".wv.bias", D);
            if (l == 0) t->ckv.b = b;
        }
        t->ckv.mat = mat(w0, 6 * 1024, D, 1);
    }
    for (int l = 0; l < 6; ++l) {
        const std::string p = "decoder.layers." + std::to_string(l);
        TrDec& L = t->dec[l];
        L.qkv = qkv(p + ".self_attn"); L.wo = lin(p + ".self_attn.wo", D, D);
        L.ln1g = add(p + ".norm1.weight", D); L.ln1b = add(p + ".norm1.bias", D);
        L.q2 = lin(p + ".cross_attn.wq", D, D); L.wo2 = lin(p + ".cross_attn.wo", D, D);
        L.ln2g = add(p + ".norm2.weight", D); L.ln2b = add(p + ".norm2.bias", D);
        L.w1 = lin(p + ".ffn.w1", F, D); L.w2 = lin(p + ".ffn.w2", D, F);
        L.ln3g = add(p + ".norm3.weight", D); L.ln3b = add(p + ".norm3.bias", D);
    }
    {   // [mel | stop] heads: 81 x 512
        size_t w = add("mel_linear.weight", (size_t)80 * D); add("stop_linear.weight", D);
        t->head.b = add("mel_linear.bias", 80); add("stop_linear.bias", 1); pad4();
        t->head.mat = mat(w, 81, D, 1);
    }
    for (int i = 0; i < 5; ++i) t->post_conv[i] = conv("postnet.convs." + std::to_string(i), i == 0 ? 80 : 512, i == 4 ? 80 : 512);
    pad4();

    CK(cudaMalloc(&t->P, t->n * 4)); CK(cudaMalloc(&t->G, t->n * 4)); CK(cudaMalloc(&t->M1, t->n * 4)); CK(cudaMalloc(&t->V2, t->n * 4));
    CK(cudaMalloc(&t->RS, t->nrs * 4)); CK(cudaMalloc(&t->wpack, t->wpack_elems * 2));
    CK(cudaMemset(t->P, 0, t->n * 4)); CK(cudaMemset(t->G, 0, t->n * 4)); CK(cudaMemset(t->M1, 0, t->n * 4)); CK(cudaMemset(t->V2, 0, t->n * 4));
    std::vector<float> host(t->n, 0.f), hrs(t->nrs, 0.f);
    for (auto& e : t->params) {
        auto it = h->staged.find(e.name);
        if (it == h->staged.end() || it->second.size() != e.numel) FAIL(TTS_E_WEIGHT, "training: missing or mis-sized weight " + e.name);
        memcpy(&host[e.off], it->second.data(), e.numel * 4);
    }
    for (auto& e : t->buffers) {
        auto it = h->staged.find(e.name);
        if (it == h->staged.end() || it->second.size() != e.numel) FAIL(TTS_E_WEIGHT, "training: missing or mis-sized buffer " + e.name);
        memcpy(&hrs[e.off], it->second.data(), e.numel * 4);
    }
    CK(cudaMemcpy(t->P, host.data(), t->n * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(t->RS, hrs.data(), t->nrs * 4, cudaMemcpyHostToDevice));
    std::vector<PackDesc> descs;
    int blk = 0;
    for (auto& m : t->mats) {
        m.fwd = t->wpack + m.fwd_off; m.bwd = t->wpack + m.bwd_off;
        for (int flip = 0; flip < 2; ++flip) {
            int nblk = 0;
            descs.push_back(tr_pack_desc(m, flip, (long)m.off, (long)(flip ? m.bwd_off : m.fwd_off), blk, &nblk));
            blk += nblk;
        }
    }
    t->n_pack = (int)descs.size(); t->pack_blocks = blk;
    CK(cudaMalloc(&t->pack_descs, descs.size() * sizeof(PackDesc)));
    CK(cudaMemcpy(t->pack_descs, descs.data(), descs.size() * sizeof(PackDesc), cudaMemcpyHostToDevice));
    return 0;
}

// bf16 operand copies of every matrix from the fp32 master (one launch over the descriptor table)
int train_repack(TtsHandle* h, cudaStream_t st) {
    TtsTrain* t = h->train;
    cast_pack_all_kernel<<<t->pack_blocks, 256, 0, st>>>(t->pack_descs, t->n_pack, t->P, t->wpack);
    ++launch_counter();
    CK(cudaGetLastError());
    return 0;
}

// ---- one forward + loss + backward -------------------------------------------------------------------------------------
struct TrCtx {
    TtsHandle* h; TtsTrain* t; TrWs w; cudaStream_t st;
    int B, S, T; const uint64_t* seed; int utt0; uint32_t thresh; float dscale;   // seed: device scalar (graph replays read the new value)
    float* P; float* G;
};

#define TRL(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { c.h->err = std::string(#call) + ": " + cudaGetErrorString(e_); return (int)e_; } } while (0)

// forward GEMM of a linear layer on rows [M][lda]
GemmParams tr_fwd(TrCtx& c, const bf16* A, int lda, int M, int Trows, const TrLin& l) {
    const TrMat& m = c.t->mats[l.mat];
    GemmParams p = gp(A, lda, m.fwd, m.Kp, M, m.N, m.Kp);
    p.T = Trows; p.B = M / Trows; p.bias = c.P + l.b; p.seed_ptr = c.seed; p.utt_offset = c.utt0;
    return p;
}
void tr_dropw(TrCtx& c, GemmParams& p, int site) {
    if (c.thresh == 0) return;
    p.dropw_site = site; p.dropw_thresh = c.thresh; p.dropw_scale = c.dscale;
}
// input-gradient GEMM: dX[M][K] = dY[M][N] . W[N][K]
GemmParams tr_dgrad(TrCtx& c, const bf16* dY, int ldy, int Kdy, int M, int Trows, int mat) {
    const TrMat& m = c.t->mats[mat];
    return tr_dgrad_params(m, m.bwd, dY, ldy, Kdy, M, Trows);
}
// weight gradient dW[N][K * taps] += sum_m dY[m][n] X[m + tap - pad][k] (+ bias gradient), accumulated into G (wgrad_tc.cuh)
int tr_wgrad(TrCtx& c, const bf16* dY, int ldy, const bf16* X, int ldx, int M, int Trows, int mat, size_t bias_off, bool has_bias = true) {
    const TrMat& m = c.t->mats[mat];
    WgradParams g;
    g.dY = dY; g.ldy = ldy; g.Cout = m.N; g.X = X; g.ldx = ldx; g.Cin = m.K; g.taps = m.taps;
    g.T = m.taps > 1 ? Trows : M; g.nb = M / g.T;
    g.dW = c.G + m.off; g.dbias = has_bias ? c.G + bias_off : nullptr;
    TRL(launch_wgrad_tc(g, c.st));
    return 0;
}
int tr_ln_bwd(TrCtx& c, const float* dx, const float* ypre, size_t g_off, size_t b_off, int M, int Trows, int site, float* dy32, bf16* dsub) {
    TRL(launch_ln_bwd(dx, ypre, c.P + g_off, c.h->cfg.ln_eps, M, Trows, dy32, dsub, c.thresh ? site : -1, c.seed, c.utt0, c.thresh, c.dscale,
                      c.G + g_off, c.G + b_off, c.st));
    return 0;
}
AttnBwdParams tr_abwd(const AttnParams& f, const bf16* dO, const float* lse, const float* dsum, float* dQ, bf16* dK, int lddk, bf16* dV, int lddv) {
    return abp_packed(f, dO, lse, dsum, dQ, 512, dK, lddk, dV, lddv);
}
__global__ void f32_to_bf16_strided_kernel(const float* __restrict__ x, bf16* __restrict__ y, long M, int ldo) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;          // one thread per 4 columns of a 512-wide row
    if (i >= M * 128) return;
    const long m = i >> 7; const int cq = (int)(i & 127) * 4;
    const float4 v = reinterpret_cast<const float4*>(x)[i];
    *reinterpret_cast<uint2*>(y + m * ldo + cq) = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
}
__global__ void add_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ o, long n) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) o[i] = a[i] + b[i];
}

// attention backward of one (self / cross) block; dQ lands (bf16) in dq16 with row stride lddq
int tr_attn_bwd(TrCtx& c, const AttnParams& f, const bf16* O, const bf16* dO, const float* lse, bf16* dq16, int lddq, bf16* dK, int lddk, bf16* dV, int lddv) {
    const long nq = (long)f.B * f.Lq * 512;
    const bool single = f.Lk <= 128;                   // one key tile (cross-attention at S <= 128): dQ needs no accumulation across CTAs
    if (!single) TRL(cudaMemsetAsync(c.w.dq32, 0, nq * 4, c.st));
    attn_dsum_kernel<<<(f.B * f.H * f.Lq + 31) / 32, 256, 0, c.st>>>(O, dO, f.o_bs, f.o_hs, f.o_rs, c.w.dsum, f.B, f.H, f.Lq);
    ++launch_counter();
    AttnBwdParams a = tr_abwd(f, dO, lse, c.w.dsum, c.w.dq32, dK, lddk, dV, lddv);
    if (single) { a.dQ16 = dq16; a.dq16_bs = (long)f.Lq * lddq; a.dq16_hs = 64; a.dq16_rs = lddq; }
    TRL(launch_flash_attn_bwd_tc(a, c.st));
    if (!single) {
        f32_to_bf16_strided_kernel<<<(unsigned)((nq / 4 + 255) / 256), 256, 0, c.st>>>(c.w.dq32, dq16, (long)f.B * f.Lq, lddq);
        ++launch_counter();
    }
    TRL(cudaGetLastError());
    return 0;
}

// conv + masked batch-statistics BN + activation + dropout (forward)
int tr_conv_fwd(TrCtx& c, const TrConv& cv, const bf16* in, int ldin, int M, int Trows, const int* lens, float* pre, float* stat, int act, int site,
                bf16* out16, int ldo, float* out32) {
    const TrMat& m = c.t->mats[cv.mat];
    GemmParams p = gp(in, ldin, m.fwd, m.Kp, M, m.N, m.Kp);
    p.taps = 5; p.T = Trows; p.B = M / Trows; p.bias = c.P + cv.b; p.out_f32 = pre; p.ldo = m.N;
    TRL(launch_gemm_tc(p, c.st));
    TRL(launch_bn_train_fwd(pre, M, m.N, Trows, c.B, lens, stat, c.P + cv.g, c.P + cv.be, c.h->cfg.bn_eps, act, site, c.seed, c.utt0, out16, ldo,
                            out32, c.t->RS + cv.rm, c.t->RS + cv.rv, c.st));
    return 0;
}
// backward of the same block: dout (grad wrt the block output) -> dpre (bf16 [M][N]), parameter gradients, input gradient din16
template <typename TD>
int tr_conv_bwd(TrCtx& c, const TrConv& cv, const TD* dout, int ldd, const float* pre, const float* stat, const bf16* in, int ldin, int M, int Trows,
                const int* lens, int act, int site, bf16* dpre, bf16* din16, int ldi) {
    const TrMat& m = c.t->mats[cv.mat];
    TRL(launch_bn_train_bwd<TD>(dout, ldd, pre, M, m.N, Trows, c.B, lens, stat, c.P + cv.g, c.P + cv.be, c.h->cfg.bn_eps, act, site, c.seed, c.utt0,
                                c.G + cv.be, c.G + cv.g, dpre, m.N, c.st));
    int r = tr_wgrad(c, dpre, m.N, in, ldin, M, Trows, cv.mat, cv.b);
    if (r) return r;
    if (din16) {
        GemmParams p = tr_dgrad(c, dpre, m.N, m.N, M, Trows, cv.mat);
        p.out_bf16 = din16; p.ldo = ldi;
        TRL(launch_gemm_tc(p, c.st));
    }
    return 0;
}

// The training step in three parts: forward, loss, backward (tts_train_step runs all three through train_forward_backward; the
// module's autograd bridge -- tts_train_forward / tts_train_backward -- runs the first and, with the caller's output gradients, the third).
// ---- train-mode forward: every activation the backward pass needs stays in the workspace
int train_forward(TrCtx& c) {
    TtsHandle* h = c.h; TtsTrain* t = c.t; TrWs& w = c.w; cudaStream_t st = c.st;
    const int B = c.B, S = c.S, T = c.T, Me = B * S, Md = B * T;
    const float eps = h->cfg.ln_eps;
    const int* plens = w.plens; const int* mlens = w.mlens;
    const int64_t* ph = w.ph_in; const float* mels = w.mels_in;
    // ================================================================ forward (train mode)
    embed_kernel<<<(Me + 3) / 4, 256, 0, st>>>(ph, plens, t->mats[t->embed].fwd, w.e[0], B, S, h->cfg.n_vocab);
    ++launch_counter();
    for (int i = 0; i < 3; ++i) {
        int r = tr_conv_fwd(c, t->enc_conv[i], w.e[i], 512, Me, S, plens, w.ec[i], w.stat + i * 1024, 1, SITE_ENC_PRENET_CONV0 + i, w.e[i + 1], 512, nullptr);
        if (r) return r;
    }
    {
        GemmParams p = tr_fwd(c, w.e[3], 512, Me, S, t->enc_proj);
        p.pe = h->pe; p.alpha_ptr = c.P + t->enc_alpha; tr_dropw(c, p, SITE_ENC_PE); p.out_bf16 = w.xe[0]; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
    }
    for (int l = 0; l < 6; ++l) {
        const TrEnc& L = t->enc[l]; auto& a = w.el[l];
        GemmParams p = tr_fwd(c, w.xe[l], 512, Me, S, L.qkv); p.out_bf16 = a.qkv; p.ldo = 1536;
        TRL(launch_gemm_tc(p, st));
        AttnParams at = ap_packed(a.qkv, 1536, a.qkv + 512, 1536, a.qkv + 1024, 1536, a.ctx, 512, B, S, S, plens, 0); at.lse = a.lse;
        TRL(launch_flash_attn_tc(at, st));
        p = tr_fwd(c, a.ctx, 512, Me, S, L.wo); tr_dropw(c, p, SITE_ENC_LAYER0 + 2 * l); p.resid_bf16 = w.xe[l]; p.ldr = 512; p.out_f32 = a.y1; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
        TRL(layernorm(a.y1, c.P + L.ln1g, c.P + L.ln1b, a.x1, nullptr, Me, eps, st));
        p = tr_fwd(c, a.x1, 512, Me, S, L.w1); p.act = ACT_RELU; p.out_bf16 = a.hdn; p.ldo = 2048;
        TRL(launch_gemm_tc(p, st));
        p = tr_fwd(c, a.hdn, 2048, Me, S, L.w2); tr_dropw(c, p, SITE_ENC_LAYER0 + 2 * l + 1); p.resid_bf16 = a.x1; p.ldr = 512; p.out_f32 = a.y2; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
        TRL(layernorm(a.y2, c.P + L.ln2g, c.P + L.ln2b, w.xe[l + 1], nullptr, Me, eps, st));
    }
    const bf16* mem = w.xe[6];
    {
        GemmParams p = tr_fwd(c, mem, 512, Me, S, t->ckv); p.out_bf16 = w.kvmem; p.ldo = 6144;
        TRL(launch_gemm_tc(p, st));
    }
    mel_to_bf16_kernel<<<(Md * 24 + 255) / 256, 256, 0, st>>>(mels, T, nullptr, 1, w.din, nullptr, B, T);
    ++launch_counter();
    {
        GemmParams p = tr_fwd(c, w.din, 96, Md, T, t->fc1); p.act = ACT_RELU; p.drop_site = SITE_DEC_PRENET_FC1; p.out_bf16 = w.h1; p.ldo = 256;
        TRL(launch_gemm_tc(p, st));
        p = tr_fwd(c, w.h1, 256, Md, T, t->fc2); p.act = ACT_RELU; p.drop_site = SITE_DEC_PRENET_FC2; p.out_bf16 = w.h2; p.ldo = 256;
        TRL(launch_gemm_tc(p, st));
        p = tr_fwd(c, w.h2, 256, Md, T, t->dproj); p.pe = h->pe; p.alpha_ptr = c.P + t->dec_alpha; tr_dropw(c, p, SITE_DEC_PE); p.out_bf16 = w.xd[0]; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
    }
    for (int l = 0; l < 6; ++l) {
        const TrDec& L = t->dec[l]; auto& a = w.dl[l];
        const int s0 = SITE_DEC_LAYER0 + 3 * l;
        GemmParams p = tr_fwd(c, w.xd[l], 512, Md, T, L.qkv); p.out_bf16 = a.qkv; p.ldo = 1536;
        TRL(launch_gemm_tc(p, st));
        AttnParams at = ap_packed(a.qkv, 1536, a.qkv + 512, 1536, a.qkv + 1024, 1536, a.ctx, 512, B, T, T, mlens, 1); at.lse = a.lse1;
        TRL(launch_flash_attn_tc(at, st));
        p = tr_fwd(c, a.ctx, 512, Md, T, L.wo); tr_dropw(c, p, s0); p.resid_bf16 = w.xd[l]; p.ldr = 512; p.out_f32 = a.y1; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
        TRL(layernorm(a.y1, c.P + L.ln1g, c.P + L.ln1b, a.x1, nullptr, Md, eps, st));
        p = tr_fwd(c, a.x1, 512, Md, T, L.q2); p.out_bf16 = a.q2; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
        at = ap_packed(a.q2, 512, w.kvmem + l * 1024, 6144, w.kvmem + l * 1024 + 512, 6144, a.ctx2, 512, B, T, S, plens, 0); at.lse = a.lse2;
        TRL(launch_flash_attn_tc(at, st));
        p = tr_fwd(c, a.ctx2, 512, Md, T, L.wo2); tr_dropw(c, p, s0 + 1); p.resid_bf16 = a.x1; p.ldr = 512; p.out_f32 = a.y2; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
        TRL(layernorm(a.y2, c.P + L.ln2g, c.P + L.ln2b, a.x2, nullptr, Md, eps, st));
        p = tr_fwd(c, a.x2, 512, Md, T, L.w1); p.act = ACT_RELU; p.out_bf16 = a.hdn; p.ldo = 2048;
        TRL(launch_gemm_tc(p, st));
        p = tr_fwd(c, a.hdn, 2048, Md, T, L.w2); tr_dropw(c, p, s0 + 2); p.resid_bf16 = a.x2; p.ldr = 512; p.out_f32 = a.y3; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
        TRL(layernorm(a.y3, c.P + L.ln3g, c.P + L.ln3b, w.xd[l + 1], nullptr, Md, eps, st));
    }
    {
        GemmParams p = tr_fwd(c, w.xd[6], 512, Md, T, t->head);
        p.lens = mlens; p.scatter = SC_HEAD; p.out_f32 = w.mel_before; p.out2_f32 = w.stop;
        TRL(launch_gemm_tc(p, st));
    }
    mel_to_bf16_kernel<<<(Md * 24 + 255) / 256, 256, 0, st>>>(w.mel_before, T, mlens, 0, w.pp[0], nullptr, B, T);
    ++launch_counter();
    for (int i = 0; i < 5; ++i) {
        int r = tr_conv_fwd(c, t->post_conv[i], w.pp[i], i == 0 ? 96 : 512, Md, T, mlens, w.pc[i], w.stat + (3 + i) * 1024, i < 4 ? 2 : 0, SITE_POSTNET_CONV0 + i,
                            i < 4 ? w.pp[i + 1] : nullptr, 512, i < 4 ? nullptr : w.p5);
        if (r) return r;
    }
    add_kernel<<<(unsigned)(((long)Md * 80 + 255) / 256), 256, 0, st>>>(w.mel_before, w.p5, w.mel_after, (long)Md * 80);
    ++launch_counter();

    TRL(cudaGetLastError());
    return 0;
}
// ---- backward from the output gradients in w.dbefore [Md][80], w.dafter [Md][80], w.dstop [Md] (fp32) into the flat gradient buffer
int train_backward(TrCtx& c) {
    TtsHandle* h = c.h; TtsTrain* t = c.t; TrWs& w = c.w; cudaStream_t st = c.st;
    const int B = c.B, S = c.S, T = c.T, Me = B * S, Md = B * T;
    const int* plens = w.plens; const int* mlens = w.mlens;
    const int64_t* ph = w.ph_in;
    TRL(cudaMemsetAsync(c.G, 0, t->n * 4, st));
    // ================================================================ backward
    // postnet: d mel_after flows into conv 4 .. 0
    {
        int r = tr_conv_bwd<float>(c, t->post_conv[4], w.dafter, 80, w.pc[4], w.stat + 7 * 1024, w.pp[4], 512, Md, T, mlens, 0, SITE_POSTNET_CONV0 + 4, w.dcv, w.dcv2, 512);
        if (r) return r;
        bf16 *din = w.dcv2, *tmp = w.dsub;              // gradient wrt the block output / spare
        for (int i = 3; i >= 0; --i) {
            r = tr_conv_bwd<bf16>(c, t->post_conv[i], din, 512, w.pc[i], w.stat + (3 + i) * 1024, w.pp[i], i == 0 ? 96 : 512, Md, T, mlens, 2, SITE_POSTNET_CONV0 + i,
                                  w.dcv, tmp, i == 0 ? 96 : 512);
            if (r) return r;
            std::swap(din, tmp);
        }
        // din now holds d(postnet input) as bf16 [Md][96]
        TRL(launch_head_grad(w.dbefore, w.dafter, din, 96, w.dstop, mlens, Md, T, w.dhead, st));
    }
    {   // heads
        int r = tr_wgrad(c, w.dhead, 128, w.xd[6], 512, Md, T, t->head.mat, t->head.b);
        if (r) return r;
        GemmParams p = tr_dgrad(c, w.dhead, 128, 128, Md, T, t->head.mat); p.out_f32 = w.dx; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
    }
    TRL(cudaMemsetAsync(w.dkv, 0, (size_t)Me * 6144 * 2, st));
    for (int l = 5; l >= 0; --l) {
        const TrDec& L = t->dec[l]; auto& a = w.dl[l];
        const int s0 = SITE_DEC_LAYER0 + 3 * l;
        int r;
        // ---- FFN
        if ((r = tr_ln_bwd(c, w.dx, a.y3, L.ln3g, L.ln3b, Md, T, s0 + 2, w.dxa, w.dsub))) return r;
        if ((r = tr_wgrad(c, w.dsub, 512, a.hdn, 2048, Md, T, L.w2.mat, L.w2.b))) return r;
        GemmParams p = tr_dgrad(c, w.dsub, 512, 512, Md, T, L.w2.mat); p.out_bf16 = w.dwide; p.ldo = 2048;
        TRL(launch_gemm_tc(p, st));
        relu_bwd_kernel<<<(unsigned)(((long)Md * 256 + 255) / 256), 256, 0, st>>>(w.dwide, a.hdn, (long)Md * 256, 1.f);
        ++launch_counter();
        if ((r = tr_wgrad(c, w.dwide, 2048, a.x2, 512, Md, T, L.w1.mat, L.w1.b))) return r;
        p = tr_dgrad(c, w.dwide, 2048, 2048, Md, T, L.w1.mat); p.resid_f32 = w.dxa; p.ldr = 512; p.out_f32 = w.dx; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
        // ---- cross attention
        if ((r = tr_ln_bwd(c, w.dx, a.y2, L.ln2g, L.ln2b, Md, T, s0 + 1, w.dxa, w.dsub))) return r;
        if ((r = tr_wgrad(c, w.dsub, 512, a.ctx2, 512, Md, T, L.wo2.mat, L.wo2.b))) return r;
        p = tr_dgrad(c, w.dsub, 512, 512, Md, T, L.wo2.mat); p.out_bf16 = w.dctx; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
        AttnParams at = ap_packed(a.q2, 512, w.kvmem + l * 1024, 6144, w.kvmem + l * 1024 + 512, 6144, a.ctx2, 512, B, T, S, plens, 0);
        if ((r = tr_attn_bwd(c, at, a.ctx2, w.dctx, a.lse2, w.dqkv, 512, w.dkv + l * 1024, 6144, w.dkv + l * 1024 + 512, 6144))) return r;
        if ((r = tr_wgrad(c, w.dqkv, 512, a.x1, 512, Md, T, L.q2.mat, L.q2.b))) return r;
        p = tr_dgrad(c, w.dqkv, 512, 512, Md, T, L.q2.mat); p.resid_f32 = w.dxa; p.ldr = 512; p.out_f32 = w.dx; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
        // ---- causal self attention
        if ((r = tr_ln_bwd(c, w.dx, a.y1, L.ln1g, L.ln1b, Md, T, s0, w.dxa, w.dsub))) return r;
        if ((r = tr_wgrad(c, w.dsub, 512, a.ctx, 512, Md, T, L.wo.mat, L.wo.b))) return r;
        p = tr_dgrad(c, w.dsub, 512, 512, Md, T, L.wo.mat); p.out_bf16 = w.dctx; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
        at = ap_packed(a.qkv, 1536, a.qkv + 512, 1536, a.qkv + 1024, 1536, a.ctx, 512, B, T, T, mlens, 1);
        if ((r = tr_attn_bwd(c, at, a.ctx, w.dctx, a.lse1, w.dqkv, 1536, w.dqkv + 512, 1536, w.dqkv + 1024, 1536))) return r;
        if ((r = tr_wgrad(c, w.dqkv, 1536, w.xd[l], 512, Md, T, L.qkv.mat, L.qkv.b))) return r;
        p = tr_dgrad(c, w.dqkv, 1536, 1536, Md, T, L.qkv.mat); p.resid_f32 = w.dxa; p.ldr = 512; p.out_f32 = w.dx; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
    }
    {   // decoder prenet
        TRL(launch_dropw_bwd(true, w.dx, w.dsub, Md, T, c.thresh ? (int)SITE_DEC_PE : -1, c.seed, c.utt0, c.thresh, c.dscale, h->pe, c.G + t->dec_alpha, st));
        int r;
        if ((r = tr_wgrad(c, w.dsub, 512, w.h2, 256, Md, T, t->dproj.mat, t->dproj.b))) return r;
        GemmParams p = tr_dgrad(c, w.dsub, 512, 512, Md, T, t->dproj.mat); p.out_bf16 = w.dctx; p.ldo = 256;
        TRL(launch_gemm_tc(p, st));
        relu_bwd_kernel<<<(unsigned)(((long)Md * 32 + 255) / 256), 256, 0, st>>>(w.dctx, w.h2, (long)Md * 32, 2.f);
        ++launch_counter();
        if ((r = tr_wgrad(c, w.dctx, 256, w.h1, 256, Md, T, t->fc2.mat, t->fc2.b))) return r;
        p = tr_dgrad(c, w.dctx, 256, 256, Md, T, t->fc2.mat); p.out_bf16 = w.dcv; p.ldo = 256;
        TRL(launch_gemm_tc(p, st));
        relu_bwd_kernel<<<(unsigned)(((long)Md * 32 + 255) / 256), 256, 0, st>>>(w.dcv, w.h1, (long)Md * 32, 2.f);
        ++launch_counter();
        if ((r = tr_wgrad(c, w.dcv, 256, w.din, 96, Md, T, t->fc1.mat, t->fc1.b))) return r;
    }
    {   // cross-attention K/V projections -> gradient of the encoder memory
        int r = tr_wgrad(c, w.dkv, 6144, w.xe[6], 512, Me, S, t->ckv.mat, t->ckv.b);
        if (r) return r;
        GemmParams p = tr_dgrad(c, w.dkv, 6144, 6144, Me, S, t->ckv.mat); p.out_f32 = w.dx; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
    }
    for (int l = 5; l >= 0; --l) {
        const TrEnc& L = t->enc[l]; auto& a = w.el[l];
        int r;
        if ((r = tr_ln_bwd(c, w.dx, a.y2, L.ln2g, L.ln2b, Me, S, SITE_ENC_LAYER0 + 2 * l + 1, w.dxa, w.dsub))) return r;
        if ((r = tr_wgrad(c, w.dsub, 512, a.hdn, 2048, Me, S, L.w2.mat, L.w2.b))) return r;
        GemmParams p = tr_dgrad(c, w.dsub, 512, 512, Me, S, L.w2.mat); p.out_bf16 = w.dwide; p.ldo = 2048;
        TRL(launch_gemm_tc(p, st));
        relu_bwd_kernel<<<(unsigned)(((long)Me * 256 + 255) / 256), 256, 0, st>>>(w.dwide, a.hdn, (long)Me * 256, 1.f);
        ++launch_counter();
        if ((r = tr_wgrad(c, w.dwide, 2048, a.x1, 512, Me, S, L.w1.mat, L.w1.b))) return r;
        p = tr_dgrad(c, w.dwide, 2048, 2048, Me, S, L.w1.mat); p.resid_f32 = w.dxa; p.ldr = 512; p.out_f32 = w.dx; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
        if ((r = tr_ln_bwd(c, w.dx, a.y1, L.ln1g, L.ln1b, Me, S, SITE_ENC_LAYER0 + 2 * l, w.dxa, w.dsub))) return r;
        if ((r = tr_wgrad(c, w.dsub, 512, a.ctx, 512, Me, S, L.wo.mat, L.wo.b))) return r;
        p = tr_dgrad(c, w.dsub, 512, 512, Me, S, L.wo.mat); p.out_bf16 = w.dctx; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
        AttnParams at = ap_packed(a.qkv, 1536, a.qkv + 512, 1536, a.qkv + 1024, 1536, a.ctx, 512, B, S, S, plens, 0);
        if ((r = tr_attn_bwd(c, at, a.ctx, w.dctx, a.lse, w.dqkv, 1536, w.dqkv + 512, 1536, w.dqkv + 1024, 1536))) return r;
        if ((r = tr_wgrad(c, w.dqkv, 1536, w.xe[l], 512, Me, S, L.qkv.mat, L.qkv.b))) return r;
        p = tr_dgrad(c, w.dqkv, 1536, 1536, Me, S, L.qkv.mat); p.resid_f32 = w.dxa; p.ldr = 512; p.out_f32 = w.dx; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
    }
    {   // encoder prenet
        TRL(launch_dropw_bwd(false, w.dx, w.dsub, Me, S, c.thresh ? (int)SITE_ENC_PE : -1, c.seed, c.utt0, c.thresh, c.dscale, h->pe, c.G + t->enc_alpha, st));
        int r;
        if ((r = tr_wgrad(c, w.dsub, 512, w.e[3], 512, Me, S, t->enc_proj.mat, t->enc_proj.b))) return r;
        GemmParams p = tr_dgrad(c, w.dsub, 512, 512, Me, S, t->enc_proj.mat); p.out_bf16 = w.dctx; p.ldo = 512;
        TRL(launch_gemm_tc(p, st));
        bf16 *din = w.dctx, *tmp = w.dsub;
        for (int i = 2; i >= 0; --i) {
            r = tr_conv_bwd<bf16>(c, t->enc_conv[i], din, 512, w.ec[i], w.stat + i * 1024, w.e[i], 512, Me, S, plens, 1, SITE_ENC_PRENET_CONV0 + i, w.dcv, tmp, 512);
            if (r) return r;
            std::swap(din, tmp);
        }
        TRL(launch_embed_bwd(din, ph, plens, Me, S, h->cfg.n_vocab, c.G + t->mats[t->embed].off, st));
    }
    TRL(cudaGetLastError());
    return 0;
}

int train_forward_backward(TrCtx& c, float* loss_out, float pos_weight) {
    int r = train_forward(c);
    if (r) return r;
    // loss P13 and its gradient with respect to (mel_before, mel_after, stop_logits) -> w.dbefore / w.dafter / w.dstop
    const TrWs& w = c.w;
    TRL(launch_loss(w.mel_before, w.mel_after, w.stop, w.mels_in, w.mlens, c.B, c.T, pos_weight, w.acc, w.dbefore, w.dafter, w.dstop, loss_out, c.st));
    return train_backward(c);
}

__global__ void set_u64_kernel(uint64_t* p, uint64_t v) { *p = v; }

}  // namespace
