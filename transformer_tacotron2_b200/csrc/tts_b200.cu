// libtts_b200.so -- C ABI (include/tts_b200.h) over the sm_100a kernels.  Host-side orchestration:
// weight packing, workspace carving, encoder / decode-loop / postnet / teacher-forced schedules.
// No CPU fallback: every entry point launches CUDA kernels or fails.
#include "../../include/tts_b200.h"

#include <algorithm>
#include <cuda.h>
#include <cstdio>
#include <cstring>
#include <cmath>
#include <map>
#include <string>
#include <vector>

#include "common.cuh"
#include "philox.cuh"
#include "gemm_tc.cuh"
#include "attention_tc.cuh"
#include "attention_bwd_tc.cuh"
#include "misc_kernels.cuh"
#include "decode_cluster.cuh"
#include "train_kernels.cuh"
#include "wgrad_tc.cuh"
#include "align.cuh"
#include "speaker.cuh"

using namespace tts;

static inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// ------------------------------------------------------------------------------------------------
// Workspace layout
struct Ws {
    size_t total = 0;
    size_t self_kv, cross_kv, mel_before, stop_logits, lens, finished, scalars, ts, utt_ids, tlens;
    size_t x, x2, wide, a, y, mel16, mel32, ph, plens, mlens;         // sequence-parallel activations
    size_t sids, spembs, cond, nhat;                                  // speaker conditioning (cond_dim >= 0 only)
    int Tpad, Spad, nblk_self, nblk_cross;
    bool has_cond = false;
    size_t self_kv_bytes, cross_kv_bytes;
    // cond_dim >= 0: the handle is speaker-conditioned with x-vectors of cond_dim floats (0: speaker ids only).  Its region comes
    // first, so that tts_set_conditioning finds it from B alone; an unconditioned layout is unchanged.
    static Ws make(int B, int S, int T, int cond_dim = -1) {
        Ws w; size_t o = 0;
        auto take = [&](size_t bytes) { size_t r = o; o = align_up(o + bytes); return r; };
        if (cond_dim >= 0) {
            w.has_cond = true;
            w.sids = take((size_t)B * 4); w.spembs = take((size_t)B * cond_dim * 4 + 4);
            w.cond = take((size_t)B * kDModel * 4); w.nhat = take((size_t)B * cond_dim * 4 + 4);
        }
        const size_t P = (size_t)B * kHeads;
        const size_t M = (size_t)B * (size_t)(S > T ? S : T);
        w.Tpad = (T + 15) / 16 * 16; w.Spad = (S + 15) / 16 * 16;
        // K/V caches of the decode kernel: 64-row blocks of 16 KB (K + V interleaved, decode_cluster.cuh).  The teacher-forced
        // path keeps its cross K/V row-major in the same region ([6][2][B][H][Spad][64], never larger).
        w.nblk_self = (T + KV_BLOCK_ROWS - 1) / KV_BLOCK_ROWS; w.nblk_cross = (S + KV_BLOCK_ROWS - 1) / KV_BLOCK_ROWS;
        w.self_kv_bytes = (size_t)6 * P * w.nblk_self * KV_BLOCK_ELEMS * 2;
        w.cross_kv_bytes = (size_t)6 * P * w.nblk_cross * KV_BLOCK_ELEMS * 2;
        w.self_kv = take(w.self_kv_bytes);
        w.cross_kv = take(w.cross_kv_bytes);
        w.mel_before = take((size_t)B * T * 80 * 4);
        w.stop_logits = take((size_t)B * T * 4);
        w.lens = take(B * 4); w.finished = take(B * 4); w.scalars = take(64);          // scalars: [0] n_finished, [1] group queue
        w.utt_ids = take(B * 4); w.tlens = take(B * 4);
        w.ts = take((size_t)(T + 1) * CL_TS_COLS * 8);
        w.x = take(M * 512 * 2); w.x2 = take(M * 512 * 2); w.wide = take(M * 2048 * 2); w.a = take(M * 512 * 2);
        w.y = take(M * 512 * 4); w.mel16 = take(M * 96 * 2); w.mel32 = take(M * 80 * 4);
        w.ph = take((size_t)B * S * 8); w.plens = take(B * 4); w.mlens = take(B * 4);
        w.total = o;
        return w;
    }
};
template <typename T> static inline T* wsp(void* ws, size_t off) { return reinterpret_cast<T*>(reinterpret_cast<unsigned char*>(ws) + off); }

struct TtsTrain;
// ------------------------------------------------------------------------------------------------
struct TtsHandle {
    TtsConfig cfg;
    int device = 0, num_sms = 0;
    std::string err;
    std::map<std::string, std::vector<float>> staged;
    bool finalized = false;
    int decode_timestamps = 0, decode_debug = 0;
    int cluster_group = 0;                                            // utterances per cluster (1..8); 0 = auto
    int cluster_ok = -1, max_clusters = 0;                            // probed lazily
    unsigned char* cl_wpack = nullptr;                                // [16][CLW_RANK_BYTES] (own allocation)
    unsigned char* arena = nullptr; size_t arena_bytes = 0;
    // ---- device weights (pointers into arena)
    bf16* embed = nullptr;
    bf16* enc_conv_w[3] = {}; float* enc_conv_b[3] = {};
    bf16* enc_proj_w = nullptr; float* enc_proj_b = nullptr;
    float enc_alpha = 1.f, dec_alpha = 1.f;
    struct EncLayer { bf16 *wqkv, *wo, *w1, *w2; float *bqkv, *bo, *b1, *b2, *ln1g, *ln1b, *ln2g, *ln2b; } enc[6];
    bf16* ckv_w = nullptr; float* ckv_b = nullptr;                   // [6*1024][512]
    struct DecLayer {
        bf16 *wqkv, *wo, *wq2, *wo2, *w1, *w2;                       // row-major (teacher-forced GEMMs)
        float *bqkv, *bo, *bq2, *bo2, *b1, *b2, *ln1g, *ln1b, *ln2g, *ln2b, *ln3g, *ln3b;
    } dec[6];
    bf16 *pre_fc1, *pre_fc2, *pre_proj, *head_w;
    float *pre_b1, *pre_b2, *pre_bp, *head_b;
    bf16* post_w[5] = {}; float* post_b[5] = {};
    float* pe = nullptr;
    float *spk_table = nullptr, *spk_w = nullptr, *spk_b = nullptr;  // fp32 speaker-ID table [n_speakers][512], x-vector projection [512][D] + bias
    // conditioning staged by tts_set_conditioning / tts_train_set_conditioning into (ws, B); the next call on that workspace that
    // encodes consumes it, so a forgotten call can never reuse the previous batch's voices
    struct CondRecord { void* ws = nullptr; int B = 0; } cond_inf, cond_train;
    // ---- decode session: set up by tts_decode_begin, ended by the next tts_decode_begin or tts_finalize_weights
    struct DecodeSession {
        bool active = false; int B = 0, S = 0, T = 0, t = 0;          // T = max_len; t: frames decoded (upper bound until tts_decode_status)
        int t_status = -1, frontier = 0;                              // last tts_decode_status: frames decoded, frames final (-1: none yet)
        Ws L; ClusterParams cp;                                       // workspace layout of (B, S, T); decode kernel arguments
    } session;
    int* h_status = nullptr;                                          // pinned: t_done, n_finished
    TtsTrain* train = nullptr;                                        // training state (train.cuh), built by tts_train_begin
    int train_graph = 1;                                              // replay the train step from a CUDA graph (option "train_graph")
};

static bool conditioned(const TtsHandle* h) { return h->cfg.n_speakers > 0 || h->cfg.spk_embed_dim > 0; }
// the inference workspace layout of this handle (with the conditioning region iff the handle is conditioned)
static Ws ws_layout(const TtsHandle* h, int B, int S, int T) { return Ws::make(B, S, T, conditioned(h) ? h->cfg.spk_embed_dim : -1); }

#define CK(call)                                                                                     \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess) {                                                                     \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e_);                             \
            return (int)e_;                                                                          \
        }                                                                                            \
    } while (0)
#define FAIL(code, msg) do { h->err = (msg); return (code); } while (0)
// makes the handle's device current for the rest of the entry point and restores the caller's device on return
#define DEV_GUARD(h) DeviceGuard dev_guard_((h)->device); CK(dev_guard_.err)

static inline uint16_t f2bf(float f) {                                // round-to-nearest-even, as __float2bfloat16_rn
    uint32_t u; memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
    u += 0x7fffu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}

// ------------------------------------------------------------------------------------------------
extern "C" const char* tts_version(void) { return "tts_b200 0.1 sm_100a"; }

extern "C" unsigned long long tts_launch_count(void) { return launch_counter(); }

extern "C" const char* tts_last_error_string(TtsHandle* h) { return h ? h->err.c_str() : "null handle"; }

extern "C" int tts_create(const TtsConfig* cfg, int device, TtsHandle** out) {
    // the size before n_speakers (callers built against the unconditioned ABI) means an unconditioned model
    if (!cfg || !out || (cfg->struct_size != sizeof(TtsConfig) && cfg->struct_size != offsetof(TtsConfig, n_speakers))) return TTS_E_ARG;
    TtsConfig c;
    memset(&c, 0, sizeof(c));
    memcpy(&c, cfg, cfg->struct_size);
    c.struct_size = sizeof(TtsConfig);
    cfg = &c;
    if (cfg->n_speakers < 0 || cfg->n_speakers > kSpkMaxSpeakers || cfg->spk_embed_dim < 0 || cfg->spk_embed_dim > kSpkMaxDim) return TTS_E_ARG;
    if (cfg->d_model != 512 || cfg->n_heads != 8 || cfg->d_ff != 2048 || cfg->n_mels != 80 || cfg->d_prenet != 256 ||
        cfg->conv_kernel != 5 || cfg->n_enc_layers != 6 || cfg->n_dec_layers != 6 || cfg->enc_conv_layers != 3 ||
        cfg->postnet_layers != 5 || cfg->postnet_channels != 512 || cfg->max_pos < 1 || cfg->n_vocab < 1 ||
        !(cfg->ln_eps > 0.f) || !(cfg->bn_eps > 0.f))
        return TTS_E_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return TTS_E_DEVICE;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10) return TTS_E_DEVICE;
    TtsHandle* h = new TtsHandle();
    h->cfg = *cfg; h->device = device; h->num_sms = prop.multiProcessorCount;
    DeviceGuard dev_guard_(device);
    if (dev_guard_.err != cudaSuccess) { delete h; return TTS_E_DEVICE; }
    if (cudaMallocHost(&h->h_status, 64) != cudaSuccess) { delete h; return TTS_E_DEVICE; }
    *out = h;
    return 0;
}

extern "C" int tts_train_end(TtsHandle* h);
extern "C" int tts_destroy(TtsHandle* h) {
    if (!h) return TTS_E_ARG;
    DeviceGuard dev_guard_(h->device);
    if (h->arena) cudaFree(h->arena);
    if (h->pe) cudaFree(h->pe);
    if (h->cl_wpack) cudaFree(h->cl_wpack);
    if (h->h_status) cudaFreeHost(h->h_status);
    tts_train_end(h);
    delete h;
    return 0;
}

extern "C" int tts_set_option(TtsHandle* h, const char* key, int64_t value) {
    if (!h || !key) return TTS_E_ARG;
    if (!strcmp(key, "decode_timestamps")) { h->decode_timestamps = value ? 1 : 0; return 0; }
    if (!strcmp(key, "decode_debug")) { if (value < 0 || value > 8) FAIL(TTS_E_ARG, "decode_debug: 0 off, 1 + rank of the dumping CTA"); h->decode_debug = (int)value; return 0; }
    if (!strcmp(key, "cluster_group")) { if (value < 0 || value > CL_G) FAIL(TTS_E_ARG, "cluster_group must be 0 (auto) or 1..5"); h->cluster_group = (int)value; return 0; }
    if (!strcmp(key, "train_graph")) { h->train_graph = value ? 1 : 0; return 0; }
    if (!strcmp(key, "print_info")) { fprintf(stderr, "[tts_b200] sms=%d cluster_ok=%d max_clusters=%d group=%d ngroups=%d\n", h->num_sms, h->cluster_ok, h->max_clusters, h->session.cp.G, h->session.cp.ngroups); return 0; }
    FAIL(TTS_E_ARG, std::string("unknown option ") + key);
}

extern "C" int tts_load_weight(TtsHandle* h, const char* name, const float* host_data, int64_t numel) {
    if (!h || !name || !host_data || numel <= 0) return TTS_E_ARG;
    h->staged[name].assign(host_data, host_data + numel);
    h->finalized = false;
    return 0;
}

// ---- packing helpers ---------------------------------------------------------------------------
namespace {
struct Arena {
    std::vector<unsigned char> host;
    size_t take(size_t bytes) { size_t o = align_up(host.size()); host.resize(o + bytes, 0); return o; }
};

// row-major bf16 [taps][Nw][Kp] from fp32 W laid out as w[(n * K + k) * taps + tap] (conv) or [n][k] (taps = 1),
// scaled per output channel.
size_t pack_rowmajor(Arena& ar, const float* w, int N, int K, int taps, int Nw, int Kp, const float* scale) {
    size_t off = ar.take((size_t)taps * Nw * Kp * 2);
    uint16_t* dst = reinterpret_cast<uint16_t*>(ar.host.data() + off);
    for (int tap = 0; tap < taps; ++tap)
        for (int n = 0; n < N; ++n)
            for (int k = 0; k < K; ++k) {
                float v = w[((size_t)n * K + k) * taps + tap] * (scale ? scale[n] : 1.f);
                dst[((size_t)tap * Nw + n) * Kp + k] = f2bf(v);
            }
    return off;
}
size_t pack_f32(Arena& ar, const float* v, size_t n, size_t npad = 0) {
    size_t off = ar.take((npad > n ? npad : n) * 4);
    memcpy(ar.host.data() + off, v, n * 4);
    return off;
}
inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// One segment of a cluster rank's weight stream (decode_cluster.cuh: cl_gemm).  rows[] lists the global output row of every
// local column (NT tiles x 16; -1 = zero row).  Warp w owns tiles w*TW .. w*TW + TW-1 over the k-pairs (32 columns each)
// [kp_base, kp_base + KP); its run is [kp][j] blocks of 16(n) x 32(k) in mma.sync m16n8k16 A-fragment order (2 x 32 lanes x
// uint4 = 1 KB), the warps' runs follow each other -- exactly the order the consumer warps read them.
void pack_cluster_segment(std::vector<unsigned char>& out, const float* w, int N, int K, const std::vector<int>& rows,
                          int kp_base, int KP, int TW) {
    const int NT = (int)rows.size() / 16;
    auto at = [&](int row, int k) -> uint32_t { return (row >= 0 && row < N && k < K) ? f2bf(w[(size_t)row * K + k]) : 0; };
    for (int wi = 0; wi < NT / TW; ++wi)
        for (int kpl = 0; kpl < KP; ++kpl)
            for (int j = 0; j < TW; ++j) {
                const int tile = wi * TW + j, kp = kp_base + kpl;
                const size_t base = out.size();
                out.resize(base + 1024, 0);
                uint32_t* blk = reinterpret_cast<uint32_t*>(out.data() + base);
                for (int ks = 0; ks < 2; ++ks)
                    for (int lane = 0; lane < 32; ++lane) {
                        const int g = lane >> 2, t4 = lane & 3, k0 = kp * 32 + ks * 16 + t4 * 2;
                        const int r0 = rows[tile * 16 + g], r1 = rows[tile * 16 + g + 8];
                        uint32_t* q = blk + (ks * 32 + lane) * 4;
                        q[0] = at(r0, k0) | (at(r0, k0 + 1) << 16);
                        q[1] = at(r1, k0) | (at(r1, k0 + 1) << 16);
                        q[2] = at(r0, k0 + 8) | (at(r0, k0 + 9) << 16);
                        q[3] = at(r1, k0 + 8) | (at(r1, k0 + 9) << 16);
                    }
            }
}
std::vector<int> iota_rows(int lo, int n) { std::vector<int> r(n); for (int i = 0; i < n; ++i) r[i] = lo + i; return r; }
}  // namespace

extern "C" int tts_finalize_weights(TtsHandle* h) {
    if (!h) return TTS_E_ARG;
    DEV_GUARD(h);
    const TtsConfig& c = h->cfg;
    std::string missing;
    auto get = [&](const std::string& k, size_t numel) -> const float* {
        auto it = h->staged.find(k);
        if (it == h->staged.end() || it->second.size() != numel) { missing = k; return nullptr; }
        return it->second.data();
    };
#define GET(var, key, numel) const float* var = get(key, numel); if (!var) FAIL(TTS_E_WEIGHT, "missing or mis-sized weight: " + missing)
    Arena ar;
    struct Fix { void** dst; size_t off; };
    std::vector<Fix> fixes;
    auto bind = [&](auto** dst, size_t off) { fixes.push_back({reinterpret_cast<void**>(dst), off}); };
    const int D = 512, F = 2048;

    {   // embedding
        GET(w, "enc_prenet.embed.weight", (size_t)c.n_vocab * D);
        bind(&h->embed, pack_rowmajor(ar, w, c.n_vocab, D, 1, c.n_vocab, D, nullptr));
    }
    auto fold_conv = [&](const std::string& pre, int cin, int cout, int cin_pad, bf16** wd, float** bd) -> int {
        GET(w, pre + ".conv.weight", (size_t)cout * cin * 5);
        GET(b, pre + ".conv.bias", (size_t)cout);
        GET(g, pre + ".bn.weight", (size_t)cout);
        GET(be, pre + ".bn.bias", (size_t)cout);
        GET(rm, pre + ".bn.running_mean", (size_t)cout);
        GET(rv, pre + ".bn.running_var", (size_t)cout);
        std::vector<float> sc(cout), bias(cout);
        for (int o = 0; o < cout; ++o) {                              // P5: eval-mode BN folded into the conv
            sc[o] = g[o] / std::sqrt(rv[o] + c.bn_eps);
            bias[o] = (b[o] - rm[o]) * sc[o] + be[o];
        }
        bind(wd, pack_rowmajor(ar, w, cout, cin, 5, round_up(cout, 128), cin_pad, sc.data()));
        bind(bd, pack_f32(ar, bias.data(), cout));
        return 0;
    };
    for (int i = 0; i < 3; ++i) { int r = fold_conv("enc_prenet.convs." + std::to_string(i), D, D, D, &h->enc_conv_w[i], &h->enc_conv_b[i]); if (r) return r; }
    for (int i = 0; i < 5; ++i) {
        const int cin = i == 0 ? 80 : 512, cout = i == 4 ? 80 : 512;
        int r = fold_conv("postnet.convs." + std::to_string(i), cin, cout, i == 0 ? 96 : 512, &h->post_w[i], &h->post_b[i]); if (r) return r;
    }
    auto linear_rm = [&](const std::string& pre, int N, int K, int Kp, bf16** wd, float** bd) -> int {
        GET(w, pre + ".weight", (size_t)N * K); GET(b, pre + ".bias", (size_t)N);
        bind(wd, pack_rowmajor(ar, w, N, K, 1, round_up(N, 128), Kp, nullptr));
        bind(bd, pack_f32(ar, b, N, round_up(N, 128)));
        return 0;
    };
    auto vec = [&](const std::string& key, int n, float** dst) -> int { GET(v, key, (size_t)n); bind(dst, pack_f32(ar, v, n)); return 0; };
    auto cat3 = [&](const std::string& pre, std::vector<float>& w, std::vector<float>& b) -> int {
        w.clear(); b.clear();
        for (const char* nm : {"wq", "wk", "wv"}) {
            GET(ww, pre + "." + nm + ".weight", (size_t)D * D); GET(bb, pre + "." + nm + ".bias", (size_t)D);
            w.insert(w.end(), ww, ww + (size_t)D * D); b.insert(b.end(), bb, bb + D);
        }
        return 0;
    };
    int r;
    if ((r = linear_rm("enc_prenet.proj", D, D, D, &h->enc_proj_w, &h->enc_proj_b))) return r;
    { GET(a, "enc_alpha", 1); h->enc_alpha = a[0]; }
    { GET(a, "dec_alpha", 1); h->dec_alpha = a[0]; }
    std::vector<float> w3, b3;
    for (int l = 0; l < 6; ++l) {
        const std::string p = "encoder.layers." + std::to_string(l);
        auto& L = h->enc[l];
        if ((r = cat3(p + ".self_attn", w3, b3))) return r;
        bind(&L.wqkv, pack_rowmajor(ar, w3.data(), 3 * D, D, 1, 3 * D, D, nullptr)); bind(&L.bqkv, pack_f32(ar, b3.data(), 3 * D));
        if ((r = linear_rm(p + ".self_attn.wo", D, D, D, &L.wo, &L.bo))) return r;
        if ((r = linear_rm(p + ".ffn.w1", F, D, D, &L.w1, &L.b1))) return r;
        if ((r = linear_rm(p + ".ffn.w2", D, F, F, &L.w2, &L.b2))) return r;
        if ((r = vec(p + ".norm1.weight", D, &L.ln1g)) || (r = vec(p + ".norm1.bias", D, &L.ln1b)) ||
            (r = vec(p + ".norm2.weight", D, &L.ln2g)) || (r = vec(p + ".norm2.bias", D, &L.ln2b))) return r;
    }
    {   // hoisted cross-K/V projection of all 6 decoder layers as one [6*1024][512] weight
        std::vector<float> w((size_t)6 * 1024 * D), b(6 * 1024);
        for (int l = 0; l < 6; ++l) {
            const std::string p = "decoder.layers." + std::to_string(l) + ".cross_attn";
            GET(wk, p + ".wk.weight", (size_t)D * D); GET(wv, p + ".wv.weight", (size_t)D * D);
            GET(bk, p + ".wk.bias", (size_t)D); GET(bv, p + ".wv.bias", (size_t)D);
            memcpy(&w[(size_t)(l * 1024) * D], wk, (size_t)D * D * 4); memcpy(&w[(size_t)(l * 1024 + 512) * D], wv, (size_t)D * D * 4);
            memcpy(&b[l * 1024], bk, D * 4); memcpy(&b[l * 1024 + 512], bv, D * 4);
        }
        bind(&h->ckv_w, pack_rowmajor(ar, w.data(), 6 * 1024, D, 1, 6 * 1024, D, nullptr));
        bind(&h->ckv_b, pack_f32(ar, b.data(), 6 * 1024));
    }
    for (int l = 0; l < 6; ++l) {
        const std::string p = "decoder.layers." + std::to_string(l);
        auto& L = h->dec[l];
        if ((r = cat3(p + ".self_attn", w3, b3))) return r;
        bind(&L.wqkv, pack_rowmajor(ar, w3.data(), 3 * D, D, 1, 3 * D, D, nullptr)); bind(&L.bqkv, pack_f32(ar, b3.data(), 3 * D));
        if ((r = linear_rm(p + ".self_attn.wo", D, D, D, &L.wo, &L.bo))) return r;
        if ((r = linear_rm(p + ".cross_attn.wq", D, D, D, &L.wq2, &L.bq2))) return r;
        if ((r = linear_rm(p + ".cross_attn.wo", D, D, D, &L.wo2, &L.bo2))) return r;
        if ((r = linear_rm(p + ".ffn.w1", F, D, D, &L.w1, &L.b1))) return r;
        if ((r = linear_rm(p + ".ffn.w2", D, F, F, &L.w2, &L.b2))) return r;
        if ((r = vec(p + ".norm1.weight", D, &L.ln1g)) || (r = vec(p + ".norm1.bias", D, &L.ln1b)) ||
            (r = vec(p + ".norm2.weight", D, &L.ln2g)) || (r = vec(p + ".norm2.bias", D, &L.ln2b)) ||
            (r = vec(p + ".norm3.weight", D, &L.ln3g)) || (r = vec(p + ".norm3.bias", D, &L.ln3b))) return r;
    }
    if ((r = linear_rm("dec_prenet.fc1", 256, 80, 96, &h->pre_fc1, &h->pre_b1))) return r;
    if ((r = linear_rm("dec_prenet.fc2", 256, 256, 256, &h->pre_fc2, &h->pre_b2))) return r;
    if ((r = linear_rm("dec_prenet.proj", 512, 256, 256, &h->pre_proj, &h->pre_bp))) return r;
    {   // [mel | stop] heads fused into one 81-row matrix (C7)
        GET(wm, "mel_linear.weight", (size_t)80 * D); GET(bm, "mel_linear.bias", 80);
        GET(wsx, "stop_linear.weight", (size_t)D); GET(bs, "stop_linear.bias", 1);
        std::vector<float> w((size_t)81 * D), b(81);
        memcpy(w.data(), wm, (size_t)80 * D * 4); memcpy(&w[(size_t)80 * D], wsx, D * 4);
        memcpy(b.data(), bm, 80 * 4); b[80] = bs[0];
        bind(&h->head_w, pack_rowmajor(ar, w.data(), 81, D, 1, 128, D, nullptr));
        bind(&h->head_b, pack_f32(ar, b.data(), 81, 128));
    }
    h->spk_table = h->spk_w = h->spk_b = nullptr;                       // speaker conditioning, kept fp32 (speaker.cuh)
    if (c.n_speakers > 0) { GET(e, "speaker_embed.weight", (size_t)c.n_speakers * D); bind(&h->spk_table, pack_f32(ar, e, (size_t)c.n_speakers * D)); }
    if (c.spk_embed_dim > 0) {
        GET(w, "spk_proj.weight", (size_t)D * c.spk_embed_dim); GET(b, "spk_proj.bias", (size_t)D);
        bind(&h->spk_w, pack_f32(ar, w, (size_t)D * c.spk_embed_dim)); bind(&h->spk_b, pack_f32(ar, b, D));
    }
    if (!h->pe) {   // P4 sinusoid table, fp32 rounded from float64 (same definition as oracle.sinusoid_table).  Its own allocation,
                    // made once per handle: a captured training graph and a live decode session keep its address across re-finalisation
        std::vector<float> pe((size_t)c.max_pos * D);
        for (int pos = 0; pos < c.max_pos; ++pos)
            for (int i = 0; i < D; i += 2) {
                const double ang = (double)pos / std::pow(10000.0, (double)i / D);
                pe[(size_t)pos * D + i] = (float)std::sin(ang); pe[(size_t)pos * D + i + 1] = (float)std::cos(ang);
            }
        CK(cudaMalloc(&h->pe, pe.size() * 4));
        CK(cudaMemcpy(h->pe, pe.data(), pe.size() * 4, cudaMemcpyHostToDevice));
    }
    // ---- per-rank weight streams of the cluster decode kernel (decode_cluster.cuh), in consumption order
    std::vector<unsigned char> clw((size_t)CL_SIZE * CLW_RANK_BYTES);
    {
        GET(wf1, "dec_prenet.fc1.weight", (size_t)256 * 80); GET(wf2, "dec_prenet.fc2.weight", (size_t)256 * 256);
        GET(wpj, "dec_prenet.proj.weight", (size_t)512 * 256);
        GET(wm, "mel_linear.weight", (size_t)80 * D); GET(wsx, "stop_linear.weight", (size_t)D);
        std::vector<float> whead((size_t)81 * D);
        memcpy(whead.data(), wm, (size_t)80 * D * 4); memcpy(&whead[(size_t)80 * D], wsx, D * 4);
        for (int rk = 0; rk < CL_SIZE; ++rk) {
            std::vector<unsigned char> seg;
            seg.reserve(CLW_RANK_BYTES);
            pack_cluster_segment(seg, wf1, 256, 80, iota_rows(32 * rk, 32), 0, 4, 1);      // K 80 -> 128 (zeros)
            pack_cluster_segment(seg, wf2, 256, 256, iota_rows(32 * rk, 32), 0, 8, 1);
            pack_cluster_segment(seg, wpj, 512, 256, iota_rows(64 * rk, 64), 0, 8, 1);
            for (int l = 0; l < 6; ++l) {
                const std::string p = "decoder.layers." + std::to_string(l);
                if ((r = cat3(p + ".self_attn", w3, b3))) return r;
                GET(wo, p + ".self_attn.wo.weight", (size_t)D * D); GET(wq2, p + ".cross_attn.wq.weight", (size_t)D * D);
                GET(wo2, p + ".cross_attn.wo.weight", (size_t)D * D);
                GET(w1, p + ".ffn.w1.weight", (size_t)F * D); GET(w2, p + ".ffn.w2.weight", (size_t)D * F);
                std::vector<int> qrows(192);                      // q, k, v (64 dims each) of head rk
                for (int cc = 0; cc < 192; ++cc) qrows[cc] = (cc >> 6) * 512 + rk * 64 + (cc & 63);
                pack_cluster_segment(seg, w3.data(), 3 * D, D, qrows, 0, 8, 1);                // wide GEMMs: K in two halves, all warps'
                pack_cluster_segment(seg, w3.data(), 3 * D, D, qrows, 8, 8, 1);                // first halves first (cl_gemm<.., 2>)
                pack_cluster_segment(seg, wo, D, D, iota_rows(64 * rk, 64), 0, 16, 1);
                pack_cluster_segment(seg, wq2, D, D, iota_rows(64 * rk, 64), 0, 16, 1);
                pack_cluster_segment(seg, wo2, D, D, iota_rows(64 * rk, 64), 0, 16, 1);
                pack_cluster_segment(seg, w1, F, D, iota_rows(256 * rk, 256), 0, 8, 1);
                pack_cluster_segment(seg, w1, F, D, iota_rows(256 * rk, 256), 8, 8, 1);
                pack_cluster_segment(seg, w2, D, F, iota_rows(0, 512), 8 * rk, 4, 2);          // K-slice [256 rk, 256 rk + 256), two tiles per warp
                pack_cluster_segment(seg, w2, D, F, iota_rows(0, 512), 8 * rk + 4, 4, 2);
            }
            std::vector<int> hrows(16);
            for (int i = 0; i < 16; ++i) hrows[i] = (rk < 6 && 16 * rk + i < 81) ? 16 * rk + i : -1;
            pack_cluster_segment(seg, whead.data(), 81, D, hrows, 0, 16, 1);
            if (seg.size() != CLW_RANK_BYTES) FAIL(TTS_E_STATE, "cluster weight stream size mismatch");
            memcpy(clw.data() + (size_t)rk * CLW_RANK_BYTES, seg.data(), CLW_RANK_BYTES);
        }
    }
#undef GET
    if (h->cl_wpack) { cudaFree(h->cl_wpack); h->cl_wpack = nullptr; }
    CK(cudaMalloc(&h->cl_wpack, clw.size()));
    CK(cudaMemcpy(h->cl_wpack, clw.data(), clw.size(), cudaMemcpyHostToDevice));
    if (h->arena) { cudaFree(h->arena); h->arena = nullptr; }
    h->arena_bytes = align_up(ar.host.size());
    CK(cudaMalloc(&h->arena, h->arena_bytes));
    CK(cudaMemcpy(h->arena, ar.host.data(), ar.host.size(), cudaMemcpyHostToDevice));
    for (auto& f : fixes) *f.dst = h->arena + f.off;
    CK(cudaDeviceSynchronize());
    h->session.active = false;                                        // a decode session holds pointers into the old arena
    h->finalized = true;                                              // (the staged fp32 copies stay: tts_train_begin builds the master from them)
    return 0;
}

extern "C" size_t tts_workspace_bytes(TtsHandle* h, int B, int S, int T) {
    if (!h || B <= 0 || S <= 0 || T <= 0) return 0;
    return ws_layout(h, B, S, T).total;
}

// ------------------------------------------------------------------------------------------------
// sequence-parallel building blocks
namespace {
GemmParams gp(const bf16* A, int lda, const bf16* W, int ldw, int M, int N, int K) {
    GemmParams p; memset(&p, 0, sizeof(p));
    p.A = A; p.lda = lda; p.W = W; p.ldw = ldw; p.M = M; p.N = N; p.K = K; p.taps = 1; p.Nw = round_up(N, 128);
    p.T = M; p.drop_site = -1; p.dropw_site = -1; p.B = 1;
    return p;
}
AttnParams ap_packed(const bf16* Q, int ldq, const bf16* K, int ldk, const bf16* V, int ldv, bf16* O, int ldo,
                     int B, int Lq, int Lk, const int* klens, int causal) {
    AttnParams a; memset(&a, 0, sizeof(a));
    a.Q = Q; a.K = K; a.V = V; a.O = O;
    a.q_bs = (long)Lq * ldq; a.q_hs = 64; a.q_rs = ldq;
    a.k_bs = (long)Lk * ldk; a.k_hs = 64; a.k_rs = ldk;
    a.v_bs = (long)Lk * ldv; a.v_hs = 64; a.v_rs = ldv;
    a.o_bs = (long)Lq * ldo; a.o_hs = 64; a.o_rs = ldo;
    a.B = B; a.H = kHeads; a.Lq = Lq; a.Lk = Lk; a.klens = klens; a.causal = causal;
    a.scale_log2 = 0.125f * kLog2e;
    return a;
}
cudaError_t layernorm(const float* x, const float* g, const float* b, bf16* o16, float* o32, int M, float eps, cudaStream_t st) {
    layernorm512_kernel<false><<<(M + 7) / 8, 256, 0, st>>>(x, g, b, o16, o32, M, eps, nullptr, 0);
    ++launch_counter();
    return cudaGetLastError();
}
}  // namespace

// Encoder (C1-C4) + hoisted cross-K/V projection.  Result: memory in ws.x (bf16 [B*S][512]).  A conditioned layout adds the speaker
// vector of every utterance (speaker.cuh, from the inputs staged by tts_set_conditioning) inside the last LayerNorm.
static int run_encoder(TtsHandle* h, void* ws, const Ws& L, const int64_t* ph, const int* plens, int B, int S, bool v_blocked, cudaStream_t st) {
    const int M = B * S;
    bf16 *x = wsp<bf16>(ws, L.x), *x2 = wsp<bf16>(ws, L.x2), *wide = wsp<bf16>(ws, L.wide), *a = wsp<bf16>(ws, L.a);
    float* y = wsp<float>(ws, L.y);
    if (L.has_cond)
        CK(launch_speaker_cond(wsp<int>(ws, L.sids), wsp<float>(ws, L.spembs), B, h->cfg.n_speakers, h->cfg.spk_embed_dim, h->spk_table, h->spk_w,
                               h->spk_b, wsp<float>(ws, L.cond), wsp<float>(ws, L.nhat), st));
    embed_kernel<<<(M + 3) / 4, 256, 0, st>>>(ph, plens, h->embed, x, B, S, h->cfg.n_vocab);
    ++launch_counter();
    CK(cudaGetLastError());
    for (int i = 0; i < 3; ++i) {                                      // conv k5 + folded BN + ReLU + length mask
        GemmParams p = gp(x, 512, h->enc_conv_w[i], 512, M, 512, 512);
        p.taps = 5; p.T = S; p.bias = h->enc_conv_b[i]; p.act = ACT_RELU; p.lens = plens; p.out_bf16 = x2; p.ldo = 512;
        CK(launch_gemm_tc(p, st));
        std::swap(x, x2);
    }
    {   // linear + alpha * PE
        GemmParams p = gp(x, 512, h->enc_proj_w, 512, M, 512, 512);
        p.T = S; p.bias = h->enc_proj_b; p.pe = h->pe; p.alpha = h->enc_alpha; p.out_bf16 = x2; p.ldo = 512;
        CK(launch_gemm_tc(p, st));
        std::swap(x, x2);
    }
    for (int l = 0; l < 6; ++l) {
        auto& W = h->enc[l];
        GemmParams p = gp(x, 512, W.wqkv, 512, M, 1536, 512); p.bias = W.bqkv; p.out_bf16 = wide; p.ldo = 1536;
        CK(launch_gemm_tc(p, st));
        AttnParams at = ap_packed(wide, 1536, wide + 512, 1536, wide + 1024, 1536, a, 512, B, S, S, plens, 0);
        CK(launch_flash_attn_tc(at, st));
        p = gp(a, 512, W.wo, 512, M, 512, 512); p.bias = W.bo; p.resid_bf16 = x; p.ldr = 512; p.out_f32 = y; p.ldo = 512;
        CK(launch_gemm_tc(p, st));
        CK(layernorm(y, W.ln1g, W.ln1b, x, nullptr, M, h->cfg.ln_eps, st));
        p = gp(x, 512, W.w1, 512, M, 2048, 512); p.bias = W.b1; p.act = ACT_RELU; p.out_bf16 = wide; p.ldo = 2048;
        CK(launch_gemm_tc(p, st));
        p = gp(wide, 2048, W.w2, 2048, M, 512, 2048); p.bias = W.b2; p.resid_bf16 = x; p.ldr = 512; p.out_f32 = y; p.ldo = 512;
        CK(launch_gemm_tc(p, st));
        if (l == 5 && L.has_cond) CK(launch_layernorm_cond(y, W.ln2g, W.ln2b, x, nullptr, M, h->cfg.ln_eps, wsp<float>(ws, L.cond), S, st));
        else CK(layernorm(y, W.ln2g, W.ln2b, x, nullptr, M, h->cfg.ln_eps, st));
    }
    if (x != wsp<bf16>(ws, L.x)) {                                     // keep memory in ws.x
        CK(cudaMemcpyAsync(wsp<bf16>(ws, L.x), x, (size_t)M * 512 * 2, cudaMemcpyDeviceToDevice, st));
    }
    {   // cross K/V of all decoder layers -> cache [6][2][B][H][S][64]
        GemmParams p = gp(wsp<bf16>(ws, L.x), 512, h->ckv_w, 512, M, 6 * 1024, 512);
        // rows past S of every (layer, b, h) stay zero: the decode kernel copies the cache at 16-row granularity
        CK(cudaMemsetAsync(wsp<bf16>(ws, L.cross_kv), 0, L.cross_kv_bytes, st));
        p.T = S; p.B = B; p.Lpad = v_blocked ? L.nblk_cross * KV_BLOCK_ROWS : L.Spad; p.bias = h->ckv_b; p.scatter = v_blocked ? SC_CROSS_KV_VT : SC_CROSS_KV; p.out_bf16 = wsp<bf16>(ws, L.cross_kv);
        CK(launch_gemm_tc(p, st));
    }
    return 0;
}

// Postnet (C8) over compact rows: in16 bf16 [B*T][96] masked, resid32 fp32 [B*T][80] masked -> mel_after [B*T][80]; x / x2 are
// bf16 [B*T][512] activations.  max_ctas caps the persistent GEMM grid (0: one CTA per SM).
static int run_postnet_rows(TtsHandle* h, const bf16* in16, const float* resid32, bf16* x, bf16* x2, const int* mlens, int B, int T,
                            float* mel_after, int max_ctas, cudaStream_t st) {
    const int M = B * T;
    const bf16* in = in16;
    for (int i = 0; i < 5; ++i) {
        const int K = i == 0 ? 96 : 512, N = i == 4 ? 80 : 512;
        GemmParams p = gp(in, K, h->post_w[i], K, M, N, K);
        p.taps = 5; p.T = T; p.bias = h->post_b[i]; p.lens = mlens; p.max_ctas = max_ctas;
        if (i < 4) { p.act = ACT_TANH; p.out_bf16 = x; p.ldo = 512; }
        else { p.resid_f32 = resid32; p.ldr = 80; p.out_f32 = mel_after; p.ldo = 80; }
        CK(launch_gemm_tc(p, st));
        in = x; std::swap(x, x2);
    }
    return 0;
}
static int run_postnet(TtsHandle* h, void* ws, const Ws& L, const int* mlens, int B, int T, float* mel_after, cudaStream_t st) {
    return run_postnet_rows(h, wsp<bf16>(ws, L.mel16), wsp<float>(ws, L.mel32), wsp<bf16>(ws, L.x2), wsp<bf16>(ws, L.a), mlens, B, T,
                            mel_after, 0, st);
}

// ------------------------------------------------------------------------------------------------
// Consumes the conditioning record of a conditioned handle: it must name this workspace and batch size.
static int take_conditioning(TtsHandle* h, TtsHandle::CondRecord& rec, void* ws, int B, const char* setter) {
    if (!conditioned(h)) return 0;
    if (rec.ws != ws || rec.B != B) FAIL(TTS_E_STATE, std::string("speaker-conditioned model: ") + setter + " must stage this batch's speakers first");
    rec = TtsHandle::CondRecord();
    return 0;
}
// Copies sids int32 [B] / spembs fp32 [B][spk_embed_dim] (device) into the conditioning region at the start of ws.
static int stage_conditioning(TtsHandle* h, void* ws, int B, const int32_t* sids, const float* spembs, size_t sids_off, size_t spembs_off,
                              cudaStream_t st) {
    if (!ws || B <= 0) return TTS_E_ARG;
    if (!conditioned(h)) FAIL(TTS_E_STATE, "the model has no speaker conditioning (n_speakers = spk_embed_dim = 0)");
    if (!sids != !(h->cfg.n_speakers > 0)) FAIL(TTS_E_ARG, "sids must be given exactly when n_speakers > 0");
    if (!spembs != !(h->cfg.spk_embed_dim > 0)) FAIL(TTS_E_ARG, "spembs must be given exactly when spk_embed_dim > 0");
    if (sids) CK(cudaMemcpyAsync(wsp<int>(ws, sids_off), sids, (size_t)B * 4, cudaMemcpyDeviceToDevice, st));
    if (spembs) CK(cudaMemcpyAsync(wsp<float>(ws, spembs_off), spembs, (size_t)B * h->cfg.spk_embed_dim * 4, cudaMemcpyDeviceToDevice, st));
    return 0;
}

extern "C" int tts_set_conditioning(TtsHandle* h, void* ws, int B, const int32_t* sids, const float* spembs, void* stream) {
    if (!h) return TTS_E_ARG;
    DEV_GUARD(h);
    const Ws L = Ws::make(B, 1, 1, h->cfg.spk_embed_dim);            // the region's offsets depend on B only
    int r = stage_conditioning(h, ws, B, sids, spembs, L.sids, L.spembs, (cudaStream_t)stream);
    if (r) return r;
    h->cond_inf = {ws, B};
    return 0;
}

extern "C" int tts_encode(TtsHandle* h, void* ws, const int64_t* phonemes, const int32_t* phoneme_lens, int B, int S, int T,
                          float* memory_out, void* stream) {
    if (!h || !ws || !phonemes || !phoneme_lens || B <= 0 || S <= 0 || T <= 0) return TTS_E_ARG;
    if (!h->finalized) FAIL(TTS_E_STATE, "weights not finalised");
    if (S > h->cfg.max_pos) FAIL(TTS_E_ARG, "S exceeds max_pos");
    DEV_GUARD(h);
    if (int r = take_conditioning(h, h->cond_inf, ws, B, "tts_set_conditioning")) return r;
    cudaStream_t st = (cudaStream_t)stream;
    const Ws L = ws_layout(h, B, S, T);
    // the decode phases read the key-padding lengths from the workspace copy
    CK(cudaMemcpyAsync(wsp<int>(ws, L.plens), phoneme_lens, (size_t)B * 4, cudaMemcpyDeviceToDevice, st));
    int r = run_encoder(h, ws, L, phonemes, wsp<int>(ws, L.plens), B, S, true, st);
    if (r) return r;
    if (memory_out) {
        size_t n = (size_t)B * S * 512;
        bf16_to_f32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(wsp<bf16>(ws, L.x), memory_out, n);
        ++launch_counter();
        CK(cudaGetLastError());
    }
    return 0;
}

extern "C" int tts_decode_begin(TtsHandle* h, void* ws, int B, int S, int max_len, uint64_t seed, int utt_offset, void* stream) {
    if (!h || !ws || B <= 0 || S <= 0 || max_len <= 0) return TTS_E_ARG;
    if (!h->finalized) FAIL(TTS_E_STATE, "weights not finalised");
    if (max_len > h->cfg.max_pos) FAIL(TTS_E_ARG, "max_len exceeds max_pos");
    DEV_GUARD(h);
    cudaStream_t st = (cudaStream_t)stream;
    auto& ds = h->session;
    ds.active = true; ds.B = B; ds.S = S; ds.T = max_len; ds.t = 0; ds.t_status = -1; ds.frontier = 0;
    ds.L = ws_layout(h, B, S, max_len);
    const Ws& L = ds.L;
    init_decode_state_kernel<<<(std::max(B, 4) + 255) / 256, 256, 0, st>>>(wsp<int>(ws, L.lens), wsp<int>(ws, L.finished),
                                                                          wsp<int>(ws, L.scalars), B, max_len);
    ++launch_counter();
    CK(cudaGetLastError());
    // cache rows are copied at 16-row granularity: rows not yet written must be finite, so the self cache starts zeroed
    CK(cudaMemsetAsync(wsp<bf16>(ws, L.self_kv), 0, L.self_kv_bytes, st));

    if (h->cluster_ok < 0) {                                            // how many 8-CTA clusters of this kernel can be co-resident?
        h->cluster_ok = 0;
        if (cudaFuncSetAttribute(decode_cluster_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, CL_SMEM_BYTES) == cudaSuccess &&
            cudaFuncSetAttribute(decode_cluster_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, CL_SMEM_BYTES) == cudaSuccess) {
            cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof(cfg));
            cfg.gridDim = dim3(CL_SIZE * 8); cfg.blockDim = dim3(CL_THREADS); cfg.dynamicSmemBytes = CL_SMEM_BYTES;
            cudaLaunchAttribute at[1]; at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = CL_SIZE; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            cfg.attrs = at; cfg.numAttrs = 1;
            int n = 0;
            if (cudaOccupancyMaxActiveClusters(&n, decode_cluster_kernel<true>, &cfg) == cudaSuccess && n > 0) { h->cluster_ok = 1; h->max_clusters = n; }
        }
        cudaGetLastError();
    }
    if (h->cluster_ok != 1) FAIL(TTS_E_DEVICE, "device cannot co-schedule an 8-CTA cluster of the decode kernel");

    ClusterParams& cp = ds.cp; memset(&cp, 0, sizeof(cp));
    cp.B = B; cp.Tmax = max_len; cp.S = S; cp.nblk_self = L.nblk_self; cp.nblk_cross = L.nblk_cross;
    // utterances per cluster: as few as the co-resident cluster count allows (more SMs stream K/V), at most 8
    cp.G = h->cluster_group > 0 ? std::min(CL_G, h->cluster_group)
                                : std::min(CL_G, std::max(1, (B + h->max_clusters - 1) / h->max_clusters));
    cp.ngroups = (B + cp.G - 1) / cp.G;
    cp.seed = seed; cp.utt_offset = utt_offset; cp.dec_alpha = h->dec_alpha; cp.ln_eps = h->cfg.ln_eps; cp.pe = h->pe;
    cp.wpack = h->cl_wpack; cp.b_fc1 = h->pre_b1; cp.b_fc2 = h->pre_b2; cp.b_proj = h->pre_bp; cp.b_head = h->head_b;
    for (int l = 0; l < 6; ++l) {
        auto& W = h->dec[l];
        cp.layer[l] = ClusterLayerParams{W.bqkv, W.bo, W.bq2, W.bo2, W.b1, W.b2, W.ln1g, W.ln1b, W.ln2g, W.ln2b, W.ln3g, W.ln3b};
    }
    cp.self_kv = wsp<bf16>(ws, L.self_kv); cp.cross_kv = wsp<bf16>(ws, L.cross_kv); cp.plens = wsp<int>(ws, L.plens);
    cp.mel_before = wsp<float>(ws, L.mel_before); cp.stop_logits = wsp<float>(ws, L.stop_logits);
    cp.lens = wsp<int>(ws, L.lens); cp.finished = wsp<int>(ws, L.finished); cp.n_finished = wsp<int>(ws, L.scalars);
    return 0;
}

extern "C" int tts_decode_steps(TtsHandle* h, void* ws, int n_steps, void* stream) {
    if (!h || !ws || n_steps < 0) return TTS_E_ARG;
    auto& ds = h->session;
    if (!ds.active) FAIL(TTS_E_STATE, "tts_decode_begin not called");
    DEV_GUARD(h);
    cudaStream_t st = (cudaStream_t)stream;
    n_steps = std::min(n_steps, ds.T - ds.t);
    if (n_steps <= 0) return 0;
    ClusterParams& cp = ds.cp;
    cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof(cfg));
    const int ncl = std::min(cp.ngroups, h->max_clusters);
    cfg.gridDim = dim3(CL_SIZE * ncl); cfg.blockDim = dim3(CL_THREADS); cfg.dynamicSmemBytes = CL_SMEM_BYTES; cfg.stream = st;
    cudaLaunchAttribute at[1]; at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = CL_SIZE; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    cp.ts = h->decode_timestamps ? wsp<unsigned long long>(ws, ds.L.ts) : nullptr;
    if (cp.group_queue) CK(cudaMemsetAsync(cp.group_queue, 0, 4, st));  // work stealing: every launch starts from a fresh queue
    // (the debug dump lands in the `wide` activation buffer, idle during the decode loop: >= B * 2048 * 2 bytes per row of S/T)
    cp.dbg_rank = h->decode_debug - 1;
    cp.dbg = h->decode_debug ? wsp<float>(ws, ds.L.wide) : nullptr;
    if (cp.ts || cp.dbg) CK(cudaLaunchKernelEx(&cfg, decode_cluster_kernel<true>, cp, ds.t, n_steps));
    else CK(cudaLaunchKernelEx(&cfg, decode_cluster_kernel<false>, cp, ds.t, n_steps));
    ++launch_counter();
    ds.t += n_steps;                                                    // upper bound; tts_decode_status refines it
    return 0;
}

// Frames on each side of a frame that the postnet's output at that frame depends on: layers x (kernel / 2).
static int postnet_halo(const TtsHandle* h) { return h->cfg.postnet_layers * (h->cfg.conv_kernel / 2); }

extern "C" int tts_decode_status(TtsHandle* h, void* ws, int* t_done, int* n_finished, void* stream) {
    if (!h || !ws) return TTS_E_ARG;
    auto& ds = h->session;
    if (!ds.active) FAIL(TTS_E_STATE, "tts_decode_begin not called");
    DEV_GUARD(h);
    cudaStream_t st = (cudaStream_t)stream;
    CK(cudaMemcpyAsync(h->h_status, ds.cp.n_finished, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const int nf = h->h_status[0];
    if (nf >= ds.B) {                                     // every utterance fired: the frames run = the longest utterance
        std::vector<int> lens(ds.B);
        CK(cudaMemcpyAsync(lens.data(), ds.cp.lens, (size_t)ds.B * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        int mx = 0; for (int v : lens) mx = std::max(mx, v);
        ds.t = mx;
    }
    // tts_decode_emit's frontier: a frame's postnet output is final once the postnet's halo past it is decoded, or once the session
    // has ended (every utterance stopped, or max_len reached).  Only this call moves it; tts_decode_steps does not.
    const bool ended = nf >= ds.B || ds.t >= ds.T;
    ds.t_status = ds.t;
    ds.frontier = ended ? ds.t : std::max(0, ds.t - postnet_halo(h));
    if (n_finished) *n_finished = nf;
    if (t_done) *t_done = ds.t;
    return 0;
}

extern "C" int tts_decode_set_batch(TtsHandle* h, void* ws, const int32_t* utt_ids, const int32_t* max_lens, int work_stealing, void* stream) {
    if (!h || !ws) return TTS_E_ARG;
    auto& ds = h->session;
    if (!ds.active || ds.t != 0) FAIL(TTS_E_STATE, "tts_decode_set_batch belongs between tts_decode_begin and the first tts_decode_steps");
    DEV_GUARD(h);
    cudaStream_t st = (cudaStream_t)stream;
    int* ids = utt_ids ? wsp<int>(ws, ds.L.utt_ids) : nullptr;
    int* tlens = max_lens ? wsp<int>(ws, ds.L.tlens) : nullptr;
    if (ids) CK(cudaMemcpyAsync(ids, utt_ids, (size_t)ds.B * 4, cudaMemcpyDeviceToDevice, st));
    if (tlens) CK(cudaMemcpyAsync(tlens, max_lens, (size_t)ds.B * 4, cudaMemcpyDeviceToDevice, st));
    ds.cp.utt_ids = ids; ds.cp.tlens = tlens;
    ds.cp.group_queue = work_stealing ? wsp<int>(ws, ds.L.scalars) + 1 : nullptr;
    return 0;
}

extern "C" int tts_decode_set_frame(TtsHandle* h, void* ws, int t, const float* frames, void* stream) {
    if (!h || !ws || !frames) return TTS_E_ARG;
    const auto& ds = h->session;
    if (!ds.active) FAIL(TTS_E_STATE, "tts_decode_begin not called");
    if (t < 0 || t >= ds.t) FAIL(TTS_E_ARG, "frame index must lie in [0, frames decoded so far)");
    DEV_GUARD(h);
    CK(cudaMemcpy2DAsync(wsp<float>(ws, ds.L.mel_before) + (size_t)t * 80, (size_t)ds.T * 80 * 4, frames, 80 * 4, 80 * 4, (size_t)ds.B,
                         cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return 0;
}

extern "C" int tts_decode_get_frame(TtsHandle* h, void* ws, int t, float* frames, float* stop_logits, void* stream) {
    if (!h || !ws || !frames) return TTS_E_ARG;
    const auto& ds = h->session;
    if (!ds.active) FAIL(TTS_E_STATE, "tts_decode_begin not called");
    if (t < 0 || t >= ds.t) FAIL(TTS_E_ARG, "frame index must lie in [0, frames decoded so far)");
    DEV_GUARD(h);
    CK(cudaMemcpy2DAsync(frames, 80 * 4, wsp<float>(ws, ds.L.mel_before) + (size_t)t * 80, (size_t)ds.T * 80 * 4, 80 * 4, (size_t)ds.B,
                         cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    if (stop_logits)
        CK(cudaMemcpy2DAsync(stop_logits, 4, wsp<float>(ws, ds.L.stop_logits) + t, (size_t)ds.T * 4, 4, (size_t)ds.B, cudaMemcpyDeviceToDevice,
                             (cudaStream_t)stream));
    return 0;
}

extern "C" int tts_decode_end(TtsHandle* h, void* ws, int T_out, float* mel_after, int32_t* mel_lens, float* stop_logits,
                              float* mel_before, void* stream) {
    if (!h || !ws || !mel_after || T_out <= 0) return TTS_E_ARG;
    const auto& ds = h->session;
    if (!ds.active) FAIL(TTS_E_STATE, "tts_decode_begin not called");
    if (T_out > ds.T) FAIL(TTS_E_ARG, "T_out exceeds max_len");
    DEV_GUARD(h);
    cudaStream_t st = (cudaStream_t)stream;
    const int B = ds.B;
    const Ws& L = ds.L;
    const int* lens = wsp<int>(ws, L.lens);
    const int n = B * T_out * 24;
    mel_to_bf16_kernel<<<(n + 255) / 256, 256, 0, st>>>(wsp<float>(ws, L.mel_before), ds.T, lens, 0,
                                                        wsp<bf16>(ws, L.mel16), wsp<float>(ws, L.mel32), B, T_out);
    ++launch_counter();
    CK(cudaGetLastError());
    if (stop_logits || mel_lens) {
        float* so = stop_logits ? stop_logits : wsp<float>(ws, L.y);
        finalize_stop_kernel<<<(std::max(B * T_out, B) + 255) / 256, 256, 0, st>>>(wsp<float>(ws, L.stop_logits), ds.T, lens, so, mel_lens, B, T_out);
        ++launch_counter();
        CK(cudaGetLastError());
    }
    if (mel_before) CK(cudaMemcpyAsync(mel_before, wsp<float>(ws, L.mel32), (size_t)B * T_out * 80 * 4, cudaMemcpyDeviceToDevice, st));
    return run_postnet(h, ws, L, lens, B, T_out, mel_after, st);
}

// ------------------------------------------------------------------------------------------------
// Streaming: the postnet over a window of frames of a running decode session.  Scratch: postnet input bf16 [B][W][96] | residual
// fp32 [B][W][80] | two bf16 activations [B][W][512] | output fp32 [B][W][80] | window lengths int32 [B].
namespace {
struct StreamScratch {
    size_t in16, res32, xa, xb, out32, wlens, total;
    static StreamScratch make(int B, int W) {
        StreamScratch s; size_t o = 0;
        auto take = [&](size_t bytes) { size_t r = o; o = align_up(o + bytes); return r; };
        const size_t rows = (size_t)B * W;
        s.in16 = take(rows * 96 * 2); s.res32 = take(rows * 80 * 4); s.xa = take(rows * 512 * 2); s.xb = take(rows * 512 * 2);
        s.out32 = take(rows * 80 * 4); s.wlens = take((size_t)B * 4);
        s.total = o;
        return s;
    }
};
}  // namespace

extern "C" size_t tts_stream_scratch_bytes(TtsHandle* h, int B, int max_frames) {
    if (!h || B <= 0 || max_frames <= 0) return 0;
    return StreamScratch::make(B, max_frames + 2 * postnet_halo(h)).total;
}

extern "C" int tts_decode_emit(TtsHandle* h, void* ws, void* scratch, size_t scratch_bytes, int t_begin, int t_end, float* mel_after,
                               float* stop_logits, int32_t* mel_lens, float* mel_before, void* stream) {
    if (!h || !ws || !scratch || !mel_after || !stop_logits) return TTS_E_ARG;
    const auto& ds = h->session;
    if (!ds.active) FAIL(TTS_E_STATE, "tts_decode_begin not called");
    if (ds.t_status < 0) FAIL(TTS_E_STATE, "tts_decode_emit needs a tts_decode_status call first");
    if (t_begin < 0 || t_end <= t_begin) FAIL(TTS_E_ARG, "frame range must be non-empty and start at >= 0");
    if (t_end > ds.frontier) FAIL(TTS_E_ARG, "t_end lies past the frontier of the last tts_decode_status");
    const int halo = postnet_halo(h), B = ds.B, n = t_end - t_begin;
    const int a = std::max(0, t_begin - halo), e = std::min(t_end + halo, ds.t_status), W = e - a;
    const StreamScratch S = StreamScratch::make(B, W);
    if (S.total > scratch_bytes) FAIL(TTS_E_ARG, "scratch too small for this window (tts_stream_scratch_bytes)");
    // the decode kernel holds CL_SIZE SMs per co-resident cluster while it runs; the postnet GEMMs take only the others
    const int max_ctas = h->num_sms - CL_SIZE * std::min(ds.cp.ngroups, h->max_clusters);
    if (max_ctas < 1) FAIL(TTS_E_DEVICE, "no SM left beside the decode kernel");
    DEV_GUARD(h);
    cudaStream_t st = (cudaStream_t)stream;
    const Ws& L = ds.L;
    const int nthreads = std::max(B * W * 24, B * n);
    stream_window_kernel<<<(nthreads + 255) / 256, 256, 0, st>>>(wsp<float>(ws, L.mel_before), wsp<float>(ws, L.stop_logits), ds.T,
                                                                 wsp<int>(ws, L.lens), ds.t_status, a, W, t_begin, n,
                                                                 wsp<bf16>(scratch, S.in16), wsp<float>(scratch, S.res32),
                                                                 wsp<int>(scratch, S.wlens), stop_logits, mel_lens, B);
    ++launch_counter();
    CK(cudaGetLastError());
    // Rows within `halo` of a window edge that is not a true edge (t = 0 or the session's end) see zeros where the whole-utterance
    // postnet sees frames: they are computed and dropped.  Rows [t_begin, t_end) see exactly what that postnet sees.
    int r = run_postnet_rows(h, wsp<bf16>(scratch, S.in16), wsp<float>(scratch, S.res32), wsp<bf16>(scratch, S.xa), wsp<bf16>(scratch, S.xb),
                             wsp<int>(scratch, S.wlens), B, W, wsp<float>(scratch, S.out32), max_ctas, st);
    if (r) return r;
    const size_t row_bytes = (size_t)n * 80 * 4, pitch = (size_t)W * 80 * 4, off = (size_t)(t_begin - a) * 80;
    CK(cudaMemcpy2DAsync(mel_after, row_bytes, wsp<float>(scratch, S.out32) + off, pitch, row_bytes, (size_t)B, cudaMemcpyDeviceToDevice, st));
    if (mel_before)
        CK(cudaMemcpy2DAsync(mel_before, row_bytes, wsp<float>(scratch, S.res32) + off, pitch, row_bytes, (size_t)B, cudaMemcpyDeviceToDevice, st));
    return 0;
}

extern "C" int tts_infer_host(TtsHandle* h, void* ws, const int64_t* phonemes, const int32_t* phoneme_lens, int B, int S,
                              int max_len, uint64_t seed, int utt_offset, float* mel_after, int32_t* mel_lens,
                              float* stop_logits, int* T_out, void* stream) {
    if (!h || !ws || !phonemes || !phoneme_lens || !mel_after || !mel_lens || !stop_logits || !T_out) return TTS_E_ARG;
    if (B <= 0 || S <= 0 || max_len <= 0) FAIL(TTS_E_ARG, "B, S and max_len must be positive");
    if (!h->finalized) FAIL(TTS_E_STATE, "weights not finalised");
    if (S > h->cfg.max_pos) FAIL(TTS_E_ARG, "S exceeds max_pos");              // checked before any copy or launch
    if (max_len > h->cfg.max_pos) FAIL(TTS_E_ARG, "max_len exceeds max_pos");
    if (conditioned(h)) FAIL(TTS_E_STATE, "speaker-conditioned model: use the device path (tts_set_conditioning, tts_encode, tts_decode_*)");
    DEV_GUARD(h);
    cudaStream_t st = (cudaStream_t)stream;
    const Ws L = Ws::make(B, S, max_len);
    CK(cudaMemcpyAsync(wsp<int64_t>(ws, L.ph), phonemes, (size_t)B * S * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(wsp<int>(ws, L.plens), phoneme_lens, (size_t)B * 4, cudaMemcpyHostToDevice, st));
    int r = tts_decode_begin(h, ws, B, S, max_len, seed, utt_offset, stream);   // fixes the layout (T = max_len) first
    if (r) return r;
    if ((r = run_encoder(h, ws, L, wsp<int64_t>(ws, L.ph), wsp<int>(ws, L.plens), B, S, true, st))) return r;
    int td = 0, nf = 0;
    if ((r = tts_decode_steps(h, ws, max_len, stream))) return r;           // every cluster stops on the device once its utterances fired
    if ((r = tts_decode_status(h, ws, &td, &nf, stream))) return r;
    // outputs staged in the (now free) sequence buffers, then copied to the host
    float* d_after = wsp<float>(ws, L.y);
    float* d_stop = reinterpret_cast<float*>(wsp<bf16>(ws, L.wide));
    int* d_lens = wsp<int>(ws, L.mlens);
    if ((r = tts_decode_end(h, ws, td, d_after, d_lens, d_stop, nullptr, stream))) return r;
    CK(cudaMemcpyAsync(mel_after, d_after, (size_t)B * td * 80 * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(stop_logits, d_stop, (size_t)B * td * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(mel_lens, d_lens, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    *T_out = td;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Where the teacher-forced forward sends the cross-attention of the decoder layers in layer_mask: P of the selected layers in
// ascending layer order (align, may be null) and the per-row statistics [6][B][H][T] (rowmax / argmax, may be null).
struct AlignSink {
    uint32_t layer_mask;
    float* align;
    float* rowmax;
    int16_t* argmax;
};

// Teacher-forced eval forward (encoder, prenet, decoder, heads, postnet).  With a sink, the cross-attention probabilities of the
// selected layers are computed right after that layer's flash launch, while x2 still holds its queries; without one the
// launches are exactly those of tts_forward.  mel_before == null skips the heads and the postnet.
static int run_teacher_forced(TtsHandle* h, void* ws, const Ws& L, const int64_t* phonemes, const int32_t* phoneme_lens, const float* mels,
                              const int32_t* mel_lens, int B, int S, int T, uint64_t seed, int utt_offset, float* mel_before,
                              float* mel_after, float* stop_logits, const AlignSink* sink, cudaStream_t st) {
    int r = run_encoder(h, ws, L, phonemes, phoneme_lens, B, S, false, st);
    if (r) return r;
    const int M = B * T;
    // decoder activations must not alias the memory kept in ws.x during cross-attention: cross K/V is
    // already in the cache, so ws.x is free again.
    bf16 *x = wsp<bf16>(ws, L.x), *x2 = wsp<bf16>(ws, L.x2), *wide = wsp<bf16>(ws, L.wide), *a = wsp<bf16>(ws, L.a);
    float* y = wsp<float>(ws, L.y);
    bf16* mel16 = wsp<bf16>(ws, L.mel16);
    {   // P8: shift right, zero go-frame
        const int n = M * 24;
        mel_to_bf16_kernel<<<(n + 255) / 256, 256, 0, st>>>(mels, T, mel_lens, 1, mel16, nullptr, B, T);
        ++launch_counter();
        CK(cudaGetLastError());
    }
    {   // decoder prenet: dropout ALWAYS on (P7), masks keyed by (site, t, global utterance id)
        GemmParams p = gp(mel16, 96, h->pre_fc1, 96, M, 256, 96);
        p.T = T; p.bias = h->pre_b1; p.act = ACT_RELU; p.drop_site = SITE_DEC_PRENET_FC1; p.seed = seed; p.utt_offset = utt_offset; p.out_bf16 = x; p.ldo = 256;
        CK(launch_gemm_tc(p, st));
        p = gp(x, 256, h->pre_fc2, 256, M, 256, 256);
        p.T = T; p.bias = h->pre_b2; p.act = ACT_RELU; p.drop_site = SITE_DEC_PRENET_FC2; p.seed = seed; p.utt_offset = utt_offset; p.out_bf16 = x2; p.ldo = 256;
        CK(launch_gemm_tc(p, st));
        p = gp(x2, 256, h->pre_proj, 256, M, 512, 256);
        p.T = T; p.bias = h->pre_bp; p.pe = h->pe; p.alpha = h->dec_alpha; p.out_bf16 = x; p.ldo = 512;
        CK(launch_gemm_tc(p, st));
    }
    const bf16* ckv = wsp<bf16>(ws, L.cross_kv);
    const size_t ckv_layer = (size_t)B * kHeads * L.Spad * kDHead;
    for (int l = 0; l < 6; ++l) {
        auto& W = h->dec[l];
        GemmParams p = gp(x, 512, W.wqkv, 512, M, 1536, 512); p.bias = W.bqkv; p.out_bf16 = wide; p.ldo = 1536;
        CK(launch_gemm_tc(p, st));
        AttnParams at = ap_packed(wide, 1536, wide + 512, 1536, wide + 1024, 1536, a, 512, B, T, T, mel_lens, 1);
        CK(launch_flash_attn_tc(at, st));
        p = gp(a, 512, W.wo, 512, M, 512, 512); p.bias = W.bo; p.resid_bf16 = x; p.ldr = 512; p.out_f32 = y; p.ldo = 512;
        CK(launch_gemm_tc(p, st));
        CK(layernorm(y, W.ln1g, W.ln1b, x, nullptr, M, h->cfg.ln_eps, st));
        p = gp(x, 512, W.wq2, 512, M, 512, 512); p.bias = W.bq2; p.out_bf16 = x2; p.ldo = 512;
        CK(launch_gemm_tc(p, st));
        at = ap_packed(x2, 512, nullptr, 64, nullptr, 64, a, 512, B, T, S, phoneme_lens, 0);
        at.K = ckv + (size_t)(l * 2) * ckv_layer; at.V = ckv + (size_t)(l * 2 + 1) * ckv_layer;     // [B][H][S][64]
        at.k_bs = at.v_bs = (long)kHeads * L.Spad * kDHead; at.k_hs = at.v_hs = (long)L.Spad * kDHead; at.k_rs = at.v_rs = kDHead;
        CK(launch_flash_attn_tc(at, st));
        if (sink && ((sink->layer_mask >> l) & 1u)) {
            AlignParams al; memset(&al, 0, sizeof(al));
            al.Q = x2; al.q_bs = (long)T * 512; al.q_rs = 512;
            al.K = at.K; al.k_bs = at.k_bs; al.k_hs = at.k_hs;
            al.qlens = mel_lens; al.klens = phoneme_lens;
            al.B = B; al.H = kHeads; al.Lq = T; al.Lk = S; al.scale_log2 = at.scale_log2;
            const size_t per_layer = (size_t)B * kHeads * T;
            if (sink->align) al.P = sink->align + (size_t)__builtin_popcount(sink->layer_mask & ((1u << l) - 1u)) * per_layer * S;
            if (sink->rowmax) al.rowmax = sink->rowmax + (size_t)l * per_layer;
            if (sink->argmax) al.argmax = sink->argmax + (size_t)l * per_layer;
            CK(launch_cross_align(al, st));
        }
        p = gp(a, 512, W.wo2, 512, M, 512, 512); p.bias = W.bo2; p.resid_bf16 = x; p.ldr = 512; p.out_f32 = y; p.ldo = 512;
        CK(launch_gemm_tc(p, st));
        CK(layernorm(y, W.ln2g, W.ln2b, x, nullptr, M, h->cfg.ln_eps, st));
        p = gp(x, 512, W.w1, 512, M, 2048, 512); p.bias = W.b1; p.act = ACT_RELU; p.out_bf16 = wide; p.ldo = 2048;
        CK(launch_gemm_tc(p, st));
        p = gp(wide, 2048, W.w2, 2048, M, 512, 2048); p.bias = W.b2; p.resid_bf16 = x; p.ldr = 512; p.out_f32 = y; p.ldo = 512;
        CK(launch_gemm_tc(p, st));
        CK(layernorm(y, W.ln3g, W.ln3b, x, nullptr, M, h->cfg.ln_eps, st));
    }
    if (!mel_before) return 0;
    {   // [mel | stop] heads, zeroed past mel_lens
        GemmParams p = gp(x, 512, h->head_w, 512, M, 81, 512);
        p.T = T; p.bias = h->head_b; p.lens = mel_lens; p.scatter = SC_HEAD; p.out_f32 = mel_before; p.out2_f32 = stop_logits;
        CK(launch_gemm_tc(p, st));
    }
    {
        const int n = M * 24;
        mel_to_bf16_kernel<<<(n + 255) / 256, 256, 0, st>>>(mel_before, T, mel_lens, 0, mel16, wsp<float>(ws, L.mel32), B, T);
        ++launch_counter();
        CK(cudaGetLastError());
    }
    return run_postnet(h, ws, L, mel_lens, B, T, mel_after, st);
}

extern "C" int tts_forward(TtsHandle* h, void* ws, const int64_t* phonemes, const int32_t* phoneme_lens, const float* mels,
                           const int32_t* mel_lens, int B, int S, int T, uint64_t seed, int utt_offset, float* mel_before,
                           float* mel_after, float* stop_logits, void* stream) {
    if (!h || !ws || !phonemes || !phoneme_lens || !mels || !mel_lens || !mel_before || !mel_after || !stop_logits) return TTS_E_ARG;
    if (B <= 0 || S <= 0 || T <= 0) return TTS_E_ARG;
    if (!h->finalized) FAIL(TTS_E_STATE, "weights not finalised");
    if (S > h->cfg.max_pos || T > h->cfg.max_pos) FAIL(TTS_E_ARG, "sequence exceeds max_pos");
    DEV_GUARD(h);
    if (int r = take_conditioning(h, h->cond_inf, ws, B, "tts_set_conditioning")) return r;
    return run_teacher_forced(h, ws, ws_layout(h, B, S, T), phonemes, phoneme_lens, mels, mel_lens, B, S, T, seed, utt_offset, mel_before,
                              mel_after, stop_logits, nullptr, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------
// alignments and durations (align.cuh).  Scratch: rowmax fp32 [6][B][H][T] | argmax int16 [6][B][H][T] | focus fp32 [6][B][H].
namespace {
struct AlignScratch {
    size_t rowmax, argmax, focus, total;
    static AlignScratch make(int B, int T) {
        AlignScratch a; size_t o = 0;
        auto take = [&](size_t bytes) { size_t r = o; o = align_up(o + bytes); return r; };
        const size_t rows = (size_t)6 * B * kHeads * T;
        a.rowmax = take(rows * 4); a.argmax = take(rows * 2); a.focus = take((size_t)6 * B * kHeads * 4);
        a.total = o;
        return a;
    }
};
}  // namespace

extern "C" size_t tts_align_scratch_bytes(TtsHandle* h, int B, int S, int T) {
    if (!h || B <= 0 || S <= 0 || T <= 0) return 0;
    return AlignScratch::make(B, T).total;
}

extern "C" int tts_forward_align(TtsHandle* h, void* ws, void* scratch, const int64_t* phonemes, const int32_t* phoneme_lens,
                                 const float* mels, const int32_t* mel_lens, int B, int S, int T, uint64_t seed, int utt_offset,
                                 uint32_t layer_mask, int fixed_head, float* mel_before, float* mel_after, float* stop_logits,
                                 float* align, float* focus, int32_t* durations, int32_t* head, void* stream) {
    if (!h || !ws || !phonemes || !phoneme_lens || !mels || !mel_lens || B <= 0 || S <= 0 || T <= 0) return TTS_E_ARG;
    if (!h->finalized) FAIL(TTS_E_STATE, "weights not finalised");
    if (S > h->cfg.max_pos || T > h->cfg.max_pos) FAIL(TTS_E_ARG, "sequence exceeds max_pos");
    if (S > 32767) FAIL(TTS_E_ARG, "S exceeds the int16 range of the per-row argmax");
    if (!mel_before != !mel_after || !mel_before != !stop_logits) FAIL(TTS_E_ARG, "mel_before, mel_after and stop_logits: all or none");
    if (layer_mask == 0 || layer_mask > 0x3fu) FAIL(TTS_E_ARG, "layer_mask must select decoder layers 0..5 (1 .. 0x3f)");
    if (fixed_head < -1 || fixed_head >= 6 * kHeads || (fixed_head >= 0 && !((layer_mask >> (fixed_head / kHeads)) & 1u)))
        FAIL(TTS_E_ARG, "fixed_head must be -1 or layer * 8 + h of a selected layer");
    const bool stats = focus || durations || head;
    if (stats && !scratch) FAIL(TTS_E_ARG, "focus / durations / head need the scratch of tts_align_scratch_bytes");
    DEV_GUARD(h);
    if (int r = take_conditioning(h, h->cond_inf, ws, B, "tts_set_conditioning")) return r;
    cudaStream_t st = (cudaStream_t)stream;
    const AlignScratch A = AlignScratch::make(B, T);
    AlignSink sink{layer_mask, align, stats ? wsp<float>(scratch, A.rowmax) : nullptr, stats ? wsp<int16_t>(scratch, A.argmax) : nullptr};
    int r = run_teacher_forced(h, ws, ws_layout(h, B, S, T), phonemes, phoneme_lens, mels, mel_lens, B, S, T, seed, utt_offset, mel_before,
                               mel_after, stop_logits, (align || stats) ? &sink : nullptr, st);
    if (r) return r;
    float* f = focus ? focus : wsp<float>(scratch, A.focus);
    if (focus || ((durations || head) && fixed_head < 0)) {
        const int warps = 6 * B * kHeads;
        focus_kernel<<<(warps + 7) / 8, 256, 0, st>>>(sink.rowmax, mel_lens, B, kHeads, T, layer_mask, f);
        ++launch_counter();
        CK(cudaGetLastError());
    }
    if (durations || head) {
        durations_kernel<<<B, 256, (size_t)S * 4, st>>>(f, sink.argmax, mel_lens, phoneme_lens, B, kHeads, S, T, layer_mask, fixed_head,
                                                        durations, head);
        ++launch_counter();
        CK(cudaGetLastError());
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------
// profiling aid: copy the per-phase globaltimer stamps of the persistent decode kernel to the host.
extern "C" int tts_debug_phase_timestamps(TtsHandle* h, void* ws, unsigned long long* out, int n_steps, void* stream) {
    if (!h || !ws || !out || n_steps <= 0) return TTS_E_ARG;
    const auto& ds = h->session;
    if (!ds.active || n_steps != ds.T) FAIL(TTS_E_STATE, "no decode session / n_steps must equal max_len");
    CK(cudaMemcpyAsync(out, wsp<unsigned long long>(ws, ds.L.ts), (size_t)(n_steps + 1) * CL_TS_COLS * 8, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CK(cudaStreamSynchronize((cudaStream_t)stream));
    return 52;
}

extern "C" int tts_debug_read_dump(TtsHandle* h, void* ws, int64_t offset, int64_t n, float* out_host, void* stream) {
    if (!h || !ws || !out_host || offset < 0 || n <= 0) return TTS_E_ARG;
    const auto& ds = h->session;
    if (!ds.active) FAIL(TTS_E_STATE, "no decode session");
    const size_t cap = (size_t)ds.B * (size_t)std::max(ds.S, ds.T) * 2048 * 2 / 4;
    if ((size_t)(offset + n) > cap) FAIL(TTS_E_ARG, "dump range exceeds the debug buffer");
    CK(cudaMemcpyAsync(out_host, wsp<float>(ws, ds.L.wide) + offset, (size_t)n * 4, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CK(cudaStreamSynchronize((cudaStream_t)stream));
    return 0;
}

extern "C" int tts_debug_kv_index(int row, int dim, int which) {
    if (row < 0 || row >= KV_BLOCK_ROWS || dim < 0 || dim >= kDHead || which < 0 || which > 1) return -1;
    return which ? kv_v_elem(row, dim) : kv_k_elem(row, dim);
}

extern "C" int64_t tts_debug_pack_segment(const float* w, int N, int K, const int32_t* rows, int nrows, int kp_base, int KP, int TW,
                                          unsigned char* out, int64_t out_bytes) {
    if (!w || !rows || N <= 0 || K <= 0 || nrows <= 0 || KP <= 0 || kp_base < 0 || TW <= 0 || nrows % (16 * TW) != 0) return -1;
    const int64_t need = (int64_t)(nrows / 16) * KP * 1024;
    if (!out || out_bytes < need) return need;
    std::vector<unsigned char> seg;
    seg.reserve((size_t)need);
    pack_cluster_segment(seg, w, N, K, std::vector<int>(rows, rows + nrows), kp_base, KP, TW);
    memcpy(out, seg.data(), seg.size());
    return (int64_t)seg.size();
}

// per-kernel test entry points
extern "C" int tts_k_gemm(const void* A, const void* W, const float* bias, float* C, int M, int N, int K, int act, void* stream) {
    if (!A || !W || !C || M <= 0 || N <= 0 || K <= 0 || (K % 8) || (N % 128)) return TTS_E_ARG;
    GemmParams p = gp((const bf16*)A, K, (const bf16*)W, K, M, N, K);
    p.bias = bias; p.act = act; p.out_f32 = C; p.ldo = N;
    return (int)launch_gemm_tc(p, (cudaStream_t)stream);
}
extern "C" int tts_k_conv5(const void* X, const void* W, const float* bias, const int32_t* lens, float* Y, int B, int T, int Cin,
                              int Cout, int act, void* stream) {
    if (!X || !W || !Y || B <= 0 || T <= 0 || (Cin % 8) || (Cout % 128)) return TTS_E_ARG;
    GemmParams p = gp((const bf16*)X, Cin, (const bf16*)W, Cin, B * T, Cout, Cin);
    p.taps = 5; p.T = T; p.bias = bias; p.act = act; p.lens = lens; p.out_f32 = Y; p.ldo = Cout;
    return (int)launch_gemm_tc(p, (cudaStream_t)stream);
}
extern "C" int tts_k_attention(const void* Q, const void* K, const void* V, void* O, const int32_t* klens, int B, int H, int Lq,
                               int Lk, int causal, void* stream) {
    if (!Q || !K || !V || !O || B <= 0 || H <= 0 || Lq <= 0 || Lk <= 0) return TTS_E_ARG;
    const int ld = H * 64;
    AttnParams a = ap_packed((const bf16*)Q, ld, (const bf16*)K, ld, (const bf16*)V, ld, (bf16*)O, ld, B, Lq, Lk, klens, causal);
    a.H = H;
    return (int)launch_flash_attn_tc(a, (cudaStream_t)stream);
}
extern "C" int tts_k_attention_lse(const void* Q, const void* K, const void* V, void* O, float* lse, const int32_t* klens, int B, int H,
                                   int Lq, int Lk, int causal, void* stream) {
    if (!Q || !K || !V || !O || !lse || B <= 0 || H <= 0 || Lq <= 0 || Lk <= 0) return TTS_E_ARG;
    const int ld = H * 64;
    AttnParams a = ap_packed((const bf16*)Q, ld, (const bf16*)K, ld, (const bf16*)V, ld, (bf16*)O, ld, B, Lq, Lk, klens, causal);
    a.H = H; a.lse = lse;
    return (int)launch_flash_attn_tc(a, (cudaStream_t)stream);
}
extern "C" int tts_k_cross_align(const void* Q, int ldq, const void* K, const int32_t* qlens, const int32_t* klens, int B, int H, int Lq,
                                 int Lk, float* P, float* rowmax, int16_t* argmax, void* stream) {
    if (!Q || !K || B <= 0 || H <= 0 || Lq <= 0 || Lk <= 0 || Lk > 32767 || ldq < H * 64 || (ldq % 8)) return TTS_E_ARG;
    AlignParams a; memset(&a, 0, sizeof(a));
    a.Q = (const bf16*)Q; a.q_bs = (long)Lq * ldq; a.q_rs = ldq;
    a.K = (const bf16*)K; a.k_hs = (long)Lk * 64; a.k_bs = (long)H * Lk * 64;
    a.qlens = qlens; a.klens = klens; a.B = B; a.H = H; a.Lq = Lq; a.Lk = Lk; a.scale_log2 = 0.125f * kLog2e;
    a.P = P; a.rowmax = rowmax; a.argmax = argmax;
    return (int)launch_cross_align(a, (cudaStream_t)stream);
}
namespace {
// fp32 -> bf16 rows (dQ accumulator -> operand)
__global__ void f32_to_bf16_kernel(const float* __restrict__ x, bf16* __restrict__ y, long n4) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n4) {
        const float4 v = reinterpret_cast<const float4*>(x)[i];
        reinterpret_cast<uint2*>(y)[i] = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
    }
}
AttnBwdParams abp_packed(const AttnParams& f, const bf16* dO, const float* lse, const float* dsum, float* dQ, int lddq, bf16* dK, int lddk,
                         bf16* dV, int lddv) {
    AttnBwdParams a; memset(&a, 0, sizeof(a));
    a.Q = f.Q; a.K = f.K; a.V = f.V; a.dO = dO;
    a.q_bs = f.q_bs; a.q_hs = f.q_hs; a.q_rs = f.q_rs; a.k_bs = f.k_bs; a.k_hs = f.k_hs; a.k_rs = f.k_rs;
    a.v_bs = f.v_bs; a.v_hs = f.v_hs; a.v_rs = f.v_rs; a.o_bs = f.o_bs; a.o_hs = f.o_hs; a.o_rs = f.o_rs;
    a.lse = lse; a.dsum = dsum;
    a.dQ = dQ; a.dq_bs = (long)f.Lq * lddq; a.dq_hs = 64; a.dq_rs = lddq;
    a.dK = dK; a.dk_bs = (long)f.Lk * lddk; a.dk_hs = 64; a.dk_rs = lddk;
    a.dV = dV; a.dv_bs = (long)f.Lk * lddv; a.dv_hs = 64; a.dv_rs = lddv;
    a.B = f.B; a.H = f.H; a.Lq = f.Lq; a.Lk = f.Lk; a.klens = f.klens; a.causal = f.causal;
    a.scale_log2 = f.scale_log2; a.scale = 0.125f;
    return a;
}
}  // namespace
extern "C" int tts_k_attention_bwd(const void* Q, const void* K, const void* V, const void* O, const void* dO, const float* lse,
                                   const int32_t* klens, void* dQ, void* dK, void* dV, float* scratch, int B, int H, int Lq, int Lk,
                                   int causal, void* stream) {
    if (!Q || !K || !V || !O || !dO || !lse || !dQ || !dK || !dV || !scratch || B <= 0 || H <= 0 || Lq <= 0 || Lk <= 0) return TTS_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const int ld = H * 64;
    const long nq = (long)B * Lq * ld;
    float* dq32 = scratch; float* dsum = scratch + nq;
    AttnParams f = ap_packed((const bf16*)Q, ld, (const bf16*)K, ld, (const bf16*)V, ld, (bf16*)const_cast<void*>(O), ld, B, Lq, Lk, klens, causal);
    f.H = H;
    cudaError_t e = cudaMemsetAsync(dq32, 0, nq * 4, st);
    if (e != cudaSuccess) return (int)e;
    attn_dsum_kernel<<<(B * H * Lq + 31) / 32, 256, 0, st>>>((const bf16*)O, (const bf16*)dO, f.o_bs, f.o_hs, f.o_rs, dsum, B, H, Lq);
    ++launch_counter();
    AttnBwdParams a = abp_packed(f, (const bf16*)dO, lse, dsum, dq32, ld, (bf16*)dK, ld, (bf16*)dV, ld);
    e = launch_flash_attn_bwd_tc(a, st);
    if (e != cudaSuccess) return (int)e;
    f32_to_bf16_kernel<<<(unsigned)((nq / 4 + 255) / 256), 256, 0, st>>>(dq32, (bf16*)dQ, nq / 4);
    ++launch_counter();
    return (int)cudaGetLastError();
}
extern "C" int tts_k_layernorm(const float* X, const float* gamma, const float* beta, void* Y, int M, float eps, void* stream) {
    if (!X || !gamma || !beta || !Y || M <= 0) return TTS_E_ARG;
    return (int)layernorm(X, gamma, beta, (bf16*)Y, nullptr, M, eps, (cudaStream_t)stream);
}
extern "C" int tts_k_speaker_cond(const int32_t* sids, const float* spembs, int B, int n_speakers, int D, const float* table, const float* W,
                                  const float* bias, float* cond, float* nhat, void* stream) {
    if (!cond || B <= 0 || n_speakers < 0 || D < 0 || D > kSpkMaxDim || (!table && !W) || (table && (!sids || n_speakers == 0)) ||
        (!W != (D == 0)) || (W && (!bias || !spembs || !nhat)))
        return TTS_E_ARG;
    return (int)launch_speaker_cond(sids, spembs, B, n_speakers, D, table, W, bias, cond, nhat, (cudaStream_t)stream);
}
extern "C" int tts_k_layernorm_cond(const float* X, const float* gamma, const float* beta, const float* cond, void* Y, int M, int S, float eps,
                                    void* stream) {
    if (!X || !gamma || !beta || !cond || !Y || M <= 0 || S <= 0) return TTS_E_ARG;
    return (int)launch_layernorm_cond(X, gamma, beta, (bf16*)Y, nullptr, M, eps, cond, S, (cudaStream_t)stream);
}
extern "C" int tts_k_speaker_cond_bwd(const float* dmem, const int32_t* plens, const int32_t* sids, const float* nhat, int B, int S, int n_speakers,
                                      int D, float* dcond, float* dE, float* dW, float* dbias, void* stream) {
    if (!dmem || !plens || !dcond || B <= 0 || S <= 0 || n_speakers < 0 || D < 0 || (!dE && !dW) || (dE && (!sids || n_speakers == 0)) ||
        (!dW != (D == 0)) || (dW && (!dbias || !nhat)))
        return TTS_E_ARG;
    return (int)launch_speaker_cond_bwd(dmem, plens, sids, nhat, B, S, n_speakers, D, dcond, dE, dW, dbias, (cudaStream_t)stream);
}
extern "C" int tts_k_philox_bits(uint64_t seed, int site, int T, int B, int C, int utt_offset, uint8_t* out, void* stream) {
    if (!out || T <= 0 || B <= 0 || C <= 0) return TTS_E_ARG;
    const int n = T * B * C;
    philox_bits_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(seed, site, T, B, C, utt_offset, out);
    ++launch_counter();
    return (int)cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// training (train.cuh)
#include "train.cuh"

// per-kernel test entry points of the training step: each launches what the step launches, through the same helpers
extern "C" int tts_k_wgrad(const void* dY, int ldy, int Cout, const void* X, int ldx, int Cin, int taps, int T, int nb, float* dW, float* dbias,
                           void* stream) {
    if (!dY || !X || !dW || Cout <= 0 || Cin <= 0 || T <= 0 || nb <= 0 || (taps != 1 && taps != 5) || ldy < Cout || ldx < Cin) return TTS_E_ARG;
    WgradParams g;
    g.dY = (const bf16*)dY; g.ldy = ldy; g.Cout = Cout; g.X = (const bf16*)X; g.ldx = ldx; g.Cin = Cin; g.taps = taps;
    g.T = T; g.nb = nb; g.dW = dW; g.dbias = dbias;
    return (int)launch_wgrad_tc(g, (cudaStream_t)stream);
}
extern "C" int tts_k_dgrad(const float* W, int N, int K, int taps, const void* dY, int ldy, int Kdy, int M, int T, float* out_f32, void* out_bf16,
                           int ldo, void* scratch, void* stream) {
    if (!W || !dY || !scratch || (!out_f32 == !out_bf16) || N <= 0 || K <= 0 || M <= 0 || T <= 0 || (M % T) || (taps != 1 && taps != 5) ||
        Kdy < N || ldy < Kdy || ldo < K)
        return TTS_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const TrMat m = tr_mat_dims(N, K, taps);
    int blocks = 0;
    const PackDesc d = tr_pack_desc(m, 1, 0, 0, 0, &blocks);
    PackDesc* dd = nullptr;
    cudaError_t e = cudaMallocAsync(&dd, sizeof(PackDesc), st);
    if (e != cudaSuccess) return (int)e;
    e = cudaMemcpyAsync(dd, &d, sizeof(PackDesc), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
        cast_pack_all_kernel<<<blocks, 256, 0, st>>>(dd, 1, W, (bf16*)scratch);
        ++launch_counter();
        e = cudaGetLastError();
    }
    const cudaError_t ef = cudaFreeAsync(dd, st);
    if (e != cudaSuccess) return (int)e;
    if (ef != cudaSuccess) return (int)ef;
    GemmParams p = tr_dgrad_params(m, (const bf16*)scratch, (const bf16*)dY, ldy, Kdy, M, T);
    p.out_f32 = out_f32; p.out_bf16 = (bf16*)out_bf16; p.ldo = ldo;
    return (int)launch_gemm_tc(p, st);
}
extern "C" int tts_k_bn_train_fwd(const float* x, int B, int T, int C, const int32_t* lens, float* stat, const float* gamma, const float* beta,
                                  float eps, int act, int site, const uint64_t* seed, int utt_offset, void* out16, int ldo, float* out32,
                                  float* run_mean, float* run_var, void* stream) {
    if (!x || !lens || !stat || !gamma || !beta || !seed || B <= 0 || T <= 0 || C <= 0 || (C % 4) || 2 * C > BN_STAT_FLOATS ||
        (out16 && (ldo < C || (ldo % 4))) || (!run_mean != !run_var))
        return TTS_E_ARG;
    return (int)launch_bn_train_fwd(x, B * T, C, T, B, lens, stat, gamma, beta, eps, act, site, seed, utt_offset, (bf16*)out16, ldo, out32, run_mean,
                                    run_var, (cudaStream_t)stream);
}
extern "C" int tts_k_bn_train_bwd(const void* dout, int dout_bf16, int ldd, const float* x, int B, int T, int C, const int32_t* lens, const float* stat,
                                  const float* gamma, const float* beta, float eps, int act, int site, const uint64_t* seed, int utt_offset,
                                  float* dgamma, float* dbeta, void* dx, int ldx, void* stream) {
    if (!dout || !x || !lens || !stat || !gamma || !beta || !seed || !dgamma || !dbeta || !dx || B <= 0 || T <= 0 || C <= 0 || (C % 4) ||
        2 * C > BN_STAT_FLOATS || ldd < C || ldx < C || (ldx % 4))
        return TTS_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (dout_bf16)
        return (int)launch_bn_train_bwd<bf16>((const bf16*)dout, ldd, x, B * T, C, T, B, lens, stat, gamma, beta, eps, act, site, seed, utt_offset, dbeta,
                                              dgamma, (bf16*)dx, ldx, st);
    return (int)launch_bn_train_bwd<float>((const float*)dout, ldd, x, B * T, C, T, B, lens, stat, gamma, beta, eps, act, site, seed, utt_offset, dbeta,
                                           dgamma, (bf16*)dx, ldx, st);
}
extern "C" int tts_k_ln_bwd(const float* dx, const float* ypre, const float* gamma, float eps, int M, int T, float* dy32, void* dsub16, int site,
                            const uint64_t* seed, int utt_offset, uint32_t thresh, float dscale, float* dgamma, float* dbeta, void* stream) {
    if (!dx || !ypre || !gamma || !seed || !dgamma || !dbeta || M <= 0 || T <= 0) return TTS_E_ARG;
    return (int)launch_ln_bwd(dx, ypre, gamma, eps, M, T, dy32, (bf16*)dsub16, site, seed, utt_offset, thresh, dscale, dgamma, dbeta, (cudaStream_t)stream);
}
extern "C" int tts_k_loss(const float* before, const float* after, const float* stop, const float* target, const int32_t* lens, int B, int T,
                          float pos_weight, float* acc, float* dbefore, float* dafter, float* dstop, float* loss, void* stream) {
    if (!before || !after || !stop || !target || !lens || !acc || !dbefore || !dafter || !dstop || !loss || B <= 0 || T <= 0) return TTS_E_ARG;
    return (int)launch_loss(before, after, stop, target, lens, B, T, pos_weight, acc, dbefore, dafter, dstop, loss, (cudaStream_t)stream);
}
extern "C" int tts_k_head_grad(const float* dbefore, const float* dafter, const void* dpost0, int ldp, const float* dstop, const int32_t* lens, int B,
                               int T, void* dhead, void* stream) {
    if (!dbefore || !dafter || !dpost0 || !dstop || !lens || !dhead || B <= 0 || T <= 0 || ldp < 80) return TTS_E_ARG;
    return (int)launch_head_grad(dbefore, dafter, (const bf16*)dpost0, ldp, dstop, lens, B * T, T, (bf16*)dhead, (cudaStream_t)stream);
}
extern "C" int tts_k_dropw_bwd(const float* d, void* out, int B, int T, int site, const uint64_t* seed, int utt_offset, uint32_t thresh, float dscale,
                               const float* pe, float* dalpha, int decoder, void* stream) {
    if (!d || !out || !seed || !pe || !dalpha || B <= 0 || T <= 0) return TTS_E_ARG;
    return (int)launch_dropw_bwd(decoder != 0, d, (bf16*)out, B * T, T, site, seed, utt_offset, thresh, dscale, pe, dalpha, (cudaStream_t)stream);
}
extern "C" int tts_k_embed_bwd(const void* d, const int64_t* ph, const int32_t* lens, int B, int S, int V, float* dE, void* stream) {
    if (!d || !ph || !lens || !dE || B <= 0 || S <= 0 || V <= 0) return TTS_E_ARG;
    return (int)launch_embed_bwd((const bf16*)d, ph, lens, B * S, S, V, dE, (cudaStream_t)stream);
}

extern "C" int tts_train_begin(TtsHandle* h) {
    if (!h) return TTS_E_ARG;
    if (!h->finalized) FAIL(TTS_E_STATE, "weights not finalised");
    DEV_GUARD(h);
    train_free(h);
    int r = train_build(h);
    if (r) { train_free(h); return r; }
    if ((r = train_repack(h, 0))) return r;
    CK(cudaDeviceSynchronize());
    return 0;
}
extern "C" int tts_train_end(TtsHandle* h) { if (!h) return TTS_E_ARG; DeviceGuard dev_guard_(h->device); return train_free(h); }
extern "C" size_t tts_train_workspace_bytes(TtsHandle* h, int B, int S, int T) {
    if (!h || B <= 0 || S <= 0 || T <= 0) return 0;
    return TrWs::make(nullptr, B, S, T, conditioned(h) ? h->cfg.spk_embed_dim : -1).total;
}
namespace {
// context of one training call: workspace views, dropout threshold / scale, flat parameter and gradient buffers
TrCtx train_ctx(TtsHandle* h, void* ws, int B, int S, int T, int utt_offset, double p_residual, cudaStream_t st) {
    TrCtx c;
    TtsTrain* t = h->train;
    c.h = h; c.t = t; c.w = TrWs::make(reinterpret_cast<unsigned char*>(ws), B, S, T, conditioned(h) ? h->cfg.spk_embed_dim : -1); c.st = st;
    c.B = B; c.S = S; c.T = T; c.seed = c.w.seed_dev; c.utt0 = utt_offset;
    c.thresh = (uint32_t)(p_residual * 4294967296.0); c.dscale = 1.0f / (float)(1.0 - p_residual);
    c.P = t->P; c.G = t->G;
    return c;
}
// Checks the arguments of a training call that takes a batch, builds its context and stages the inputs: the step itself (eager
// or replayed from its CUDA graph) reads workspace memory only.  The caller holds the device guard.
int train_stage(TrCtx& c, TtsHandle* h, void* ws, const int64_t* phonemes, const int32_t* phoneme_lens, const float* mels, const int32_t* mel_lens,
                int B, int S, int T, uint64_t seed, int utt_offset, double p_residual, cudaStream_t st) {
    if (!ws || !phonemes || !phoneme_lens || !mels || !mel_lens || B <= 0 || S <= 0 || T <= 0) return TTS_E_ARG;
    if (!h->train) FAIL(TTS_E_STATE, "tts_train_begin has not been called");
    if (S > h->cfg.max_pos || T > h->cfg.max_pos) FAIL(TTS_E_ARG, "sequence exceeds max_pos");
    if (p_residual < 0.0 || p_residual >= 1.0) FAIL(TTS_E_ARG, "p_residual out of range");
    if (int r = take_conditioning(h, h->cond_train, ws, B, "tts_train_set_conditioning")) return r;
    c = train_ctx(h, ws, B, S, T, utt_offset, p_residual, st);
    CK(cudaMemcpyAsync(c.w.plens, phoneme_lens, (size_t)B * 4, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(c.w.mlens, mel_lens, (size_t)B * 4, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(c.w.ph_in, phonemes, (size_t)B * S * 8, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(c.w.mels_in, mels, (size_t)B * T * 80 * 4, cudaMemcpyDeviceToDevice, st));
    set_u64_kernel<<<1, 1, 0, st>>>(c.w.seed_dev, seed);
    ++launch_counter();
    return 0;
}
}  // namespace
extern "C" int tts_train_set_conditioning(TtsHandle* h, void* ws, int B, const int32_t* sids, const float* spembs, void* stream) {
    if (!h) return TTS_E_ARG;
    if (!h->train) FAIL(TTS_E_STATE, "tts_train_begin has not been called");
    DEV_GUARD(h);
    const TrWs w = TrWs::make(nullptr, B, 1, 1, h->cfg.spk_embed_dim);  // the region's offsets depend on B only
    int r = stage_conditioning(h, ws, B, sids, spembs, (size_t)w.sids, (size_t)w.spembs, (cudaStream_t)stream);
    if (r) return r;
    h->cond_train = {ws, B};
    return 0;
}
extern "C" int tts_train_step(TtsHandle* h, void* ws, const int64_t* phonemes, const int32_t* phoneme_lens, const float* mels, const int32_t* mel_lens,
                              int B, int S, int T, uint64_t seed, int utt_offset, double p_residual, float pos_weight, float* loss_out, void* stream) {
    if (!h || !loss_out) return TTS_E_ARG;
    DEV_GUARD(h);
    TrCtx c;
    int r = train_stage(c, h, ws, phonemes, phoneme_lens, mels, mel_lens, B, S, T, seed, utt_offset, p_residual, (cudaStream_t)stream);
    if (r) return r;
    TtsTrain* t = h->train;
    const TtsTrain::GraphKey key{ws, B, S, T, utt_offset, p_residual, pos_weight, loss_out, c.st};
    if (h->train_graph && t->graph_exec && key == t->graph_key) {
        CK(cudaGraphLaunch(t->graph_exec, c.st));
        launch_counter() += t->graph_launches;
        return 0;
    }
    if (h->train_graph && key == t->seen_key) {                          // second step of this shape: capture, then replay
        if (t->graph_exec) { cudaGraphExecDestroy(t->graph_exec); t->graph_exec = nullptr; }
        const unsigned long long l0 = launch_counter();
        cudaGraph_t graph = nullptr;
        // (the caller's stream may be the legacy default stream, which cannot be captured: record on a stream of our own)
        if (!t->cap_stream) CK(cudaStreamCreateWithFlags(&t->cap_stream, cudaStreamNonBlocking));
        cudaStream_t user_st = c.st;
        c.st = t->cap_stream;
        CK(cudaStreamBeginCapture(c.st, cudaStreamCaptureModeThreadLocal));
        r = train_forward_backward(c, loss_out, pos_weight);
        cudaError_t e = cudaStreamEndCapture(c.st, &graph);
        c.st = user_st;
        if (r) { if (graph) cudaGraphDestroy(graph); return r; }
        CK(e);
        t->graph_launches = launch_counter() - l0;
        launch_counter() = l0;
        e = cudaGraphInstantiate(&t->graph_exec, graph, 0);
        cudaGraphDestroy(graph);
        CK(e);
        t->graph_key = key;
        CK(cudaGraphLaunch(t->graph_exec, c.st));
        launch_counter() += t->graph_launches;
        return 0;
    }
    t->seen_key = key;
    return train_forward_backward(c, loss_out, pos_weight);
}
extern "C" int tts_train_forward(TtsHandle* h, void* ws, const int64_t* phonemes, const int32_t* phoneme_lens, const float* mels, const int32_t* mel_lens,
                                 int B, int S, int T, uint64_t seed, int utt_offset, double p_residual, void* stream) {
    if (!h) return TTS_E_ARG;
    DEV_GUARD(h);
    TrCtx c;
    int r = train_stage(c, h, ws, phonemes, phoneme_lens, mels, mel_lens, B, S, T, seed, utt_offset, p_residual, (cudaStream_t)stream);
    return r ? r : train_forward(c);
}
extern "C" int tts_train_backward(TtsHandle* h, void* ws, int B, int S, int T, int utt_offset, double p_residual, const float* d_before,
                                  const float* d_after, const float* d_stop, void* stream) {
    if (!h || !ws || !d_before || !d_after || !d_stop || B <= 0 || S <= 0 || T <= 0) return TTS_E_ARG;
    if (!h->train) FAIL(TTS_E_STATE, "tts_train_begin has not been called");
    if (p_residual < 0.0 || p_residual >= 1.0) FAIL(TTS_E_ARG, "p_residual out of range");
    DEV_GUARD(h);
    TrCtx c = train_ctx(h, ws, B, S, T, utt_offset, p_residual, (cudaStream_t)stream);      // (the seed staged by the forward is still in the workspace)
    const size_t n = (size_t)B * T;
    CK(cudaMemcpyAsync(c.w.dbefore, d_before, n * 80 * 4, cudaMemcpyDeviceToDevice, c.st));
    CK(cudaMemcpyAsync(c.w.dafter, d_after, n * 80 * 4, cudaMemcpyDeviceToDevice, c.st));
    CK(cudaMemcpyAsync(c.w.dstop, d_stop, n * 4, cudaMemcpyDeviceToDevice, c.st));
    return train_backward(c);
}
extern "C" int tts_train_write(TtsHandle* h, int which, int64_t offset, int64_t numel, const float* host_in) {
    if (!h || !h->train || !host_in || offset < 0 || numel <= 0) return TTS_E_ARG;
    TtsTrain* t = h->train;
    float* dst = which == 0 ? t->P : which == 2 ? t->RS : nullptr;
    const size_t lim = which == 2 ? t->nrs : t->n;
    if (!dst || (size_t)(offset + numel) > lim) return TTS_E_ARG;
    DEV_GUARD(h);
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(dst + offset, host_in, (size_t)numel * 4, cudaMemcpyHostToDevice));
    return 0;
}
extern "C" int tts_train_outputs(TtsHandle* h, void* ws, int B, int S, int T, float* mel_before, float* mel_after, float* stop_logits, void* stream) {
    if (!h || !ws || !h->train) return TTS_E_ARG;
    TrWs w = TrWs::make(reinterpret_cast<unsigned char*>(ws), B, S, T, conditioned(h) ? h->cfg.spk_embed_dim : -1);
    cudaStream_t st = (cudaStream_t)stream;
    if (mel_before) CK(cudaMemcpyAsync(mel_before, w.mel_before, (size_t)B * T * 80 * 4, cudaMemcpyDeviceToDevice, st));
    if (mel_after) CK(cudaMemcpyAsync(mel_after, w.mel_after, (size_t)B * T * 80 * 4, cudaMemcpyDeviceToDevice, st));
    if (stop_logits) CK(cudaMemcpyAsync(stop_logits, w.stop, (size_t)B * T * 4, cudaMemcpyDeviceToDevice, st));
    return 0;
}
extern "C" int tts_train_grads(TtsHandle* h, float** grads_dev, int64_t* numel) {
    if (!h || !h->train || !grads_dev || !numel) return TTS_E_ARG;
    *grads_dev = h->train->G; *numel = (int64_t)h->train->n;
    return 0;
}
extern "C" int tts_train_adam(TtsHandle* h, float lr, float beta1, float beta2, float eps, float grad_scale, void* stream) {
    if (!h || !h->train) return TTS_E_ARG;
    DEV_GUARD(h);
    TtsTrain* t = h->train;
    cudaStream_t st = (cudaStream_t)stream;
    ++t->step;
    const float bc1 = 1.f - std::pow(beta1, (float)t->step), bc2 = 1.f - std::pow(beta2, (float)t->step);
    adam_kernel<<<1184, 256, 0, st>>>(t->P, t->G, t->M1, t->V2, (long)t->n, lr, beta1, beta2, eps, bc1, bc2, grad_scale);
    ++launch_counter();
    CK(cudaGetLastError());
    return train_repack(h, st);
}
// ---- data-parallel peers: fused reduce-scatter -> Adam -> all-gather over NVLink peer memory -------------------------------
extern "C" int tts_train_ipc_handles(TtsHandle* h, void* handle_P_64, void* handle_G_64) {
    if (!h || !h->train || !handle_P_64 || !handle_G_64) return TTS_E_ARG;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    DEV_GUARD(h);
    CK(cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(handle_P_64), h->train->P));
    CK(cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(handle_G_64), h->train->G));
    return 0;
}
extern "C" int tts_train_set_peers(TtsHandle* h, int rank, int world, const void* handles_P, const void* handles_G) {
    if (!h || !h->train || world < 1 || world > 8 || rank < 0 || rank >= world || (world > 1 && (!handles_P || !handles_G))) return TTS_E_ARG;
    DEV_GUARD(h);
    TtsTrain* t = h->train;
    for (void*& q : t->ipc_opened) if (q) { cudaIpcCloseMemHandle(q); q = nullptr; }
    t->rank = rank; t->world = world;
    for (int r = 0; r < world; ++r) {
        if (r == rank) { t->peers.P[r] = t->P; t->peers.G[r] = t->G; continue; }
        cudaIpcMemHandle_t hp, hg;
        memcpy(&hp, reinterpret_cast<const char*>(handles_P) + 64 * r, 64); memcpy(&hg, reinterpret_cast<const char*>(handles_G) + 64 * r, 64);
        void *pp = nullptr, *pg = nullptr;
        CK(cudaIpcOpenMemHandle(&pp, hp, cudaIpcMemLazyEnablePeerAccess));
        t->ipc_opened[2 * r] = pp;
        CK(cudaIpcOpenMemHandle(&pg, hg, cudaIpcMemLazyEnablePeerAccess));
        t->ipc_opened[2 * r + 1] = pg;
        t->peers.P[r] = reinterpret_cast<float*>(pp); t->peers.G[r] = reinterpret_cast<const float*>(pg);
    }
    return 0;
}
// The caller orders this between two cross-rank barriers on the stream: every rank's backward is complete before, every
// rank's shard has been written everywhere after (then tts_train_repack refreshes the bf16 operand copies).
extern "C" int tts_train_adam_peers(TtsHandle* h, float lr, float beta1, float beta2, float eps, void* stream) {
    if (!h || !h->train) return TTS_E_ARG;
    DEV_GUARD(h);
    TtsTrain* t = h->train;
    ++t->step;
    const float bc1 = 1.f - std::pow(beta1, (float)t->step), bc2 = 1.f - std::pow(beta2, (float)t->step);
    const long n4 = (long)(t->n / 4), per = (n4 + t->world - 1) / t->world;
    const long lo4 = std::min(n4, per * t->rank), hi4 = std::min(n4, lo4 + per);
    PeerPtrs pp = t->peers;
    if (t->world == 1) { pp.P[0] = t->P; pp.G[0] = t->G; }
    // local buffer first: the kernel reads the old parameter from P[0]
    std::swap(pp.P[0], pp.P[t->rank]);
    adam_peer_kernel<<<1184, 256, 0, (cudaStream_t)stream>>>(pp, t->world, t->M1, t->V2, lo4, hi4, lr, beta1, beta2, eps, bc1, bc2, 1.f / (float)t->world);
    ++launch_counter();
    CK(cudaGetLastError());
    return 0;
}
extern "C" int tts_train_repack(TtsHandle* h, void* stream) {
    if (!h || !h->train) return TTS_E_ARG;
    DEV_GUARD(h);
    return train_repack(h, (cudaStream_t)stream);
}
extern "C" int tts_train_num_tensors(TtsHandle* h) { return (h && h->train) ? (int)(h->train->params.size() + h->train->buffers.size()) : -1; }
extern "C" int tts_train_tensor_info(TtsHandle* h, int index, const char** name, int64_t* offset, int64_t* numel, int* is_buffer) {
    if (!h || !h->train || !name || !offset || !numel || !is_buffer || index < 0) return TTS_E_ARG;
    TtsTrain* t = h->train;
    const int np = (int)t->params.size();
    if (index >= np + (int)t->buffers.size()) return TTS_E_ARG;
    const TrEntry& e = index < np ? t->params[index] : t->buffers[index - np];
    *name = e.name.c_str(); *offset = (int64_t)e.off; *numel = (int64_t)e.numel; *is_buffer = index >= np;
    return 0;
}
extern "C" int tts_train_read(TtsHandle* h, int which, int64_t offset, int64_t numel, float* host_out) {
    if (!h || !h->train || !host_out || offset < 0 || numel <= 0) return TTS_E_ARG;
    TtsTrain* t = h->train;
    const float* src = which == 0 ? t->P : which == 1 ? t->G : which == 2 ? t->RS : nullptr;
    const size_t lim = which == 2 ? t->nrs : t->n;
    if (!src || (size_t)(offset + numel) > lim) return TTS_E_ARG;
    DEV_GUARD(h);
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(host_out, src + offset, (size_t)numel * 4, cudaMemcpyDeviceToHost));
    return 0;
}
