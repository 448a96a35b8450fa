/* tts_b200.h -- C ABI of libtts_b200.so: the B200-native (sm_100a) Transformer-TTS hot path.
 *
 * What this boundary replaces.  The reference repository (keonlee9420/Transformer-tacotron2)
 * ships NO code -- /root/reference/README.md:1-3 is its whole content (title, one sentence and
 * the link to Li et al., AAAI 2019 at README.md:3).  BASELINE.json `north_star` therefore defines
 * the interface to keep as a torch.nn.Module:
 *
 *     TransformerTTS.forward(phonemes, phoneme_lens, mels, mel_lens)   -> mel_before, mel_after, stop_logits
 *     TransformerTTS.inference(phonemes, phoneme_lens, max_len, seed)  -> mel_after, mel_lens, stop_logits
 *     + the training loop around them: model.train(); loss = tts_loss(model(...)); loss.backward(); all-reduce; Adam.step()
 *
 * (SURVEY.md section 8(b); restated executable in oracle/transformer_tts.py:TransformerTTS).  The entry
 * points below are exactly what a Python binding of those two methods calls (the ctypes stub is in
 * INTEGRATION.md and, live, in transformer_tacotron2_b200/_lib.py).  Each declaration cites the
 * interface it stands behind.
 *
 * Conventions: plain C types only; raw DEVICE pointers + explicit sizes + a cudaStream_t passed as
 * void*; the caller owns every buffer including the workspace (sized by tts_workspace_bytes); the
 * handle owns only the packed weights.  All work is enqueued on the caller's stream; calls marked
 * [sync] synchronise that stream.  Return value: 0 = ok, < 0 = argument error (TTS_E_*),
 * > 0 = cudaError_t.  tts_last_error_string() gives detail.  A handle is bound to one device and is
 * not thread-safe.  There is no CPU fallback: without an sm_100 device tts_create fails.
 */
#ifndef TTS_B200_H_
#define TTS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TTS_E_ARG (-1)       /* bad argument / shape */
#define TTS_E_STATE (-2)     /* call order (weights not finalised, decode not begun, ...) */
#define TTS_E_WEIGHT (-3)    /* unknown / missing / mis-sized weight */
#define TTS_E_DEVICE (-4)    /* no sm_100 device */

typedef struct TtsHandle TtsHandle;

/* oracle/transformer_tts.py:TTSConfig (SURVEY.md section 5 "Config / flags").  Only the base model
 * (d_model 512, 8 heads, d_ff 2048, 80 mels, prenet 256, kernel 5) is accepted. */
typedef struct TtsConfig {
    uint32_t struct_size;
    int32_t n_vocab, d_model, n_heads, n_enc_layers, n_dec_layers, d_ff, n_mels, d_prenet;
    int32_t enc_conv_layers, conv_kernel, postnet_channels, postnet_layers, max_pos;
    float ln_eps, bn_eps;
} TtsConfig;

/* ---- lifetime ------------------------------------------------------------------------------ */
/* TransformerTTS.__init__ (oracle/transformer_tts.py:TransformerTTS.__init__). */
int tts_create(const TtsConfig* cfg, int device, TtsHandle** out);
int tts_destroy(TtsHandle* h);
const char* tts_last_error_string(TtsHandle* h);
/* Library / build identification ("tts_b200 <version> sm_100a"). */
const char* tts_version(void);
/* Kernel launches issued by the library since it was loaded (bench.py: gpu_launches). */
unsigned long long tts_launch_count(void);

/* ---- weights: nn.Module.load_state_dict (same keys as the oracle's state_dict) --------------- */
/* Stage one fp32 tensor (HOST pointer, `numel` elements, C-contiguous) under its state_dict key. */
int tts_load_weight(TtsHandle* h, const char* name, const float* host_data, int64_t numel);
/* Pack everything staged so far: bf16 cast, BatchNorm folded into the convs (P5), Q/K/V and
 * [mel|stop] concatenated, decode-step weights swizzled into MMA fragment order; uploads. [sync] */
int tts_finalize_weights(TtsHandle* h);

/* ---- options ---------------------------------------------------------------------------------- */
/* "cluster_group": utterances per 8-CTA cluster of the decode kernel, 1..5 (0 = auto: as few as the number of
 *   co-resident clusters allows);  "decode_timestamps": 1 record per-phase timestamps (tts_debug_phase_timestamps);
 *   "decode_debug": 1 dump layer-0 activations of the first step (tts_debug_read_dump);
 *   "train_graph": 1 (default) replay tts_train_step from a CUDA graph captured on the second step of a shape, 0 eager;
 *   "print_info": print device / cluster geometry to stderr. */
int tts_set_option(TtsHandle* h, const char* key, int64_t value);

/* ---- workspace ---------------------------------------------------------------------------------- */
/* Bytes of caller-owned device scratch (KV caches, activations) for batch B, S phonemes, T frames. */
size_t tts_workspace_bytes(TtsHandle* h, int B, int S, int T);

/* ---- TransformerTTS.inference (oracle/transformer_tts.py:TransformerTTS.inference) ---------- */
/* Encoder + hoisted cross-K/V projection.  phonemes [B][S] int64, phoneme_lens [B] int32 (device).
 * T = the frame count the workspace was sized for (max_len of the decode that follows).
 * memory_out: optional fp32 [B][S][512] copy of the encoder output (may be NULL). */
int tts_encode(TtsHandle* h, void* ws, const int64_t* phonemes, const int32_t* phoneme_lens,
               int B, int S, int T, float* memory_out, void* stream);
/* Reset the AR state (KV cache cursor, lengths, stop flags).  utt_offset = global id of utterance 0
 * (dropout masks are keyed by global utterance id so a sharded batch reproduces the unsharded one). */
int tts_decode_begin(TtsHandle* h, void* ws, int B, int S, int max_len, uint64_t seed, int utt_offset, void* stream);
/* Run up to n_steps decoder steps (stops early, on the device, once every utterance has fired). */
int tts_decode_steps(TtsHandle* h, void* ws, int n_steps, void* stream);
/* [sync] steps completed so far and number of finished utterances. */
int tts_decode_status(TtsHandle* h, void* ws, int* t_done, int* n_finished, void* stream);
/* Mask past the stop frame, run the postnet, add the residual.  T_out = t_done.  Outputs (device):
 * mel_after [B][T_out][80] f32, mel_lens [B] i32, stop_logits [B][T_out] f32, mel_before (optional). */
int tts_decode_end(TtsHandle* h, void* ws, int T_out, float* mel_after, int32_t* mel_lens,
                   float* stop_logits, float* mel_before, void* stream);
/* Streaming: postnet-refined frames of a running decode session, emitted while the decoder keeps going.
 * The postnet is eval-mode arithmetic with a receptive field of halo = postnet_layers * (conv_kernel / 2) = 10 frames per side, so
 * frame t is final once frame t + halo is decoded.  Every tts_decode_status fixes the frontier: the decoded frame count if every
 * utterance has stopped or max_len is reached, else that count - halo; tts_decode_steps does not move it.
 * Bytes of device scratch for tts_decode_emit calls of at most max_frames frames (window = max_frames + 2 * halo rows). */
size_t tts_stream_scratch_bytes(TtsHandle* h, int B, int max_frames);
/* mel_after / stop_logits of frames [t_begin, t_end) of every utterance of the running decode session, as tts_decode_end would
 * return them: compact [B][t_end - t_begin][80] / [B][t_end - t_begin] fp32, zero at t >= the utterance's length.  Optional:
 * mel_before (same layout) and mel_lens int32 [B] (the length of every utterance that had stopped by the last status, as
 * tts_decode_end's mel_lens; -1 for one still running).  t_end must not exceed the frontier; scratch holds scratch_bytes bytes,
 * at least what tts_stream_scratch_bytes gives for t_end - t_begin frames.  TTS_E_STATE without a session or before its first
 * status call, TTS_E_ARG for t_begin < 0, t_end <= t_begin, t_end past the frontier or a scratch too small, all before any launch.
 * May run on another stream concurrently with tts_decode_steps: it reads only frames below the frontier, writes only the scratch
 * and the outputs, and its GEMMs use only the SMs the decode kernel's clusters leave free.  One window kernel and five
 * postnet GEMM launches per call. */
int tts_decode_emit(TtsHandle* h, void* ws, void* scratch, size_t scratch_bytes, int t_begin, int t_end, float* mel_after,
                    float* stop_logits, int32_t* mel_lens, float* mel_before, void* stream);
/* The whole of .inference() with HOST buffers (pageable or pinned): H2D, encode, decode loop,
 * postnet, D2H.  Outputs are written compactly as [B][T_out]...; *T_out returns the frames run.
 * `ws` is device scratch of tts_workspace_bytes(B, S, max_len). [sync] */
int tts_infer_host(TtsHandle* h, void* ws, const int64_t* phonemes, const int32_t* phoneme_lens, int B, int S,
                   int max_len, uint64_t seed, int utt_offset, float* mel_after, int32_t* mel_lens,
                   float* stop_logits, int* T_out, void* stream);

/* ---- TransformerTTS.forward, eval mode (oracle/transformer_tts.py:TransformerTTS.forward) --- */
/* Teacher-forced forward.  Device pointers: phonemes [B][S] i64, lens i32, mels [B][T][80] f32,
 * outputs mel_before / mel_after [B][T][80] f32 and stop_logits [B][T] f32 (zero past mel_lens). */
int tts_forward(TtsHandle* h, void* ws, const int64_t* phonemes, const int32_t* phoneme_lens,
                const float* mels, const int32_t* mel_lens, int B, int S, int T, uint64_t seed, int utt_offset,
                float* mel_before, float* mel_after, float* stop_logits, void* stream);

/* ---- encoder-decoder attention alignments and phoneme durations (teacher-forced, eval mode) ----------------------------- */
/* Bytes of device scratch tts_forward_align needs for focus / durations / head: per-row statistics of the cross-attention,
 * rowmax fp32 + argmax int16 [6][B][H][T], and the focus rates fp32 [6][B][H]. */
size_t tts_align_scratch_bytes(TtsHandle* h, int B, int S, int T);
/* Teacher-forced eval forward, launch for launch tts_forward, plus the cross-attention P[b][h][t][s] = softmax_s(q_t . k_s / 8)
 * of the decoder layers in layer_mask (bit l = layer l, 1 .. 0x3f), computed from the same bf16 operands as the forward's
 * attention.  Keys s >= phoneme_lens[b] and rows t >= mel_lens[b] are zero.  Device pointers; every output may be NULL:
 *   mel_before / mel_after / stop_logits  as tts_forward; all three NULL skips the heads and the postnet (all or none);
 *   align      fp32 [popcount(layer_mask)][B][H][T][S], the selected layers in ascending order;
 *   focus      fp32 [6][B][H]: focus rate = mean over t < mel_lens[b] of max_s P (unselected layers -1);
 *   durations  int32 [B][S]: number of frames t < mel_lens[b] whose first-maximal key is s (sums to mel_lens[b] when
 *              phoneme_lens[b] >= 1), for the head head[b] (int32 [B], = layer * 8 + h): the one with the largest focus rate
 *              among the selected layers (ties: lowest index), or fixed_head if >= 0 (its layer must be selected).
 * scratch (tts_align_scratch_bytes) is needed when focus, durations or head is requested.  No host synchronisation. */
int tts_forward_align(TtsHandle* h, void* ws, void* scratch, const int64_t* phonemes, const int32_t* phoneme_lens,
                      const float* mels, const int32_t* mel_lens, int B, int S, int T, uint64_t seed, int utt_offset,
                      uint32_t layer_mask, int fixed_head, float* mel_before, float* mel_after, float* stop_logits,
                      float* align, float* focus, int32_t* durations, int32_t* head, void* stream);

/* Optional per-utterance controls of a decode session (between tts_decode_begin and the first tts_decode_steps; device int32 [B],
 * either may be NULL):
 *   utt_ids   global utterance id of every row = its dropout key (default utt_offset + row).  With ids the batch may be decoded in
 *             ANY order -- e.g. sorted by length so that the utterances of a cluster group stop together -- with bit-identical
 *             per-utterance results (SURVEY.md 8(f)-2);
 *   max_lens  per-utterance frame budget <= max_len: the utterance also stops (length = budget) when it is used up;
 *   work_stealing != 0: the clusters draw their utterance groups from a device-side queue instead of a static round-robin, so a
 *             cluster whose group has stopped immediately starts the next one (8(f)-3: continuous batching at group granularity). */
int tts_decode_set_batch(TtsHandle* h, void* ws, const int32_t* utt_ids, const int32_t* max_lens, int work_stealing, void* stream);

/* Forced ("step-locked") decoding: overwrite frame t (< frames decoded so far) of the session's mel_before buffer with
 * frames [B][80] fp32 (device memory).  The next tts_decode_steps() call resumes from frame t_done - 1, so writing frame
 * t_done - 1 between single-step calls feeds the decoder somebody else's trajectory (the parity tests feed the oracle's). */
int tts_decode_set_frame(TtsHandle* h, void* ws, int t, const float* frames, void* stream);
/* Read frame t of the session back: frames [B][80] fp32 (mel_before) and, if not NULL, stop_logits [B] (device memory). */
int tts_decode_get_frame(TtsHandle* h, void* ws, int t, float* frames, float* stop_logits, void* stream);

/* Profiling aid: with option "decode_timestamps" = 1 the persistent decode kernel stamps %globaltimer
 * after every phase; this copies [n_steps][n_phases] stamps (ns) to the host and returns n_phases. [sync] */
int tts_debug_phase_timestamps(TtsHandle* h, void* ws, unsigned long long* out, int n_steps, void* stream);
/* Debugging aid: with option "decode_debug" = 1 cluster 0 / CTA 0 of the decode kernel dumps the activations of the group's
 * rows after the prenet and after every sub-layer of decoder layer 0 at the first step of each launch (slots of 2560 floats,
 * see decode_cluster.cuh: dbg_dump); this copies `n` floats starting at float `offset` of that dump to the host. [sync] */
int tts_debug_read_dump(TtsHandle* h, void* ws, int64_t offset, int64_t n, float* out_host, void* stream);

/* Layout of the decode kernel's K/V cache (host arithmetic only, no device work): element index (0 .. 8191) of K[row][dim]
 * (which = 0) or V[row][dim] (which = 1) inside a 64-row cache block; row in [0, 64), dim in [0, 64).  -1 on bad arguments.
 * The layout is part of the kernel contract (a ring stage must be one contiguous copy, a V fragment one 16-byte load), so the
 * CPU test suite checks it without a GPU. */
int tts_debug_kv_index(int row, int dim, int which);
/* The decode kernel's weight stream (host arithmetic only): packs rows `rows[0 .. nrows)` (nrows a multiple of 16 * TW; -1 = zero
 * row) x k-pairs [kp_base, kp_base + KP) (32 columns each) of the fp32 matrix w[N][K] exactly as tts_finalize_weights does for one
 * segment of one rank -- per warp a contiguous run of [k-pair][tile] blocks of 1 KB in mma.m16n8k16 A-fragment order, bf16.
 * Writes nrows / 16 * KP KB to `out` (returns the byte count, or the count needed if out is NULL / too small; -1 on bad
 * arguments).  The CPU tests re-read the stream with the kernel's addressing. */
int64_t tts_debug_pack_segment(const float* w, int N, int K, const int32_t* rows, int nrows, int kp_base, int KP, int TW,
                               unsigned char* out, int64_t out_bytes);

/* ---- training step (oracle: TransformerTTS.forward in .train() mode + tts_loss + autograd + torch.optim.Adam;
 *      oracle/transformer_tts.py:forward, :tts_loss, :masked_batchnorm; SURVEY.md 8(a) a12, 8(e)) ---------------- */
/* Build the training state from the weights loaded so far: one flat fp32 parameter buffer (+ gradients, Adam
 * moments), BatchNorm running statistics, bf16 operand copies.  [sync] */
int tts_train_begin(TtsHandle* h);
int tts_train_end(TtsHandle* h);
size_t tts_train_workspace_bytes(TtsHandle* h, int B, int S, int T);
/* Train-mode forward (batch-statistics BatchNorm, Philox dropout at every site), loss, full backward.  All pointers
 * are DEVICE pointers.  Afterwards the gradient of every parameter is in the flat gradient buffer (tts_train_grads),
 * loss_out[0] holds the scalar loss, and BatchNorm running statistics have been updated. */
int tts_train_step(TtsHandle* h, void* workspace, const int64_t* phonemes, const int32_t* phoneme_lens, const float* mels,
                   const int32_t* mel_lens, int B, int S, int T, uint64_t seed, int utt_offset, double p_residual,
                   float pos_weight, float* loss_out, void* stream);
/* Forward outputs of the last tts_train_step ([B][T][80], [B][T][80], [B][T] fp32, device pointers, any may be null). */
int tts_train_outputs(TtsHandle* h, void* workspace, int B, int S, int T, float* mel_before, float* mel_after,
                      float* stop_logits, void* stream);
/* The flat fp32 gradient buffer (device pointer, numel): the data-parallel exchange is ONE all-reduce over it. */
int tts_train_grads(TtsHandle* h, float** grads_dev, int64_t* numel);
/* Adam over the flat buffers (g <- grad * grad_scale, e.g. 1 / world_size after a sum all-reduce), then refresh the
 * bf16 operand copies. */
int tts_train_adam(TtsHandle* h, float lr, float beta1, float beta2, float eps, float grad_scale, void* stream);
/* Data-parallel optimiser step fused with its collective (SURVEY.md 8(f)-1): CUDA-IPC handles (64 bytes each) of this rank's
 * flat parameter and gradient buffers; tts_train_set_peers maps every rank's buffers (handles_* = [world][64] bytes, in rank
 * order; world <= 8, one node).  tts_train_adam_peers then runs ONE kernel that, for this rank's 1/world shard, sums the
 * gradient over all ranks by NVLink peer loads (reduce-scatter), applies Adam with shard-local moments (ZeRO-1), and stores
 * the new parameters into every rank's buffer by peer stores (all-gather).  The caller brackets it with two cross-rank
 * barriers on the stream and calls tts_train_repack afterwards. */
int tts_train_ipc_handles(TtsHandle* h, void* handle_P_64, void* handle_G_64);
int tts_train_set_peers(TtsHandle* h, int rank, int world, const void* handles_P, const void* handles_G);
int tts_train_adam_peers(TtsHandle* h, float lr, float beta1, float beta2, float eps, void* stream);
int tts_train_repack(TtsHandle* h, void* stream);
/* Enumerate the tensors inside the flat buffers: state_dict name, offset, numel; is_buffer = 1 for running stats. */
int tts_train_num_tensors(TtsHandle* h);
int tts_train_tensor_info(TtsHandle* h, int index, const char** name, int64_t* offset, int64_t* numel, int* is_buffer);
/* Copy a range of the parameter (which = 0), gradient (1) or running-statistics (2) buffer to the host. [sync] */
int tts_train_read(TtsHandle* h, int which, int64_t offset, int64_t numel, float* host_out);
/* Overwrite a range of the parameter (which = 0) or running-statistics (2) buffer from the host; parameters take effect after
 * tts_train_repack() (which refreshes the bf16 operand copies). [sync] */
int tts_train_write(TtsHandle* h, int which, int64_t offset, int64_t numel, const float* host_in);

/* ---- autograd bridge (the module's train-mode forward(): oracle `model.train(); out = model(...); loss.backward()`) ----------
 * tts_train_forward: the train-mode forward of tts_train_step alone (batch-statistics BatchNorm, every dropout site on); the
 *   activations stay in the workspace, the outputs are read with tts_train_outputs().
 * tts_train_backward: back-propagates caller-supplied output gradients d_before [B][T][80], d_after [B][T][80], d_stop [B][T]
 *   (fp32, device memory: dLoss/d(mel_before), dLoss/d(mel_after), dLoss/d(stop_logits) of ANY loss) through that forward into the
 *   flat gradient buffer (tts_train_grads).  Same workspace, shape, seed, utt_offset and p_residual as the forward it follows. */
int tts_train_forward(TtsHandle* h, void* workspace, const int64_t* phonemes, const int32_t* phoneme_lens, const float* mels,
                      const int32_t* mel_lens, int B, int S, int T, uint64_t seed, int utt_offset, double p_residual, void* stream);
int tts_train_backward(TtsHandle* h, void* workspace, int B, int S, int T, int utt_offset, double p_residual,
                       const float* d_before, const float* d_after, const float* d_stop, void* stream);

/* ---- per-kernel entry points (tests/test_gpu_kernels.py; not part of the drop-in surface) ---- */
/* C[M][N] = act(A[M][K] . W[N][K]^T + bias) ; bf16 in, fp32 out; act 0 none / 1 relu / 2 tanh (tcgen05 kernel, gemm_tc.cuh). */
int tts_k_gemm(const void* A_bf16, const void* W_bf16, const float* bias, float* C, int M, int N, int K, int act, void* stream);
/* conv1d(k=5, pad=2) over [B][T][Cin] with W [5][Cout][Cin] bf16 -> fp32 [B][T][Cout]; rows t >= lens[b] zeroed. */
int tts_k_conv5(const void* X_bf16, const void* W_bf16, const float* bias, const int32_t* lens, float* Y,
                int B, int T, int Cin, int Cout, int act, void* stream);
/* Attention core: Q [B][Lq][H*64], K/V [B][Lk][H*64] bf16 -> O [B][Lq][H*64] bf16. */
int tts_k_attention(const void* Q, const void* K, const void* V, void* O, const int32_t* klens,
                    int B, int H, int Lq, int Lk, int causal, void* stream);
/* Attention core with the per-row log-sum-exp kept for the backward pass: lse [B][H][Lq] fp32 (log2 domain). */
int tts_k_attention_lse(const void* Q, const void* K, const void* V, void* O, float* lse, const int32_t* klens,
                        int B, int H, int Lq, int Lk, int causal, void* stream);
/* Attention backward (training path): Q/K/V/O/dO as above + lse -> dQ/dK/dV bf16 in the same layouts.
 * scratch: fp32 [B*Lq*H*64 + B*H*Lq] device buffer. */
int tts_k_attention_bwd(const void* Q, const void* K, const void* V, const void* O, const void* dO, const float* lse,
                        const int32_t* klens, void* dQ, void* dK, void* dV, float* scratch,
                        int B, int H, int Lq, int Lk, int causal, void* stream);
/* Cross-attention probabilities (align.cuh): Q [B][Lq][ldq] bf16 (head h at column 64 h), K [B][H][Lk][64] bf16 ->
 * P [B][H][Lq][Lk] fp32, rowmax [B][H][Lq] fp32 (max_s P), argmax [B][H][Lq] int16 (first key with the largest score; -1 for
 * rows t >= qlens[b] or with no valid key).  qlens / klens int32 [B] may be NULL (all valid); every output may be NULL. */
int tts_k_cross_align(const void* Q, int ldq, const void* K, const int32_t* qlens, const int32_t* klens,
                      int B, int H, int Lq, int Lk, float* P, float* rowmax, int16_t* argmax, void* stream);
/* LayerNorm over rows of 512: fp32 in -> bf16 out. */
int tts_k_layernorm(const float* X, const float* gamma, const float* beta, void* Y_bf16, int M, float eps, void* stream);
/* Keep-bits of a p = 0.5 dropout site: out[t][b][c] (uint8) for t < T, b < B, c < C. */
int tts_k_philox_bits(uint64_t seed, int site, int T, int B, int C, int utt_offset, uint8_t* out, void* stream);

/* Training-step kernels (tests/test_gpu_train_kernels.py), launched exactly as tts_train_step launches them.  Rows are
 * m = b * T + t, valid iff t < lens[b]; `seed` is a DEVICE pointer to the uint64 dropout seed; site < 0 disables dropout.
 * Weight gradient (tcgen05): dW[n][k * taps + tap] += sum_{b,t} dY[b*T+t][n] X[b*T+t+tap-taps/2][k] (zero outside each
 * utterance), dbias[n] += sum dY[.][n] when dbias is not null.  dY [nb*T][ldy], X [nb*T][ldx] bf16; taps 1 or 5. */
int tts_k_wgrad(const void* dY_bf16, int ldy, int Cout, const void* X_bf16, int ldx, int Cin, int taps, int T, int nb,
                float* dW, float* dbias, void* stream);
/* Input gradient: packs the fp32 weight W [N][K][taps] (torch layout) into the transposed, tap-reversed bf16 layout
 * [taps][round_up(K,128)][round_up(N,64)] in `scratch`, then out[m][k] = sum_tap sum_{n < Kdy} dY[m+taps/2-tap][n] W[n][k][tap]
 * (conv1d input gradient; columns n >= N of dY meet zero weights).  Exactly one of out_f32 / out_bf16 (row stride ldo). */
int tts_k_dgrad(const float* W, int N, int K, int taps, const void* dY_bf16, int ldy, int Kdy, int M, int T,
                float* out_f32, void* out_bf16, int ldo, void* scratch_bf16, void* stream);
/* Masked batch-statistics BatchNorm forward over x [B*T][C] fp32 (C % 4 == 0, C <= 512): stat [1024] <- (sums, centred
 * squares) over valid rows; y = mask * dropout_0.5(act(BN(x))) (act 0 none / 1 relu / 2 tanh) -> out16 (bf16, row
 * stride ldo) and / or out32 (fp32, stride C); running stats updated (momentum 0.1, unbiased) if run_mean / run_var given. */
int tts_k_bn_train_fwd(const float* x, int B, int T, int C, const int32_t* lens, float* stat, const float* gamma,
                       const float* beta, float eps, int act, int site, const uint64_t* seed, int utt_offset, void* out16,
                       int ldo, float* out32, float* run_mean, float* run_var, void* stream);
/* Its backward from dout (fp32, or bf16 if dout_bf16; row stride ldd): dgamma / dbeta (zero on entry) get the parameter
 * gradients, dx (bf16, row stride ldx) the input gradient, zero on padded rows. */
int tts_k_bn_train_bwd(const void* dout, int dout_bf16, int ldd, const float* x, int B, int T, int C, const int32_t* lens,
                       const float* stat, const float* gamma, const float* beta, float eps, int act, int site,
                       const uint64_t* seed, int utt_offset, float* dgamma, float* dbeta, void* dx_bf16, int ldx, void* stream);
/* LayerNorm(512) backward from dx [M][512] at pre-norm input ypre: dy32 (fp32), dsub16 = bf16(dy * keep * dscale) with the
 * word-dropout site's keep mask (keep iff word >= thresh; site < 0: plain copy); dgamma / dbeta += their sums. */
int tts_k_ln_bwd(const float* dx, const float* ypre, const float* gamma, float eps, int M, int T, float* dy32, void* dsub16_bf16,
                 int site, const uint64_t* seed, int utt_offset, uint32_t thresh, float dscale, float* dgamma, float* dbeta,
                 void* stream);
/* Loss P13 over [B][T][80] / [B][T]: loss[0], and its gradients wrt mel_before, mel_after, stop_logits; acc: 16 floats scratch. */
int tts_k_loss(const float* before, const float* after, const float* stop, const float* target, const int32_t* lens, int B,
               int T, float pos_weight, float* acc, float* dbefore, float* dafter, float* dstop, float* loss, void* stream);
/* Head gradient dhead [B*T][128] bf16: [0, 80) = mask * (dbefore + dafter + dpost0), [80] = mask * dstop, rest 0. */
int tts_k_head_grad(const float* dbefore, const float* dafter, const void* dpost0_bf16, int ldp, const float* dstop,
                    const int32_t* lens, int B, int T, void* dhead_bf16, void* stream);
/* Word-dropout backward of d [B*T][512] -> out (bf16) = d * keep * dscale, dalpha += sum out_fp32 * pe[t] (pe [T][512]);
 * decoder != 0 uses the decoder's launch (1184 blocks), 0 the encoder's (592). */
int tts_k_dropw_bwd(const float* d, void* out_bf16, int B, int T, int site, const uint64_t* seed, int utt_offset,
                    uint32_t thresh, float dscale, const float* pe, float* dalpha, int decoder, void* stream);
/* Embedding backward: dE[ph[m]][c] += d[m][c] over valid rows with 0 < ph[m] < V; d [B*S][512] bf16, dE [V][512]. */
int tts_k_embed_bwd(const void* d_bf16, const int64_t* ph, const int32_t* lens, int B, int S, int V, float* dE, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TTS_B200_H_ */
