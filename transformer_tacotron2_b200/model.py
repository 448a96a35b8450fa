"""B200 backend of the Transformer-TTS module API.

Same class name, method signatures and state_dict keys as the interface BASELINE.json `north_star`
defines (restated executable in oracle/transformer_tts.py:TransformerTTS; the reference repository
itself ships no code, /root/reference/README.md:1-3).  All arithmetic happens in libtts_b200.so
(hand-written sm_100a kernels behind the C ABI of include/tts_b200.h); PyTorch is used for device
memory, streams and the nn.Module parameter container only.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, asdict
from typing import NamedTuple, Optional, Tuple

import torch
import torch.nn as nn

from . import _lib


@dataclass(frozen=True)
class TTSConfig:
    n_vocab: int = 128
    d_model: int = 512
    n_heads: int = 8
    n_enc_layers: int = 6
    n_dec_layers: int = 6
    d_ff: int = 2048
    n_mels: int = 80
    d_prenet: int = 256
    enc_conv_layers: int = 3
    conv_kernel: int = 5
    postnet_channels: int = 512
    postnet_layers: int = 5
    max_pos: int = 2048
    ln_eps: float = 1e-5
    bn_eps: float = 1e-5

    def to_dict(self):
        return asdict(self)


def postnet_halo(cfg: TTSConfig) -> int:
    """Frames on each side of a frame that the postnet's output there depends on (each conv layer reaches kernel // 2)."""
    return cfg.postnet_layers * (cfg.conv_kernel // 2)


class StreamSchedule:
    """Decode / emit schedule of TransformerTTS.inference_stream(), kept apart from the device calls so that it can be checked
    without a GPU.  The first decode launch runs chunk_frames + halo steps, every later one chunk_frames.  After each status
    (frames decoded t_done; `ended` = every utterance stopped or max_len reached), after_status() returns the steps of the next
    launch (0: none) and the frame range to emit (None: nothing new).  The range ends at the frontier: t_done once the session
    has ended, else t_done - halo, since the postnet output of a later frame still depends on frames not decoded yet."""

    def __init__(self, chunk_frames: int, halo: int, max_len: int):
        if chunk_frames < 1:
            raise ValueError("chunk_frames must be >= 1")
        self.chunk, self.halo, self.max_len, self.emitted = int(chunk_frames), int(halo), int(max_len), 0

    def first_steps(self) -> int:
        return min(self.chunk + self.halo, self.max_len)

    def max_emit_frames(self) -> int:
        """Largest range after_status() returns: chunk + halo (the first, or the last after the session ends)."""
        return min(self.chunk + self.halo, self.max_len)

    def after_status(self, t_done: int, ended: bool):
        frontier = t_done if ended else max(0, t_done - self.halo)
        rng = (self.emitted, frontier) if frontier > self.emitted else None
        self.emitted = max(self.emitted, frontier)
        return (0 if ended else self.chunk), rng


class StreamChunk(NamedTuple):
    """Frames [start, start + n) of every utterance of a streamed batch."""
    start: int
    mel_after: torch.Tensor      # [B, n, 80] fp32, zero past each utterance's end
    stop_logits: torch.Tensor    # [B, n] fp32, zero past each utterance's end
    n_valid: torch.Tensor        # [B] int32: frames of utterance b inside the chunk
    finished: torch.Tensor       # [B] bool: utterance b has stopped (or reached its frame budget / max_len)


# ---- parameter containers: the state_dict layout of the module API -----------------------------
class _MHA(nn.Module):
    def __init__(self, d):
        super().__init__()
        self.wq, self.wk, self.wv, self.wo = (nn.Linear(d, d) for _ in range(4))


class _FFN(nn.Module):
    def __init__(self, d, f):
        super().__init__()
        self.w1, self.w2 = nn.Linear(d, f), nn.Linear(f, d)


class _EncLayer(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.self_attn = _MHA(c.d_model)
        self.norm1 = nn.LayerNorm(c.d_model, eps=c.ln_eps)
        self.ffn = _FFN(c.d_model, c.d_ff)
        self.norm2 = nn.LayerNorm(c.d_model, eps=c.ln_eps)


class _DecLayer(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.self_attn = _MHA(c.d_model)
        self.norm1 = nn.LayerNorm(c.d_model, eps=c.ln_eps)
        self.cross_attn = _MHA(c.d_model)
        self.norm2 = nn.LayerNorm(c.d_model, eps=c.ln_eps)
        self.ffn = _FFN(c.d_model, c.d_ff)
        self.norm3 = nn.LayerNorm(c.d_model, eps=c.ln_eps)


class _ConvBN(nn.Module):
    def __init__(self, cin, cout, k, eps):
        super().__init__()
        self.conv = nn.Conv1d(cin, cout, k, padding=(k - 1) // 2)
        self.bn = nn.BatchNorm1d(cout, eps=eps)


class _EncPrenet(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.embed = nn.Embedding(c.n_vocab, c.d_model, padding_idx=0)
        self.convs = nn.ModuleList(_ConvBN(c.d_model, c.d_model, c.conv_kernel, c.bn_eps) for _ in range(c.enc_conv_layers))
        self.proj = nn.Linear(c.d_model, c.d_model)


class _DecPrenet(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.fc1, self.fc2, self.proj = nn.Linear(c.n_mels, c.d_prenet), nn.Linear(c.d_prenet, c.d_prenet), nn.Linear(c.d_prenet, c.d_model)


class _Postnet(nn.Module):
    def __init__(self, c):
        super().__init__()
        ch = [c.n_mels] + [c.postnet_channels] * (c.postnet_layers - 1) + [c.n_mels]
        self.convs = nn.ModuleList(_ConvBN(ch[i], ch[i + 1], c.conv_kernel, c.bn_eps) for i in range(c.postnet_layers))


class _Stack(nn.Module):
    def __init__(self, layers):
        super().__init__()
        self.layers = nn.ModuleList(layers)


class _TrainForwardFn(torch.autograd.Function):
    """model.train(); out = model(...); loss(out).backward(): the library's train-mode forward and backward behind autograd.
    The module's parameters ride along as inputs so that autograd routes the flat gradient buffer back to them."""

    @staticmethod
    def forward(ctx, model, trainer, phonemes, phoneme_lens, mels, mel_lens, seed, utt_offset, *params):
        mb, ma, st = trainer.forward_only(phonemes, phoneme_lens, mels, mel_lens, seed, utt_offset)
        ctx.model, ctx.trainer = model, trainer
        ctx.names = [n for n, _ in model.named_parameters()]
        ctx.pinfo = [(p.shape, p.device, p.dtype) for p in params]
        T = mels.shape[1]
        ctx.mask = (torch.arange(T, device=mb.device)[None, :] < mel_lens.to(mb.device)[:, None]).to(torch.float32)
        return mb, ma, st

    @staticmethod
    def backward(ctx, g_mb, g_ma, g_st):
        tr = ctx.trainer
        mask = ctx.mask
        z = lambda g, ref: torch.zeros(ref, device=mask.device) if g is None else g                      # noqa: E731
        B, T = mask.shape
        tr.backward_from(z(g_mb, (B, T, 80)) * mask[..., None], z(g_ma, (B, T, 80)) * mask[..., None], z(g_st, (B, T)) * mask)
        grads = tr.grads()                                                                               # name -> host tensor
        out = [grads[n].to(dev, dt).view(shape) for n, (shape, dev, dt) in zip(ctx.names, ctx.pinfo)]
        return (None,) * 8 + tuple(out)


class TransformerTTS(nn.Module):
    """forward(): teacher-forced (eval-mode arithmetic); inference(): greedy AR over a KV cache.

    Parameters live on the host (the packed bf16 copies the kernels read are owned by the C handle);
    call `load_state_dict` then use the module -- weights are (re)packed lazily on first use."""

    def __init__(self, cfg: Optional[TTSConfig] = None, device: int = 0):
        super().__init__()
        self.cfg = c = cfg or TTSConfig()
        self.enc_prenet = _EncPrenet(c)
        self.enc_alpha = nn.Parameter(torch.ones(()))
        self.dec_alpha = nn.Parameter(torch.ones(()))
        self.encoder = _Stack(_EncLayer(c) for _ in range(c.n_enc_layers))
        self.dec_prenet = _DecPrenet(c)
        self.decoder = _Stack(_DecLayer(c) for _ in range(c.n_dec_layers))
        self.mel_linear = nn.Linear(c.d_model, c.n_mels)
        self.stop_linear = nn.Linear(c.d_model, 1)
        self.postnet = _Postnet(c)
        self._device_index = device
        self._lib = None
        self._handle = C.c_void_p()
        self._dirty = True
        self._host_stale = False         # a Trainer has stepped the device-side parameters; the module's copies are behind
        self._trainer = None             # weakref to the Trainer that owns the training state (training.py)
        self._ag_trainer = None          # Trainer behind the autograd bridge (train-mode forward), created on first use
        self._ag_version = None
        self._synced_version = None
        self.profile_events = False      # bench.py: CUDA-event time of the decode loop per inference()
        self.decode_ms = []
        self.emit_ms = []                # inference_stream(): CUDA-event time of every tts_decode_emit (with profile_events)
        self._ws = None
        self._ws_key = None
        self._ws_uses = 0                # calls of _workspace(): an open inference_stream() detects a call that took the workspace
        self.eval()

    # ------------------------------------------------------------------ plumbing
    def _ensure_handle(self):
        if self._lib is None:
            if not torch.cuda.is_available():
                raise RuntimeError("transformer_tacotron2_b200 needs a B200 (sm_100a) GPU; there is no CPU fallback")
            self._lib = _lib.load()
            c = self.cfg
            cc = _lib.TtsConfig(C.sizeof(_lib.TtsConfig), c.n_vocab, c.d_model, c.n_heads, c.n_enc_layers, c.n_dec_layers,
                                c.d_ff, c.n_mels, c.d_prenet, c.enc_conv_layers, c.conv_kernel, c.postnet_channels,
                                c.postnet_layers, c.max_pos, c.ln_eps, c.bn_eps)
            rc = self._lib.tts_create(C.byref(cc), self._device_index, C.byref(self._handle))
            if rc != 0:
                raise _lib.TtsError(f"tts_create failed ({rc}): no sm_100 device {self._device_index}?")
        return self._lib

    def _check(self, rc, what):
        _lib.check(self._lib, self._handle, rc, what)

    def load_state_dict(self, *a, **k):
        out = super().load_state_dict(*a, **k)
        self._dirty = True
        self._host_stale = False         # explicit weights win over un-exported training state
        return out

    def _param_version(self):
        """Sum of the in-place version counters of every parameter / buffer: changes whenever an optimiser, `copy_`,
        `fill_` ... touches the module's tensors, so stale packed weights are never used silently."""
        return sum(int(t._version) for t in self._raw_state_dict().values())

    def _raw_state_dict(self):
        return super().state_dict()

    def _pull_trained_state(self):
        """After Trainer.step() the parameters the optimiser moved live in the library's training buffers; bring them
        back into the module before anything reads the module's tensors (inference, forward, state_dict)."""
        if self._host_stale:
            tr = self._trainer() if self._trainer is not None else None
            if tr is None:
                raise RuntimeError("the Trainer that stepped this module is gone and its state was never exported "
                                   "(call Trainer.export_to_module() before dropping it)")
            tr.export_to_module()

    def state_dict(self, *a, **k):
        self._pull_trained_state()
        return super().state_dict(*a, **k)

    def set_option(self, key: str, value: int):
        lib = self._ensure_handle()
        self._check(lib.tts_set_option(self._handle, key.encode(), int(value)), "tts_set_option")

    def sync_weights(self):
        """Push the module's parameters through tts_load_weight / tts_finalize_weights."""
        lib = self._ensure_handle()
        self._pull_trained_state()
        if not self._dirty and self._synced_version == self._param_version():
            return
        for name, t in self._raw_state_dict().items():
            if not t.is_floating_point():
                continue                                  # num_batches_tracked
            t = t.detach().to("cpu", torch.float32).contiguous()
            self._check(lib.tts_load_weight(self._handle, name.encode(), C.c_void_p(t.data_ptr()), t.numel()), f"tts_load_weight({name})")
        self._check(lib.tts_finalize_weights(self._handle), "tts_finalize_weights")
        self._dirty = False
        self._synced_version = self._param_version()

    def _workspace(self, B, S, T):
        lib = self._ensure_handle()
        self._ws_uses += 1
        key = (B, S, T)
        if self._ws_key != key:
            n = lib.tts_workspace_bytes(self._handle, B, S, T)
            if n == 0:
                raise _lib.TtsError("tts_workspace_bytes returned 0 (bad shape)")
            self._ws = None
            self._ws = torch.empty(n, dtype=torch.uint8, device=self.device)
            self._ws_key = key
        return self._ws

    @property
    def device(self):
        return torch.device("cuda", self._device_index)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def __del__(self):
        try:
            if self._lib is not None and self._handle:
                self._lib.tts_destroy(self._handle)
        except Exception:
            pass

    def _stage_inputs(self, phonemes, phoneme_lens, mels=None, mel_lens=None):
        """The inputs a call has, on the module's device and contiguous: phonemes int64, lengths int32, mels fp32."""
        inputs = ((phonemes, torch.int64), (phoneme_lens, torch.int32), (mels, torch.float32), (mel_lens, torch.int32))
        return tuple(t.to(self.device, dt).contiguous() for t, dt in inputs if t is not None)

    @staticmethod
    def _utt_ids(utt_ids, B, utt_offset, contiguous=False):
        """-> (offset, ids or None).  A contiguous range of utterance ids is just the offset of utterance 0; any other ids come
        back as an int32 tensor, or raise ValueError with contiguous=True (the teacher-forced C entry points take the offset only)."""
        if utt_ids is None:
            return int(utt_offset), None
        ids = torch.as_tensor([int(v) for v in utt_ids], dtype=torch.int32)
        if ids.tolist() == list(range(int(ids[0]), int(ids[0]) + B)):
            return int(ids[0]), None
        if contiguous:
            raise ValueError("utt_ids must be a contiguous range (the C ABI takes the id of utterance 0)")
        return int(utt_offset), ids

    # ------------------------------------------------------------------ teacher-forced
    def forward(self, phonemes, phoneme_lens, mels, mel_lens, seed: int = 0, utt_ids=None, utt_offset: int = 0
                ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """phonemes [B,S] i64, phoneme_lens [B], mels [B,T,80] f32, mel_lens [B]
        -> mel_before [B,T,80], mel_after [B,T,80], stop_logits [B,T]  (on the GPU, zero past mel_lens)."""
        if self.training:
            return self._train_forward(phonemes, phoneme_lens, mels, mel_lens, seed,
                                       self._utt_ids(utt_ids, phonemes.shape[0], utt_offset, contiguous=True)[0])
        with torch.no_grad():
            return self._eval_forward(phonemes, phoneme_lens, mels, mel_lens, seed, utt_ids, utt_offset)

    def _teacher_forced_setup(self, phonemes, phoneme_lens, mels, mel_lens, utt_ids, utt_offset):
        """Set-up shared by tts_forward and tts_forward_align.  -> lib, workspace, staged (ph, pl, mels, mel_lens), (B, S, T),
        offset of utterance 0."""
        lib = self._ensure_handle()
        self.sync_weights()
        B, S = phonemes.shape
        T = mels.shape[1]
        inputs = self._stage_inputs(phonemes, phoneme_lens, mels, mel_lens)
        ws = self._workspace(B, S, T)
        return lib, ws, inputs, (B, S, T), self._utt_ids(utt_ids, B, utt_offset, contiguous=True)[0]

    def _eval_forward(self, phonemes, phoneme_lens, mels, mel_lens, seed, utt_ids, utt_offset):
        lib, ws, (ph, pl, m, ml), (B, S, T), u0 = self._teacher_forced_setup(phonemes, phoneme_lens, mels, mel_lens, utt_ids, utt_offset)
        dev = self.device
        mb = torch.empty(B, T, 80, device=dev); ma = torch.empty(B, T, 80, device=dev); st = torch.empty(B, T, device=dev)
        rc = lib.tts_forward(self._handle, ws.data_ptr(), ph.data_ptr(), pl.data_ptr(), m.data_ptr(), ml.data_ptr(), B, S, T,
                             int(seed), u0, mb.data_ptr(), ma.data_ptr(), st.data_ptr(), self._stream())
        self._check(rc, "tts_forward")
        return mb, ma, st

    # ------------------------------------------------------------------ cross-attention alignments / durations
    @torch.no_grad()
    def alignments(self, phonemes, phoneme_lens, mels, mel_lens, seed: int = 0, utt_ids=None, utt_offset: int = 0, layers=None
                   ) -> torch.Tensor:
        """Encoder-decoder attention of the teacher-forced forward (eval mode): [n_layers, B, 8, T, S] fp32, P[l, b, h, t, s] =
        softmax_s(q_t . k_s / 8) of decoder layer layers[l] (default: all six, ascending), zero at frames t >= mel_lens[b] and
        phonemes s >= phoneme_lens[b].  Same inputs as forward(); CUDA tensors in -> CUDA tensor out, CPU in -> CPU out.

        Alignments of a free-running (AR) output: `_, lens, _, mb = model.inference(ph, pl, ..., return_before=True)` then
        `model.alignments(ph, pl, mb, lens)` with the same seed -- the teacher-forced decoder then sees exactly the frames the
        AR decoder fed back (shifted right behind the zero go-frame, same prenet dropout masks)."""
        ls, mask = self._align_layers(layers)
        out = self._forward_align(phonemes, phoneme_lens, mels, mel_lens, seed, utt_ids, utt_offset, mask, -1, True, False)
        return out["align"] if phonemes.is_cuda else out["align"].cpu()

    @torch.no_grad()
    def durations(self, phonemes, phoneme_lens, mels, mel_lens, seed: int = 0, utt_ids=None, utt_offset: int = 0, layers=None,
                  head: Optional[int] = None) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """FastSpeech duration targets from the teacher-forced cross-attention (Ren et al., 2019, section 3.3; ESPnet's
        DurationCalculator), computed on the GPU without forming P in memory.
        -> durations [B, S] int32 (frames t < mel_lens[b] whose most-attended phoneme is s; sums to mel_lens[b]),
           head [B] int32 (layer * 8 + h used for utterance b: the one with the largest focus rate among `layers`, lowest index
           on ties, unless `head` = layer * 8 + h fixes it), focus [6, B, 8] fp32 (focus rate = mean over valid frames of
           max_s P; -1 for layers not selected)."""
        ls, mask = self._align_layers(layers)
        fixed = -1 if head is None else int(head)
        if fixed != -1 and not (0 <= fixed < 48 and fixed // 8 in ls):
            raise ValueError("head must be layer * 8 + h of a selected layer")
        out = self._forward_align(phonemes, phoneme_lens, mels, mel_lens, seed, utt_ids, utt_offset, mask, fixed, False, True)
        res = (out["durations"], out["head"], out["focus"])
        return res if phonemes.is_cuda else tuple(t.cpu() for t in res)

    @staticmethod
    def _align_layers(layers):
        ls = list(range(6)) if layers is None else sorted({int(v) for v in layers})
        if not ls or ls[0] < 0 or ls[-1] > 5:
            raise ValueError("layers must be decoder layer indices in 0..5")
        return ls, sum(1 << v for v in ls)

    def _forward_align(self, phonemes, phoneme_lens, mels, mel_lens, seed, utt_ids, utt_offset, layer_mask, fixed_head,
                       want_align, want_durations):
        if self.training:
            raise RuntimeError("alignments() / durations() are eval-mode paths: call model.eval() first")
        lib, ws, (ph, pl, m, ml), (B, S, T), u0 = self._teacher_forced_setup(phonemes, phoneme_lens, mels, mel_lens, utt_ids, utt_offset)
        dev = self.device
        out, scratch = {}, None
        if want_align:
            out["align"] = torch.empty(bin(layer_mask).count("1"), B, 8, T, S, device=dev)
        if want_durations:
            scratch = torch.empty(lib.tts_align_scratch_bytes(self._handle, B, S, T), dtype=torch.uint8, device=dev)
            out["durations"] = torch.empty(B, S, dtype=torch.int32, device=dev)
            out["head"] = torch.empty(B, dtype=torch.int32, device=dev)
            out["focus"] = torch.empty(6, B, 8, device=dev)
        ptr = lambda k: out[k].data_ptr() if k in out else None                                          # noqa: E731
        rc = lib.tts_forward_align(self._handle, ws.data_ptr(), scratch.data_ptr() if scratch is not None else None, ph.data_ptr(),
                                   pl.data_ptr(), m.data_ptr(), ml.data_ptr(), B, S, T, int(seed), u0,
                                   layer_mask, fixed_head, None, None, None, ptr("align"), ptr("focus"), ptr("durations"), ptr("head"),
                                   self._stream())
        self._check(rc, "tts_forward_align")
        return out

    def _train_forward(self, phonemes, phoneme_lens, mels, mel_lens, seed, utt_offset):
        """Train-mode forward with autograd: `model.train(); out = model(...); loss_fn(*out).backward(); optimiser.step()` works on
        the module exactly as on the oracle (oracle/transformer_tts.py: forward in .train() mode).  Arithmetic: the library's
        training forward / backward (tts_train_forward / tts_train_backward); gradients are copied into the (host) parameters'
        .grad.  This is the compatibility path -- transformer_tacotron2_b200.training.Trainer keeps parameters, gradients and
        the optimiser on the device and is the fast one."""
        from .training import Trainer
        with torch.no_grad():
            tr = self._ag_trainer
            if tr is None:
                tr = self._ag_trainer = Trainer(self)
                self._ag_version = self._param_version()
            elif self._ag_version != self._param_version():          # an optimiser (or the user) changed the module's tensors
                tr.write_parameters(self._raw_state_dict())
                self._ag_version = self._param_version()
        out = _TrainForwardFn.apply(self, tr, phonemes, phoneme_lens, mels, mel_lens, int(seed), int(utt_offset), *list(self.parameters()))
        with torch.no_grad():                                        # BatchNorm running statistics moved in the forward: mirror them
            sd = self._raw_state_dict()
            for k, v in tr.buffers().items():
                sd[k].copy_(v)
            self._ag_version = self._param_version()
            self._dirty = True                                       # the packed inference weights fold the old statistics
        return out

    # ------------------------------------------------------------------ greedy AR
    def _start_decode(self, ws, ph, pl, max_len, seed, utt_offset, ids, max_lens, work_stealing, stream):
        """Opens a decode session in `ws` and encodes the batch: tts_decode_begin, tts_decode_set_batch when there are per-utterance
        ids or frame budgets (device int32 tensors or None), tts_encode."""
        lib, h, wsp = self._lib, self._handle, ws.data_ptr()
        B, S = ph.shape
        self._check(lib.tts_decode_begin(h, wsp, B, S, max_len, int(seed), utt_offset, stream), "tts_decode_begin")
        if ids is not None or max_lens is not None:
            ptr = lambda t: None if t is None else t.data_ptr()                                           # noqa: E731
            self._check(lib.tts_decode_set_batch(h, wsp, ptr(ids), ptr(max_lens), int(work_stealing), stream), "tts_decode_set_batch")
        self._check(lib.tts_encode(h, wsp, ph.data_ptr(), pl.data_ptr(), B, S, max_len, None, stream), "tts_encode")

    @torch.no_grad()
    def inference(self, phonemes, phoneme_lens, max_len: int = 800, seed: int = 0, utt_ids=None, utt_offset: int = 0,
                  return_before: bool = False, clone_outputs: bool = True, max_lens=None, sort_by_length: bool = False,
                  work_stealing: Optional[bool] = None):
        """-> mel_after [B,Tout,80], mel_lens [B] i32, stop_logits [B,Tout].

        CPU tensors in -> the whole call runs through tts_infer_host (H2D, encoder, decode loop,
        postnet, D2H) and CPU tensors come back.  CUDA tensors in -> device-resident pipeline
        (tts_encode / tts_decode_* ), CUDA tensors out.

        Host path: results are read back into pinned staging buffers the module keeps per (B, max_len).  With
        clone_outputs=True (default) private copies are returned; clone_outputs=False returns views of the staging buffers,
        valid until the next host-path call with the same shape (serving loops that consume the mel right away).

        Ragged batches (SURVEY.md 8(f)-2/3): `utt_ids` may be ANY ids (they key the dropout masks, so an utterance's result does
        not depend on its position in the batch); `max_lens` [B] gives every utterance its own frame budget (it stops there at
        the latest); `sort_by_length=True` decodes the batch sorted by budget / phoneme length, so that the utterances sharing
        a cluster group stop together, and returns the results in the caller's order -- bit-identical to the unsorted call;
        `work_stealing` lets a cluster whose group has stopped take the next group from a device-side queue (default: on
        whenever max_lens or sort_by_length is used)."""
        lib = self._ensure_handle()
        self.sync_weights()
        B, S = phonemes.shape
        u0, ids = self._utt_ids(utt_ids, B, utt_offset)
        ragged = ids is not None or max_lens is not None or sort_by_length
        ws = self._workspace(B, S, max_len)
        if not phonemes.is_cuda and not return_before and not ragged:
            ph = phonemes.to(torch.int64).contiguous()
            pl = phoneme_lens.to(torch.int32).contiguous()
            key = (B, int(max_len))
            if getattr(self, "_host_out_key", None) != key:
                self._host_out = (torch.empty(B, max_len, 80).pin_memory(), torch.empty(B, max_len).pin_memory(),
                                  torch.empty(B, dtype=torch.int32).pin_memory())
                self._host_out_key = key
            ma, st, ml = self._host_out
            tout = C.c_int(0)
            rc = lib.tts_infer_host(self._handle, ws.data_ptr(), ph.data_ptr(), pl.data_ptr(), B, S, int(max_len), int(seed), u0,
                                    ma.data_ptr(), ml.data_ptr(), st.data_ptr(), C.byref(tout), self._stream())
            self._check(rc, "tts_infer_host")
            T = tout.value
            out = (ma.view(-1)[: B * T * 80].view(B, T, 80), ml, st.view(-1)[: B * T].view(B, T))
            return tuple(t.clone() for t in out) if clone_outputs else out
        dev = self.device
        to_host = not phonemes.is_cuda
        ph, pl = self._stage_inputs(phonemes, phoneme_lens)
        perm = inv = None
        mlens_d = None if max_lens is None else torch.as_tensor(max_lens).to(dev, torch.int32).clamp(1, int(max_len)).contiguous()
        ids_d = None if ids is None else ids.to(dev)
        if sort_by_length:
            keyv = (mlens_d if mlens_d is not None else pl).to(torch.int64)
            perm = torch.argsort(keyv, descending=True, stable=True)
            inv = torch.empty_like(perm); inv[perm] = torch.arange(B, device=dev)
            if ids_d is None:
                ids_d = torch.arange(u0, u0 + B, device=dev, dtype=torch.int32)
            ph, pl, ids_d = ph[perm].contiguous(), pl[perm].contiguous(), ids_d[perm].contiguous()
            if mlens_d is not None:
                mlens_d = mlens_d[perm].contiguous()
        stream = self._stream()
        # a ragged batch always has ids_d or mlens_d here; work stealing is on for it unless the caller says otherwise
        self._start_decode(ws, ph, pl, int(max_len), seed, u0, ids_d, mlens_d, work_stealing is None or bool(work_stealing), stream)
        td, nf = C.c_int(0), C.c_int(0)
        chunk = int(max_len)                               # one launch: every cluster stops itself on the device
        if self.profile_events:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(torch.cuda.current_stream(dev))
        while True:
            self._check(lib.tts_decode_steps(self._handle, ws.data_ptr(), chunk, stream), "tts_decode_steps")
            if self.profile_events:
                ev1.record(torch.cuda.current_stream(dev))
            self._check(lib.tts_decode_status(self._handle, ws.data_ptr(), C.byref(td), C.byref(nf), stream), "tts_decode_status")
            if nf.value >= B or td.value >= max_len:
                break
        if self.profile_events:
            self.decode_ms.append(ev0.elapsed_time(ev1))
        T = td.value
        ma = torch.empty(B, T, 80, device=dev); st = torch.empty(B, T, device=dev)
        ml = torch.empty(B, dtype=torch.int32, device=dev)
        mb = torch.empty(B, T, 80, device=dev) if return_before else None
        rc = lib.tts_decode_end(self._handle, ws.data_ptr(), T, ma.data_ptr(), ml.data_ptr(), st.data_ptr(),
                                mb.data_ptr() if return_before else None, stream)
        self._check(rc, "tts_decode_end")
        out = (ma, ml, st, mb) if return_before else (ma, ml, st)
        if inv is not None:
            out = tuple(t[inv] for t in out)
        if to_host:
            out = tuple(t.cpu() for t in out)
        return out

    @torch.no_grad()
    def inference_stream(self, phonemes, phoneme_lens, max_len: int = 800, seed: int = 0, chunk_frames: int = 50, utt_ids=None,
                         utt_offset: int = 0, max_lens=None):
        """Greedy AR like inference(), yielding StreamChunk(start, mel_after, stop_logits, n_valid, finished) while the decoder keeps
        running.  The chunks cover consecutive frame ranges; concatenated along time they are exactly inference()'s mel_after and
        stop_logits, and their n_valid sum to its mel_lens.  CUDA inputs give CUDA chunks (ready when yielded), CPU inputs CPU chunks.

        A frame's postnet output is final once the `halo` (10) frames after it are decoded or its utterance has stopped, so the
        first chunk comes after chunk_frames + 10 decoder steps and each later one after chunk_frames more.  The decoder runs one
        chunk ahead: the next decode launch is queued on the current stream before the postnet window of the current chunk runs on
        a side stream, on the SMs the decode kernel leaves idle.  `utt_ids` / `max_lens` as in inference() (no sorting, no work
        stealing).  Closing the generator early leaves the module ready for the next call.

        The stream's decode session lives in the module's workspace until the generator is exhausted or closed.  Any other call
        on the module that runs in between (inference(), forward(), alignments(), encode(), another stream) takes that workspace
        over; the open generator then raises RuntimeError on its next step instead of yielding frames of the other call.  Serve
        concurrent requests from one module by batching them, or give each open stream its own module."""
        lib = self._ensure_handle()
        self.sync_weights()
        B, S = phonemes.shape
        max_len = int(max_len)
        u0, ids = self._utt_ids(utt_ids, B, utt_offset)
        sched = StreamSchedule(chunk_frames, postnet_halo(self.cfg), max_len)
        dev = self.device
        to_host = not phonemes.is_cuda
        ph, pl = self._stage_inputs(phonemes, phoneme_lens)
        mlens_d = None if max_lens is None else torch.as_tensor(max_lens).to(dev, torch.int32).clamp(1, max_len).contiguous()
        ids_d = None if ids is None else ids.to(dev)
        ws = self._workspace(B, S, max_len)
        ws_use = self._ws_uses
        if getattr(self, "_side_stream", None) is None:
            self._side_stream = torch.cuda.Stream(dev)
        side, cur = self._side_stream, torch.cuda.current_stream(dev)
        stream, side_ptr = self._stream(), C.c_void_p(side.cuda_stream)
        h, wsp = self._handle, ws.data_ptr()
        self._start_decode(ws, ph, pl, max_len, seed, u0, ids_d, mlens_d, False, stream)
        nbytes = lib.tts_stream_scratch_bytes(h, B, sched.max_emit_frames())
        with torch.cuda.stream(side):
            scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        self._check(lib.tts_decode_steps(h, wsp, sched.first_steps(), stream), "tts_decode_steps")
        td, nf = C.c_int(0), C.c_int(0)
        while True:
            if self._ws_uses != ws_use:
                raise RuntimeError("inference_stream(): another call on this module took its workspace and decode session "
                                   "between two chunks; the stream cannot continue")
            self._check(lib.tts_decode_status(h, wsp, C.byref(td), C.byref(nf), stream), "tts_decode_status")
            ended = nf.value >= B or td.value >= max_len
            steps, rng = sched.after_status(td.value, ended)
            if steps:                                      # decode chunk k + 1 is queued before the postnet of chunk k
                self._check(lib.tts_decode_steps(h, wsp, steps, stream), "tts_decode_steps")
            if rng is not None:
                t0, t1 = rng
                n = t1 - t0
                with torch.cuda.stream(side):
                    ma = torch.empty(B, n, 80, device=dev); st = torch.empty(B, n, device=dev)
                    ln = torch.empty(B, dtype=torch.int32, device=dev)
                    if self.profile_events:
                        ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                        ev[0].record(side)
                    self._check(lib.tts_decode_emit(h, wsp, scratch.data_ptr(), nbytes, t0, t1, ma.data_ptr(), st.data_ptr(),
                                                    ln.data_ptr(), None, side_ptr), "tts_decode_emit")
                    if self.profile_events:
                        ev[1].record(side)
                    fin = ln >= 0
                    nv = torch.where(fin, (ln - t0).clamp(0, n), torch.full_like(ln, n))
                    out = (ma, st, nv, fin)
                    if to_host:                            # copied on the side stream: the next decode launch keeps running
                        out = tuple(t.cpu() for t in out)
                side.synchronize()
                if self.profile_events:
                    self.emit_ms.append(ev[0].elapsed_time(ev[1]))
                if not to_host:
                    for t in out:                          # allocated on the side stream, consumed on the caller's
                        t.record_stream(cur)
                yield StreamChunk(t0, *out)
            if ended:
                return

    def phase_timestamps(self, n_steps: int) -> torch.Tensor:
        """[n_steps, n_phases] int64 ns stamps of the last persistent decode (option decode_timestamps = 1)."""
        out = torch.zeros(n_steps + 1, 128, dtype=torch.int64)     # last row: fine-grained debug stamps
        n = self._lib.tts_debug_phase_timestamps(self._handle, self._ws.data_ptr(), out.data_ptr(), n_steps, self._stream())
        if n <= 0:
            raise _lib.TtsError(f"tts_debug_phase_timestamps failed ({n})")
        self.debug_stamps = out[n_steps].clone()
        self.all_stamps = out[:n_steps].clone()            # incl. ad-hoc profiling columns 52..63
        return out[:n_steps, :n].clone()

    @torch.no_grad()
    def encode(self, phonemes, phoneme_lens, T: Optional[int] = None) -> torch.Tensor:
        """Encoder output ("memory") [B,S,512] fp32 on the GPU (bf16 values widened)."""
        lib = self._ensure_handle()
        self.sync_weights()
        dev = self.device
        B, S = phonemes.shape
        T = int(T or S)
        ws = self._workspace(B, S, T)
        ph, pl = self._stage_inputs(phonemes, phoneme_lens)
        mem = torch.empty(B, S, 512, device=dev)
        self._check(lib.tts_encode(self._handle, ws.data_ptr(), ph.data_ptr(), pl.data_ptr(), B, S, T, mem.data_ptr(), self._stream()), "tts_encode")
        return mem
