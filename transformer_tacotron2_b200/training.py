"""Training step of the B200 path: the counterpart of

    model.train(); out = model(ph, pl, mels, ml, seed); loss = tts_loss(*out, mels, ml); loss.backward()
    (all-reduce of the gradients across data-parallel ranks); torch.optim.Adam(...).step()

on the oracle (oracle/transformer_tts.py: TransformerTTS.forward, tts_loss).  All arithmetic runs in libtts_b200.so
(tts_train_* in include/tts_b200.h); torch is used for device memory and for the data-parallel all-reduce over the
library's single flat gradient buffer (NCCL on GPUs; SURVEY.md 8(e): one exchange step, per-rank BatchNorm statistics)."""
from __future__ import annotations

import ctypes as C
import weakref
from typing import Dict, Optional, Tuple

import torch

from .model import TransformerTTS


def allreduce_sum_(flat: torch.Tensor, group=None) -> torch.Tensor:
    """The one exchange step of data-parallel training (SURVEY.md 8(e)): sum the flat gradient buffer over the ranks, in
    place (NCCL over NVLink / NVSwitch for CUDA tensors, gloo in the CPU tests).  The mean is taken inside the Adam kernel
    (grad_scale = 1 / world_size), so no extra pass over the 53 M gradients is made."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    return flat


class _DevBuf:
    """A device range exposed through __cuda_array_interface__ so that torch can wrap it without copying."""

    def __init__(self, ptr: int, numel: int):
        self.__cuda_array_interface__ = {"shape": (numel,), "typestr": "<f4", "data": (ptr, False), "version": 3, "strides": None}


class Trainer:
    def __init__(self, model: TransformerTTS, lr: float = 1e-3, betas: Tuple[float, float] = (0.9, 0.98), eps: float = 1e-9,
                 p_residual: float = 0.1, pos_weight: float = 5.0, process_group=None, world_size: int = 1, rank: int = 0,
                 fused_peer_adam: bool = True):
        self.model = model
        self.lr, self.betas, self.eps = float(lr), (float(betas[0]), float(betas[1])), float(eps)
        self.p_residual, self.pos_weight = float(p_residual), float(pos_weight)
        self.group, self.world_size = process_group, int(world_size)
        lib = model._ensure_handle()
        model.sync_weights()
        model._check(lib.tts_train_begin(model._handle), "tts_train_begin")
        self._lib, self._h = lib, model._handle
        model._trainer = weakref.ref(self)
        ptr, n = C.c_void_p(), C.c_int64()
        model._check(lib.tts_train_grads(self._h, C.byref(ptr), C.byref(n)), "tts_train_grads")
        self.flat_grads = torch.as_tensor(_DevBuf(ptr.value, n.value), device=model.device)      # view, no copy
        self._loss = torch.zeros(1, device=model.device)
        self._ws, self._ws_key = None, None
        self._table = []
        name, off, numel, isb = C.c_char_p(), C.c_int64(), C.c_int64(), C.c_int()
        for i in range(lib.tts_train_num_tensors(self._h)):
            model._check(lib.tts_train_tensor_info(self._h, i, C.byref(name), C.byref(off), C.byref(numel), C.byref(isb)), "tts_train_tensor_info")
            self._table.append((name.value.decode(), off.value, numel.value, bool(isb.value)))
        # Data parallel on one node: map every rank's parameter / gradient buffers through CUDA IPC so that the optimiser step
        # is ONE kernel doing reduce-scatter (peer loads) -> Adam on this rank's shard -> all-gather (peer stores) over NVLink.
        self.rank, self._peers = int(rank), False
        if self.world_size > 1 and fused_peer_adam:
            self._peers = self._map_peers()
        self._tick = torch.zeros(1, device=model.device)

    def _map_peers(self) -> bool:
        import torch.distributed as dist
        hp, hg = C.create_string_buffer(64), C.create_string_buffer(64)
        self.model._check(self._lib.tts_train_ipc_handles(self._h, hp, hg), "tts_train_ipc_handles")
        gathered = [None] * self.world_size
        dist.all_gather_object(gathered, (self.rank, hp.raw, hg.raw), group=self.group)
        gathered.sort(key=lambda x: x[0])
        if [x[0] for x in gathered] != list(range(self.world_size)):
            raise ValueError(f"Trainer(rank=...) must be this process's rank in the group: got ranks {[x[0] for x in gathered]}")
        allp, allg = b"".join(x[1] for x in gathered), b"".join(x[2] for x in gathered)
        rc = self._lib.tts_train_set_peers(self._h, self.rank, self.world_size, allp, allg)
        ok = torch.tensor([1 if rc == 0 else 0], device=self.model.device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)              # all ranks take the same path
        return bool(int(ok.item()))

    def _stream_barrier(self):
        """Cross-rank barrier ordered on the CUDA stream (no host synchronisation): a 1-element all-reduce."""
        import torch.distributed as dist
        dist.all_reduce(self._tick, op=dist.ReduceOp.SUM, group=self.group)

    # ------------------------------------------------------------------ one step
    def _stage(self, phonemes, phoneme_lens, mels, mel_lens, sids=None, spembs=None):
        """Moves a batch to the device, into self._in (the library's asynchronous copies read from it), records its shape and
        returns the workspace for that shape.  A multi-speaker model's sids / spembs (as TransformerTTS.forward takes them) are
        staged into the workspace with tts_train_set_conditioning; the next training call consumes them."""
        B, S = phonemes.shape
        T = mels.shape[1]
        spk = self.model._speaker_inputs(sids, spembs, B)
        self._in = self.model._stage_inputs(phonemes, phoneme_lens, mels, mel_lens)
        if self._ws_key != (B, S, T):
            n = self._lib.tts_train_workspace_bytes(self._h, B, S, T)
            self._ws = None
            self._ws = torch.empty(n, dtype=torch.uint8, device=self.model.device)
            self._ws_key = (B, S, T)
        self._shape = (B, S, T)
        if spk is not None:
            ptr = lambda t: None if t is None else t.data_ptr()                                           # noqa: E731
            self.model._check(self._lib.tts_train_set_conditioning(self._h, self._ws.data_ptr(), B, ptr(spk[0]), ptr(spk[1]),
                                                                   self.model._stream()), "tts_train_set_conditioning")
        self._spk = spk
        return self._ws

    def forward_backward(self, phonemes, phoneme_lens, mels, mel_lens, seed: int = 0, utt_offset: int = 0, sids=None, spembs=None
                         ) -> torch.Tensor:
        """Train-mode forward + loss + backward.  Returns the loss (1-element device tensor); gradients are in flat_grads."""
        m = self.model
        ws = self._stage(phonemes, phoneme_lens, mels, mel_lens, sids, spembs)
        (ph, pl, me, ml), (B, S, T) = self._in, self._shape
        rc = self._lib.tts_train_step(self._h, ws.data_ptr(), ph.data_ptr(), pl.data_ptr(), me.data_ptr(), ml.data_ptr(), B, S, T, int(seed),
                                      int(utt_offset), self.p_residual, self.pos_weight, self._loss.data_ptr(), m._stream())
        m._check(rc, "tts_train_step")
        return self._loss

    # ------------------------------------------------------------------ autograd bridge (model.train(); model(...); loss.backward())
    def forward_only(self, phonemes, phoneme_lens, mels, mel_lens, seed: int = 0, utt_offset: int = 0, sids=None, spembs=None):
        """Train-mode forward alone; the activations stay in the workspace for backward_from().  -> (mel_before, mel_after, stop)."""
        m = self.model
        ws = self._stage(phonemes, phoneme_lens, mels, mel_lens, sids, spembs)
        (ph, pl, me, ml), (B, S, T) = self._in, self._shape
        rc = self._lib.tts_train_forward(self._h, ws.data_ptr(), ph.data_ptr(), pl.data_ptr(), me.data_ptr(), ml.data_ptr(), B, S, T, int(seed),
                                         int(utt_offset), self.p_residual, m._stream())
        m._check(rc, "tts_train_forward")
        self._fwd_args = (int(utt_offset),)
        return self.outputs()

    def backward_from(self, d_before, d_after, d_stop):
        """Back-propagate dLoss/d(mel_before), dLoss/d(mel_after), dLoss/d(stop_logits) of any loss through the last forward_only();
        the parameter gradients land in flat_grads."""
        m, dev = self.model, self.model.device
        B, S, T = self._shape
        g = [t.to(dev, torch.float32).contiguous() for t in (d_before, d_after, d_stop)]
        rc = self._lib.tts_train_backward(self._h, self._ws.data_ptr(), B, S, T, self._fwd_args[0], self.p_residual,
                                          g[0].data_ptr(), g[1].data_ptr(), g[2].data_ptr(), m._stream())
        m._check(rc, "tts_train_backward")
        torch.cuda.current_stream(dev).synchronize()           # g[] must outlive the copies

    def write_parameters(self, state: Dict[str, torch.Tensor]):
        """Overwrite the device-side parameters / BatchNorm statistics from host tensors keyed like state_dict(), then refresh the
        bf16 operand copies (the autograd bridge calls this after a torch optimiser stepped the module's parameters)."""
        flat_p, flat_b = None, None
        for name, off, numel, isb in self._table:
            t = state[name].detach().to("cpu", torch.float32).contiguous().view(-1)
            assert t.numel() == numel, name
            self.model._check(self._lib.tts_train_write(self._h, 2 if isb else 0, off, numel, C.c_void_p(t.data_ptr())), "tts_train_write")
        self.model._check(self._lib.tts_train_repack(self._h, self.model._stream()), "tts_train_repack")

    def all_reduce_grads(self):
        if self.world_size > 1:
            allreduce_sum_(self.flat_grads, self.group)

    def adam_step(self):
        rc = self._lib.tts_train_adam(self._h, self.lr, self.betas[0], self.betas[1], self.eps, 1.0 / self.world_size, self.model._stream())
        self.model._check(rc, "tts_train_adam")
        # The module's host copies are now behind the device-side parameters.  They are NOT re-staged from the host (that
        # would silently evaluate the un-trained weights): the next inference() / forward() / state_dict() on the module
        # pulls the trained state back first (TransformerTTS._pull_trained_state -> export_to_module).
        self.model._host_stale = True

    def adam_step_peers(self):
        """reduce-scatter + Adam + all-gather in one kernel over NVLink peer memory, bracketed by stream-ordered barriers."""
        m = self.model
        self._stream_barrier()                     # every rank's gradients are complete
        m._check(self._lib.tts_train_adam_peers(self._h, self.lr, self.betas[0], self.betas[1], self.eps, m._stream()), "tts_train_adam_peers")
        self._stream_barrier()                     # every shard of the new parameters has landed in every rank's buffer
        m._check(self._lib.tts_train_repack(self._h, m._stream()), "tts_train_repack")
        m._host_stale = True

    def step(self, phonemes, phoneme_lens, mels, mel_lens, seed: int = 0, utt_offset: int = 0, sids=None, spembs=None) -> torch.Tensor:
        loss = self.forward_backward(phonemes, phoneme_lens, mels, mel_lens, seed, utt_offset, sids, spembs)
        if self._peers:
            self.adam_step_peers()
        else:
            self.all_reduce_grads()
            self.adam_step()
        return loss

    # ------------------------------------------------------------------ inspection
    def outputs(self):
        B, S, T = self._shape
        dev = self.model.device
        mb, ma, st = torch.empty(B, T, 80, device=dev), torch.empty(B, T, 80, device=dev), torch.empty(B, T, device=dev)
        rc = self._lib.tts_train_outputs(self._h, self._ws.data_ptr(), B, S, T, mb.data_ptr(), ma.data_ptr(), st.data_ptr(), self.model._stream())
        self.model._check(rc, "tts_train_outputs")
        return mb, ma, st

    def _read(self, which: int) -> Dict[str, torch.Tensor]:
        shapes = {k: v.shape for k, v in self.model._raw_state_dict().items()}
        out = {}
        for name, off, numel, isb in self._table:
            if isb != (which == 2):
                continue
            t = torch.empty(numel, dtype=torch.float32)
            self.model._check(self._lib.tts_train_read(self._h, which, off, numel, C.c_void_p(t.data_ptr())), "tts_train_read")
            out[name] = t.view(shapes[name])
        return out

    def grads(self) -> Dict[str, torch.Tensor]:
        return self._read(1)

    def parameters(self) -> Dict[str, torch.Tensor]:
        return self._read(0)

    def buffers(self) -> Dict[str, torch.Tensor]:
        return self._read(2)

    def export_to_module(self):
        """Copy the trained parameters and BatchNorm statistics back into the nn.Module (for inference / state_dict())."""
        sd = self.model._raw_state_dict()
        with torch.no_grad():
            for k, v in {**self.parameters(), **self.buffers()}.items():
                sd[k].copy_(v)
        self.model._host_stale = False
        self.model._dirty = True
