"""The fused chromosome step: both strands of one chromosome through the gated GCN, loss,
backward -- one C-ABI call (`cgcn_train_step`) on a strand-interleaved `[n, 2, d]` panel.

Reference: the body of the chromosome loop, finetune.py:30-53.  What differs by design:
  * `x_f` / `x_r` are processed together (every column index of the graph is read once per layer
    for both strands); BatchNorm statistics and running-stat updates stay per strand, in the
    reference's order (forward strand first);
  * parameters and gradients live in one flat buffer each (16-byte aligned slots) so the
    optimiser is one kernel and the data-parallel all-reduce is one NCCL call;
  * nothing is synchronised: the loss goes to a device slot, probabilities into a caller-provided
    device buffer.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional

import torch

from . import _lib, ops
from .chrome_models import ChromeGCN, call_buffers, model_struct
from .graph import HiCGraph

_SLOT = 64  # floats: every parameter starts on a 256-byte boundary inside the flat buffer


class FlatParams:
    """Re-homes a ChromeGCN's parameters (and their .grad) as views into two flat fp32 buffers.
    `ensure()` is cheap and idempotent; it re-flattens after `.cuda()`, `load_state_dict` or a
    `.data = ...` assignment (main.py:78-81 does the latter) moved a parameter elsewhere."""

    def __init__(self, model: ChromeGCN):
        self.model = model
        self.flat: Optional[torch.Tensor] = None
        self.flat_grad: Optional[torch.Tensor] = None
        self.offsets: Dict[str, int] = {}
        self.total = 0
        self._plist = None
        self._named = []
        self._views_cache: Dict = {}

    def _layout(self, params: Dict[str, torch.nn.Parameter], names: List[str]):
        off, offsets = 0, {}
        for k in names:
            offsets[k] = off
            off += (params[k].numel() + _SLOT - 1) // _SLOT * _SLOT
        return offsets, off

    def ensure(self, full: bool = True) -> "FlatParams":
        """`full=False` is the per-step fast path: only checks that the cached parameter objects still
        point into the flat buffer (a dozen `data_ptr()` calls)."""
        if not full and self.flat is not None and self._plist is not None:
            base = self.flat.data_ptr()
            if all(p.data_ptr() == base + 4 * off for p, off in self._plist):
                self.attach_grads()
                return self
        names = self.model._param_names()
        params = dict(self.model.named_parameters())
        dev = params[names[0]].device
        if dev.type != "cuda":
            raise _lib.ChromeGCNNativeError("ChromeGCN parameters must be on a CUDA device (no CPU fallback)")
        offsets, total = self._layout(params, names)
        ok = (self.flat is not None and self.flat.device == dev and total == self.total and
              all(params[k].data_ptr() == self.flat.data_ptr() + 4 * offsets[k] and params[k].dtype == torch.float32
                  for k in names))
        if not ok:
            flat = torch.zeros(total, dtype=torch.float32, device=dev)
            for k in names:
                p = params[k]
                view = flat[offsets[k]: offsets[k] + p.numel()].view(p.shape)
                view.copy_(p.data.to(torch.float32))
                p.data = view
            self.flat, self.offsets, self.total = flat, offsets, total
            self.flat_grad = torch.zeros(total, dtype=torch.float32, device=dev)
            self._views_cache = {}
        self._plist = [(params[k], offsets[k]) for k in names]
        self._named = [(k, params[k]) for k in names]
        self.attach_grads()
        return self

    def attach_grads(self) -> None:
        for k, p in self._named:
            off = self.offsets[k]
            if p.grad is None or p.grad.data_ptr() != self.flat_grad.data_ptr() + 4 * off:
                view = self.flat_grad[off: off + p.numel()].view(p.shape)
                if p.grad is not None and p.grad.shape == view.shape:
                    view.copy_(p.grad)           # gradients autograd produced through the module API
                p.grad = view

    def views(self, flat: torch.Tensor) -> Dict[str, torch.Tensor]:
        key = flat.data_ptr()
        v = self._views_cache.get(key)
        if v is None:
            v = {k: flat[self.offsets[k]: self.offsets[k] + p.numel()].view(p.shape) for k, p in self._named}
            self._views_cache[key] = v
        return v


def flat_params(model: ChromeGCN, full: bool = True) -> FlatParams:
    st = getattr(model, "_flat_state", None)
    if st is None:
        st = FlatParams(model)
        object.__setattr__(model, "_flat_state", st)
        full = True
    return st.ensure(full)


class ChromosomeEngine:
    """Owns the device buffers of the fused step and grows them to the largest chromosome seen."""

    def __init__(self, model: ChromeGCN, strands: int = 2):
        self.model = model
        self.strands = strands
        self._bufs: Dict[str, torch.Tensor] = {}
        self.step_count = 0

    def _buf(self, name: str, numel: int, dtype=torch.float32) -> torch.Tensor:
        t = self._bufs.get(name)
        dev = next(self.model.parameters()).device
        if t is None or t.numel() < numel or t.device != dev:
            t = torch.empty(max(numel, 1), dtype=dtype, device=dev)
            self._bufs[name] = t
        return t

    def panel(self, n: int, d: int) -> torch.Tensor:
        return self._buf("panel", n * self.strands * d)[: n * self.strands * d].view(n, self.strands, d)

    def pack(self, x_f: torch.Tensor, x_r: torch.Tensor) -> torch.Tensor:
        """[n, d] x 2 (device) -> the [n, 2, d] panel."""
        n, d = x_f.shape
        return ops.interleave_strands([x_f, x_r], out=self.panel(n, d))

    def call_buffers(self, n: int, out_grad: bool):
        """`chrome_models.call_buffers` for a call over `n` rows, served from this engine's cache."""
        return call_buffers(self.model, n, self.strands, self._buf, out_grad)

    def loss_workspace(self, n: int) -> torch.Tensor:
        """Workspace of `ops.bce_loss` for `n` rows, served from this engine's cache."""
        return self._buf("bce_ws", _lib.load().cgcn_bce_workspace_bytes(n, self.model.out.out_features) // 4 + 64)

    def run(self, graph: HiCGraph, panel: torch.Tensor, target: torch.Tensor, probs_out: Optional[torch.Tensor],
            loss_slot: torch.Tensor, train: bool, input_grad: Optional[torch.Tensor] = None):
        """One chromosome: forward (+ loss, + backward when `train`).  Gradients land in the model's flat
        gradient buffer (== every parameter's .grad).  Returns `(out [n, S, C] (a strided view), gates)` that stay
        valid until the next call."""
        lib = _lib.load()
        model = self.model
        fp = flat_params(model, full=False)
        n, nclass = panel.shape[0], model.out.out_features
        with torch.cuda.device(panel.device):
            ws, out, dout, gates = self.call_buffers(n, out_grad=train)
            m = model_struct(model, graph=graph, strands=self.strands, x_in=panel, x_in_grad=input_grad,
                             params=fp.views(fp.flat), grads=fp.views(fp.flat_grad) if train else None, out=out,
                             gates=gates, workspace=ws, dropout_counter=model._next_dropout_counter())
            if train:
                bits = target.dtype == torch.int32            # ops.pack_targets bit rows
                if bits:
                    if target.shape != (n, (nclass + 31) // 32):
                        raise ValueError("bit-packed targets must be [n, ceil(nclass/32)] int32")
                    tgt = target.contiguous()
                else:
                    tgt = ops._f32c(target)
                step_fn = lib.cgcn_train_step_bits if bits else lib.cgcn_train_step
                _lib.check(step_fn(C.byref(m), tgt.data_ptr(), _lib.ptr(probs_out), loss_slot.data_ptr(),
                                   dout.data_ptr()), "cgcn_train_step")
                fp.attach_grads()
            else:
                _lib.check(lib.cgcn_model_forward(C.byref(m)), "cgcn_model_forward")
                ops.bce_loss(out, target, self.strands, loss_slot, want_probs=False, want_grad=False, nclass=nclass,
                             probs_out=probs_out, workspace=self.loss_workspace(n))
        self.step_count += 1
        return out[:, :, :nclass], gates
