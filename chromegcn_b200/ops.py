"""Thin tensor-level wrappers over the C ABI (one function per entry point of include/chromegcn.h).

Every function takes CUDA tensors, launches on torch's current stream and raises
`ChromeGCNNativeError` on failure.  PyTorch is used for memory and streams only.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from .graph import HiCGraph

GEMM_AUTO, GEMM_FFMA, GEMM_TCGEN05 = 0, 1, 2


def _f32c(t: torch.Tensor) -> torch.Tensor:
    if not t.is_cuda:
        raise _lib.ChromeGCNNativeError("expected a CUDA tensor (no CPU fallback)")
    if t.dtype != torch.float32:
        raise _lib.ChromeGCNNativeError("expected float32, got %s" % t.dtype)
    t = t.contiguous()
    if t.data_ptr() % 16 != 0:          # the kernels use 128-bit loads on every row / vector start
        t = t.clone()
    return t


def spmm(graph: HiCGraph, x: torch.Tensor, mean: bool = True, residual: Optional[torch.Tensor] = None,
         out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """`out[i] = (1/deg_i if mean else 1) * sum_{j in P_i} x[j] (+ residual[i])`; x is `[n, width]`."""
    lib = _lib.load()
    x = _f32c(x)
    n = graph.n
    width = x.numel() // n
    if out is None:
        out = torch.empty_like(x)
    res = _f32c(residual) if residual is not None else None
    g = graph.c_struct()
    with torch.cuda.device(x.device):
        _lib.check(lib.cgcn_spmm(C.byref(g), x.data_ptr(), out.data_ptr(), width, 1 if mean else 0,
                                 _lib.ptr(res), _lib.current_stream()), "cgcn_spmm")
    return out


def peer_panel(blocks: Sequence[int], row_begin: Sequence[int], rank: int) -> _lib.PeerPanel:
    """`cgcn_peer_panel` over `len(blocks)` exchange buffers given as device addresses."""
    world = len(blocks)
    if not 1 <= world <= _lib.MAX_PEERS or len(row_begin) != world + 1:
        raise _lib.ChromeGCNNativeError("peer_panel: world=%d (max %d)" % (world, _lib.MAX_PEERS))
    pp = _lib.PeerPanel()
    pp.world, pp.rank = world, rank
    for r in range(world):
        pp.base[r] = int(blocks[r])
        pp.row_begin[r] = int(row_begin[r])
    pp.row_begin[world] = int(row_begin[world])
    return pp


def spmm_peer(graph: HiCGraph, blocks: Sequence[torch.Tensor], rank: int, mean: bool = True,
              residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """`cgcn_spmm_peer`: `graph` holds the rows of block `rank` with global column indices; `blocks[r]` is the
    `[rows_r, width]` panel block rank r owns (tensors on this device, or peer-mapped memory)."""
    lib = _lib.load()
    blocks = [_f32c(b) for b in blocks]
    begins = [0]
    for b in blocks:
        begins.append(begins[-1] + b.shape[0])
    width = blocks[rank].numel() // max(blocks[rank].shape[0], 1)
    if out is None:
        out = torch.empty(graph.n, width, dtype=torch.float32, device=blocks[rank].device)
    res = _f32c(residual) if residual is not None else None
    g = graph.c_struct()
    pp = peer_panel([b.data_ptr() for b in blocks], begins, rank)
    with torch.cuda.device(out.device):
        _lib.check(lib.cgcn_spmm_peer(C.byref(g), C.byref(pp), out.data_ptr(), width, 1 if mean else 0, _lib.ptr(res),
                                      _lib.current_stream()), "cgcn_spmm_peer")
    return out


def _out(t: Optional[torch.Tensor], shape, device, more_rows: bool = False, align: int = 16) -> torch.Tensor:
    """Output buffer of a kernel: a new tensor, or the caller's, which the kernel writes in place (so it is checked, not
    copied like `_f32c` inputs; a view into a larger buffer is fine).  `more_rows`: the caller's tensor may have more
    rows than `shape` (per-CTA partials).  `align`: the byte alignment the kernel's stores need."""
    if t is None:
        return torch.empty(*shape, dtype=torch.float32, device=device)
    if not t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous() or t.data_ptr() % align != 0:
        raise _lib.ChromeGCNNativeError("output tensors must be contiguous, %d-byte aligned CUDA float32" % align)
    rows_ok = t.shape[0] >= shape[0] if more_rows else t.shape[0] == shape[0]
    if t.dim() != len(shape) or tuple(t.shape[1:]) != tuple(shape[1:]) or not rows_ok:
        raise _lib.ChromeGCNNativeError("output tensor of shape %s, need %s" % (tuple(t.shape), tuple(shape)))
    return t


def _max_layer_parts(n: int, strands: int, device) -> int:
    """Upper bound of the fused layer kernel's CTA count (= partial rows it writes): one CTA per 64-row panel tile, at
    most one per SM (fused_layer_grid)."""
    tiles = (n * strands + 63) // 64
    return max(1, min(tiles, torch.cuda.get_device_properties(device).multi_processor_count))


def gcn_layer_fwd(graph: HiCGraph, x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, gate_w: Optional[torch.Tensor],
                  gate_b: Optional[torch.Tensor], gate_off: bool = False, dropout_p: float = 0.0, seed: int = 0, step: int = 0,
                  site: int = 0, with_stats: bool = False, x_gather: Optional[torch.Tensor] = None,
                  x_out: Optional[torch.Tensor] = None, z_out: Optional[torch.Tensor] = None,
                  gate_out: Optional[torch.Tensor] = None, sx_out: Optional[torch.Tensor] = None,
                  stats_out: Optional[torch.Tensor] = None):
    """One gated GCN layer (models/ChromeModels.py:37-40) as one fused kernel (cgcn_gcn_layer_fwd).  `x` is
    `[n, 128]` or the strand-interleaved `[n, S, 128]`.  Returns `(x_out, z, gate, sx, stats)`; `stats` is the
    `[parts, 2*S*128]` per-CTA column sums of relu(x_out), relu(x_out)^2 (None unless `with_stats`).  The `*_out`
    tensors, when given, receive the results (`stats_out`: at least as many rows as the kernel has CTAs)."""
    lib = _lib.load()
    x = _f32c(x)
    n = graph.n
    S = x.shape[1] if x.dim() == 3 else 1
    dev = x.device
    xg = x if x_gather is None else _f32c(x_gather)
    sx, z, xo = _out(sx_out, x.shape, dev), _out(z_out, x.shape, dev), _out(x_out, x.shape, dev)
    gate = _out(gate_out, (n, S), dev)
    stats = _out(stats_out, (_max_layer_parts(n, S, dev), 2 * S * 128), dev, more_rows=True) if with_stats else None
    parts = C.c_int32(0)
    gs = graph.c_struct()
    with torch.cuda.device(dev):
        _lib.check(lib.cgcn_gcn_layer_fwd(C.byref(gs), S, xg.data_ptr(), x.data_ptr(), _f32c(weight).data_ptr(),
                                          _f32c(bias).data_ptr(), _lib.ptr(None if gate_w is None else _f32c(gate_w)),
                                          _lib.ptr(None if gate_b is None else _f32c(gate_b)), 1 if gate_off else 0,
                                          float(dropout_p), seed, step, site, sx.data_ptr(), z.data_ptr(), xo.data_ptr(),
                                          gate.data_ptr(), _lib.ptr(stats), C.byref(parts), _lib.current_stream()),
                   "cgcn_gcn_layer_fwd")
    return xo, z, gate, sx, (stats[: parts.value] if with_stats else None)


_NEW = object()          # gcn_layer_bwd(dxd_out=...) default: a new panel


def gcn_layer_bwd(graph: HiCGraph, dys_gather: torch.Tensor, dxd: torch.Tensor, weight: torch.Tensor,
                  z_prev: Optional[torch.Tensor] = None, x_prev: Optional[torch.Tensor] = None,
                  g_prev: Optional[torch.Tensor] = None, wg_prev: Optional[torch.Tensor] = None, gate_off: bool = False,
                  dropout_p: float = 0.0, seed: int = 0, step: int = 0, site_prev: int = 0,
                  dys_out: Optional[torch.Tensor] = None, dxd_out=_NEW, dx_out: Optional[torch.Tensor] = None,
                  partial: Optional[torch.Tensor] = None):
    """The backward twin of `gcn_layer_fwd` (cgcn_gcn_layer_bwd): `dys_gather` is D^-1 dy of this layer (the panel the
    column indices address), `dxd` its (1-g) dh, `weight` its `[128 in, 128 out]` W; panels as in `gcn_layer_fwd`.
    With the layer below (`z_prev`, `x_prev`, `g_prev` `[n, S]`, `wg_prev`; `dropout_p` / `seed` / `step` / `site_prev`
    draw its output's keep-mask) returns `(dys_out, dxd_out, partial[:parts])`: D^-1 dy and (1-g) dh of the layer below
    and the per-CTA column sums `d b | d w_g | d b_g` (`[parts, 260]`).  `dxd_out` may be `dxd` (updated in place) or
    None (not written).  Without it (`z_prev` None) returns `dx_out` = d loss / d x_in.  The output tensors, when given,
    receive the results (`partial`: at least as many rows as the kernel has CTAs)."""
    lib = _lib.load()
    dys_gather = _f32c(dys_gather)
    n = graph.n
    S = dys_gather.shape[1] if dys_gather.dim() == 3 else 1
    dev = dys_gather.device
    shape = dys_gather.shape
    mid = z_prev is not None
    if mid:
        dys_out = _out(dys_out, shape, dev)
        dxd_out = None if dxd_out is None else _out(None if dxd_out is _NEW else dxd_out, shape, dev)
        partial = _out(partial, (_max_layer_parts(n, S, dev), 2 * 128 + 4), dev, more_rows=True)
        dx_out = None
    else:
        dx_out = _out(dx_out, shape, dev)
        dys_out = dxd_out = partial = None
    dxd_in = dxd_out if dxd_out is dxd else _f32c(dxd)      # in place: the kernel reads and writes the caller's buffer
    opt = lambda t: _lib.ptr(None if t is None else _f32c(t))
    parts = C.c_int32(0)
    gs = graph.c_struct()
    with torch.cuda.device(dev):
        _lib.check(lib.cgcn_gcn_layer_bwd(C.byref(gs), S, dys_gather.data_ptr(), dxd_in.data_ptr(), _f32c(weight).data_ptr(),
                                          opt(z_prev), opt(x_prev), opt(g_prev), opt(wg_prev), 1 if gate_off else 0,
                                          float(dropout_p), seed, step, site_prev, _lib.ptr(dys_out), _lib.ptr(dxd_out),
                                          _lib.ptr(dx_out), _lib.ptr(partial), C.byref(parts), _lib.current_stream()),
                   "cgcn_gcn_layer_bwd")
    return (dys_out, dxd_out, partial[: parts.value]) if mid else dx_out


def gemm_rowpanel(a: torch.Tensor, b: torch.Tensor, b_transposed: bool = False, bias: Optional[torch.Tensor] = None,
                  rowscale_graph: Optional[HiCGraph] = None, rowscale_group: int = 1, impl: int = GEMM_AUTO,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """`C = rowscale * (A @ (B.T if b_transposed else B)) + bias` for a tall A `[m, k]`, k, n <= 128."""
    lib = _lib.load()
    a, b = _f32c(a), _f32c(b)
    m, k = a.shape
    n = b.shape[0] if b_transposed else b.shape[1]
    assert (b.shape[1] if b_transposed else b.shape[0]) == k
    if out is None:
        out = torch.empty(m, n, dtype=torch.float32, device=a.device)
    ws = torch.empty(1 << 20, dtype=torch.uint8, device=a.device)
    bias_c = _f32c(bias) if bias is not None else None
    with torch.cuda.device(a.device):
        _lib.check(lib.cgcn_gemm_rowpanel(a.data_ptr(), k, b.data_ptr(), int(b_transposed), _lib.ptr(bias_c),
                                          out.data_ptr(), n, m, n, k,
                                          rowscale_graph.rowptr.data_ptr() if rowscale_graph is not None else None,
                                          _lib.ptr(rowscale_graph.row_inv) if rowscale_graph is not None else None,
                                          rowscale_group, impl, ws.data_ptr(), ws.numel(), _lib.current_stream()),
                   "cgcn_gemm_rowpanel")
    return out


def gemm_gram(a: torch.Tensor, b: torch.Tensor, impl: int = GEMM_AUTO, out: Optional[torch.Tensor] = None,
              accumulate: bool = False) -> torch.Tensor:
    """`C[ka, nb] (+)= A.T @ B` for tall A `[m, ka]`, B `[m, nb]` (a reduction over the m rows)."""
    lib = _lib.load()
    a, b = _f32c(a), _f32c(b)
    m, ka = a.shape
    nb = b.shape[1]
    if out is None:
        out = torch.zeros(ka, nb, dtype=torch.float32, device=a.device)
    with torch.cuda.device(a.device):
        need = lib.cgcn_gemm_gram_workspace_bytes(m)
        ws = torch.empty(need, dtype=torch.uint8, device=a.device)
        _lib.check(lib.cgcn_gemm_gram(a.data_ptr(), ka, b.data_ptr(), nb, out.data_ptr(), nb, m, ka, nb,
                                      int(accumulate), impl, ws.data_ptr(), need, _lib.current_stream()),
                   "cgcn_gemm_gram")
    return out


def pack_targets(target: torch.Tensor, pin: bool = False) -> Optional[torch.Tensor]:
    """Host side of `cgcn_bce_loss_bits` / `cgcn_train_step_bits`: a 0/1 label matrix `[n, C]` (finetune.py:32)
    as `[n, ceil(C/32)]` int32 bit rows (bit c of a row = label c).  Returns None when some entry is neither
    0 nor 1 (soft labels keep the float path)."""
    import numpy as np
    t = target.detach().cpu().numpy()
    b = t != 0
    if not np.array_equal(b.astype(t.dtype), t):
        return None
    n, c = b.shape
    wpr = (c + 31) // 32
    packed = np.zeros((n, wpr * 4), dtype=np.uint8)
    packed[:, : (c + 7) // 8] = np.packbits(b, axis=1, bitorder="little")
    out = torch.from_numpy(packed.view("<i4").reshape(n, wpr))
    return out.pin_memory() if pin else out


def bce_loss(out: torch.Tensor, target: torch.Tensor, strands: int, loss_acc: torch.Tensor,
             want_probs: bool = True, want_grad: bool = True, n_total: int = 0, nclass: Optional[int] = None,
             probs_out: Optional[torch.Tensor] = None, grad_out: Optional[torch.Tensor] = None,
             workspace: Optional[torch.Tensor] = None):
    """finetune.py:43-45,52 on `[n, strands, ld]` logits (row pitch ld >= C): returns `(probs [n, C] | None,
    out_grad | None)` and adds the mean loss to `loss_acc[0]` (over `n_total` rows when the logits are one row block
    of a larger graph).  An int32 `target` is a `pack_targets` bit matrix (pass `nclass`).  `probs_out` / `grad_out`,
    when given, receive the results (`want_*` then does not matter); `workspace` is at least
    `cgcn_bce_workspace_bytes` long."""
    lib = _lib.load()
    out = _f32c(out)
    dev = out.device
    bits = target.dtype == torch.int32
    if bits:
        if nclass is None or target.dim() != 2 or target.shape[1] != (nclass + 31) // 32:
            raise ValueError("bit-packed targets need nclass with ceil(nclass/32) == target.shape[1]")
        target, c = target.contiguous(), int(nclass)
    else:
        target = _f32c(target)
        c = target.shape[1]
        if nclass is not None and c != nclass:
            raise ValueError("targets have %d columns, nclass is %d" % (c, nclass))
    n = target.shape[0]
    if out.shape[0] != n:
        raise ValueError("%d logit rows, %d target rows" % (out.shape[0], n))
    probs = _out(probs_out, (n, c), dev, align=4) if (probs_out is not None or want_probs) else None
    grad = _out(grad_out, tuple(out.shape), dev) if (grad_out is not None or want_grad) else None
    with torch.cuda.device(dev):
        if workspace is None:
            workspace = torch.empty(lib.cgcn_bce_workspace_bytes(n, c), dtype=torch.uint8, device=dev)
        name = "cgcn_bce_loss_bits" if bits else "cgcn_bce_loss"
        _lib.check(getattr(lib, name)(out.data_ptr(), target.data_ptr(), n, c, strands, out.shape[-1], n_total,
                                      _lib.ptr(probs), loss_acc.data_ptr(), _lib.ptr(grad), _lib.ptr(workspace),
                                      workspace.numel() * workspace.element_size(), _lib.current_stream()), name)
    return probs, grad


def sgd_step(params: torch.Tensor, grads: torch.Tensor, buf: torch.Tensor, lr: float, momentum: float = 0.9,
             weight_decay: float = 1e-6, grad_scale: float = 1.0) -> None:
    lib = _lib.load()
    with torch.cuda.device(params.device):
        _lib.check(lib.cgcn_sgd_step(params.data_ptr(), grads.data_ptr(), buf.data_ptr(), params.numel(), lr, momentum,
                                     weight_decay, grad_scale, _lib.current_stream()), "cgcn_sgd_step")


def adam_step(params: torch.Tensor, grads: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor, lr: float,
              step_index: int, beta1: float = 0.9, beta2: float = 0.98, eps: float = 1e-8, grad_scale: float = 1.0) -> None:
    lib = _lib.load()
    with torch.cuda.device(params.device):
        _lib.check(lib.cgcn_adam_step(params.data_ptr(), grads.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(),
                                      params.numel(), lr, beta1, beta2, eps, step_index, grad_scale,
                                      _lib.current_stream()), "cgcn_adam_step")


def interleave_strands(strands: Sequence[torch.Tensor], out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """`[n, d]` x S  ->  `[n, S, d]` panel."""
    lib = _lib.load()
    srcs = [_f32c(s) for s in strands]
    n, d = srcs[0].shape
    s = len(srcs)
    if out is None:
        out = torch.empty(n, s, d, dtype=torch.float32, device=srcs[0].device)
    arr = (C.c_void_p * s)(*[t.data_ptr() for t in srcs])
    with torch.cuda.device(out.device):
        _lib.check(lib.cgcn_interleave_strands(arr, s, n, d, out.data_ptr(), _lib.current_stream()),
                   "cgcn_interleave_strands")
    return out


def deinterleave_strands(panel: torch.Tensor) -> Tuple[torch.Tensor, ...]:
    """`[n, S, w]` -> S tensors `[n, w]`."""
    lib = _lib.load()
    panel = _f32c(panel)
    n, s, w = panel.shape
    outs = [torch.empty(n, w, dtype=torch.float32, device=panel.device) for _ in range(s)]
    arr = (C.c_void_p * s)(*[t.data_ptr() for t in outs])
    with torch.cuda.device(panel.device):
        _lib.check(lib.cgcn_deinterleave_strands(panel.data_ptr(), s, n, w, arr, _lib.current_stream()),
                   "cgcn_deinterleave_strands")
    return tuple(outs)


def dropout_mask(n: int, strands: int, d: int, p: float, seed: int, step: int, site: int, device=None) -> torch.Tensor:
    """Keep-mask (0 or 1/(1-p)) `[n, strands, d]` the model draws at `site` for `(seed, step)`."""
    lib = _lib.load()
    dev = _lib.require_cuda(device)
    mask = torch.empty(n, strands, d, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.cgcn_dropout_mask(mask.data_ptr(), n, strands, d, p, seed, step, site, _lib.current_stream()),
                   "cgcn_dropout_mask")
    return mask


def adjacency_build(window_starts, bin1, bin2, val, norm, resolution_kb: int, hic_edges: int, device=None):
    """Hi-C contacts -> `(indptr int32 [N+1], indices int32 [nnz])` numpy arrays of the binary symmetric
    adjacency, computed on the GPU (cgcn_adj_build; data/7create_graph_new.py:67-120).
    `norm is None` is the reference's `--norm ''` mode (first K accepted rows of a pre-sorted file)."""
    lib = _lib.load()
    dev = _lib.require_cuda(device)
    starts = np.unique(np.asarray(window_starts, dtype=np.int64))          # bed rows -> sorted unique starts (:24-44)
    n = int(starts.shape[0])
    m = int(np.asarray(bin1).shape[0])
    k_pairs = int(hic_edges / 2.0)
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(dev)
    d_b1, d_b2, d_v, d_w = t(bin1, np.int64), t(bin2, np.int64), t(val, np.float64), t(starts, np.int64)
    d_norm = t(norm, np.float64) if norm is not None else None
    cap = 2 * (k_pairs if 0 < k_pairs < m else m)
    rowptr = torch.empty(n + 1, dtype=torch.int32, device=dev)
    colidx = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
    need = C.c_size_t(0)
    nnz = C.c_int64(0)
    with torch.cuda.device(dev):
        _lib.check(lib.cgcn_adj_build_workspace_bytes(m, n, k_pairs, C.byref(need)), "cgcn_adj_build_workspace_bytes")
        ws = torch.empty(need.value, dtype=torch.uint8, device=dev)
        _lib.check(lib.cgcn_adj_build(d_b1.data_ptr(), d_b2.data_ptr(), d_v.data_ptr(), m, d_w.data_ptr(), n,
                                      _lib.ptr(d_norm), 0 if d_norm is None else d_norm.numel(),
                                      1000 * int(resolution_kb), k_pairs, 0 if d_norm is None else 1,
                                      rowptr.data_ptr(), colidx.data_ptr(), cap, C.byref(nnz), ws.data_ptr(), need.value,
                                      _lib.current_stream()), "cgcn_adj_build")
    return rowptr.cpu().numpy(), colidx[: nnz.value].cpu().numpy()
