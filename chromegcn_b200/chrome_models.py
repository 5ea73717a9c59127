"""Drop-in `GraphConvolution` and `ChromeGCN` (reference: models/SubLayers.py:7-57,
models/ChromeModels.py:21-52) running on libchromegcn's sm_100a kernels.

Same constructor arguments, parameter names / shapes (state_dicts interchange with the
reference), initialisation and `forward(x_in, adj, deg, src_dict=None, return_gate=False)`
returning `(x_in, out, (g, g2), None)`.  `adj` may be the `HiCGraph` this package's
`process_graph` returns, or the torch sparse COO tensor the reference's `process_graph` returns
(converted once on the GPU and cached).  There is no eager / CPU fallback: inputs must be CUDA
fp32 and the shared library must be built.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from . import _lib, ops
from .graph import HiCGraph

PARAM_ORDER = ["GC1.weight", "GC1.bias", "W1.weight", "W1.bias", "GC2.weight", "GC2.bias", "W2.weight", "W2.bias",
               "batch_norm.weight", "batch_norm.bias", "out.weight", "out.bias"]
MAX_LAYERS = _lib.MAX_LAYERS


def param_order(layers: int) -> List[str]:
    """State-dict names in the reference's order for an `layers`-layer model (GC3/W3... only in extended mode)."""
    names: List[str] = []
    for l in range(1, layers + 1):
        names += ["GC%d.weight" % l, "GC%d.bias" % l, "W%d.weight" % l, "W%d.bias" % l]
    return names + ["batch_norm.weight", "batch_norm.bias", "out.weight", "out.bias"]


def padded_classes(nclass: int) -> int:
    """Row pitch (floats) of the logit buffers: a multiple of 4 keeps rows 16-byte aligned, which puts the
    head contractions on the tcgen05 path."""
    return (nclass + 3) // 4 * 4


def bn_momentum(bn: nn.BatchNorm1d) -> float:
    """The exponential factor of the running statistics.  `momentum=None` (cumulative moving average with factor
    1 / num_batches_tracked) is not what the reference builds (models/ChromeModels.py:30: `nn.BatchNorm1d(nfeat)`)
    and is not implemented by the kernels: refuse it instead of silently using 0.1."""
    if bn.momentum is None:
        raise NotImplementedError("BatchNorm1d(momentum=None) (cumulative moving average) is not supported by the "
                                  "CUDA path; the reference uses the default momentum 0.1")
    return float(bn.momentum)


def _as_graph(adj, cache: Dict) -> HiCGraph:
    if isinstance(adj, HiCGraph):
        return adj
    if isinstance(adj, torch.Tensor) and adj.layout == torch.sparse_coo:
        key = (adj._values().data_ptr(), adj._indices().data_ptr(), adj._nnz(), tuple(adj.shape))
        g = cache.get(key)
        if g is None:
            g = HiCGraph.from_torch_coo(adj)
            if len(cache) > 64:
                cache.clear()
            cache[key] = g
        return g
    raise TypeError("adj must be a HiCGraph or a torch tensor (sparse COO or dense)")


class _GraphConvFn(torch.autograd.Function):
    """y = (A_hat x) W + b   (models/SubLayers.py:42-52), A_hat = D^-1 bin(A+I) given as a pattern."""

    @staticmethod
    def forward(ctx, x, weight, bias, graph):
        x = ops._f32c(x)
        ax = ops.spmm(graph, x, mean=True) if graph is not None else x
        y = ops.gemm_rowpanel(ax, weight.detach(), False, bias.detach() if bias is not None else None)
        ctx.graph = graph
        ctx.has_bias = bias is not None
        ctx.save_for_backward(ax, weight)
        return y

    @staticmethod
    def backward(ctx, dy):
        ax, weight = ctx.saved_tensors
        dy = ops._f32c(dy)
        graph = ctx.graph
        dw = ops.gemm_gram(ax, dy) if ctx.needs_input_grad[1] else None
        db = dy.sum(0) if (ctx.has_bias and ctx.needs_input_grad[2]) else None
        dx = None
        if ctx.needs_input_grad[0]:
            if graph is None:
                dx = ops.gemm_rowpanel(dy, weight.detach(), True)
            else:
                t = ops.gemm_rowpanel(dy, weight.detach(), True, rowscale_graph=graph, rowscale_group=1)
                dx = ops.spmm(graph, t, mean=False)
        return dx, dw, db, None


class GraphConvolution(nn.Module):
    """models/SubLayers.py:7-57.  Standalone use runs SpMM + GEMM kernels; inside `ChromeGCN` the
    whole model runs as one fused sequence instead."""

    def __init__(self, in_features, out_features, bias=True, init="xavier"):
        super().__init__()
        self.in_features = in_features
        self.out_features = out_features
        self.weight = nn.Parameter(torch.empty(in_features, out_features))
        if bias:
            self.bias = nn.Parameter(torch.empty(out_features))
        else:
            self.register_parameter("bias", None)
        if init == "xavier":                      # models/SubLayers.py:32-35
            nn.init.xavier_normal_(self.weight.data, gain=0.02)
        elif init == "kaiming":                   # models/SubLayers.py:37-40
            nn.init.kaiming_normal_(self.weight.data, a=0, mode="fan_in")
        elif init == "uniform":                   # models/SubLayers.py:26-30
            stdv = 1.0 / (self.weight.size(1) ** 0.5)
            self.weight.data.uniform_(-stdv, stdv)
            if self.bias is not None:
                self.bias.data.uniform_(-stdv, stdv)
        else:
            raise NotImplementedError
        if self.bias is not None and init != "uniform":
            nn.init.constant_(self.bias.data, 0.0)
        self._graph_cache: Dict = {}

    def forward(self, input, adj, deg=None):
        _lib.require_cuda()
        graph = _as_graph(adj, self._graph_cache) if adj is not None else None
        return _GraphConvFn.apply(input, self.weight, self.bias, graph)

    def __repr__(self):
        return "%s (%d -> %d)" % (self.__class__.__name__, self.in_features, self.out_features)


def fill_params(ps: _lib.Params, tensors: Dict[str, Optional[torch.Tensor]], layers: int) -> None:
    def p(name):
        t = tensors.get(name)
        return None if t is None else _lib.ptr(t)
    for l in range(layers):
        ps.gc_w[l] = p("GC%d.weight" % (l + 1))
        ps.gc_b[l] = p("GC%d.bias" % (l + 1))
        ps.gate_w[l] = p("W%d.weight" % (l + 1))
        ps.gate_b[l] = p("W%d.bias" % (l + 1))
    ps.bn_w, ps.bn_b = p("batch_norm.weight"), p("batch_norm.bias")
    ps.out_w, ps.out_b = p("out.weight"), p("out.bias")


def call_buffers(model: "ChromeGCN", n: int, strands: int, alloc: Callable[[str, int], torch.Tensor],
                 out_grad: bool = False):
    """The buffers of one model call over `n` rows: `(workspace, out, out_grad, gates)` -- the workspace
    `cgcn_model_workspace_bytes` asks for, the logits `[n, strands, padded_classes(nclass)]`, their gradient (None unless
    `out_grad`) and one `[n, strands]` gate per layer.  `alloc(name, numel)` returns a float32 tensor of at least `numel`
    elements: a fresh one, or a cached one that is reused from call to call."""
    d, nclass, layers = model.GC1.in_features, model.out.out_features, model.num_layers
    ws_bytes = _lib.load().cgcn_model_workspace_bytes(n, d, nclass, layers, strands)
    if ws_bytes == 0:
        raise _lib.ChromeGCNNativeError("cgcn_model_workspace_bytes rejected n=%d d=%d" % (n, d))
    shape = (n, strands, padded_classes(nclass))
    logits = n * strands * shape[2]
    ws = alloc("ws", ws_bytes // 4)
    out = alloc("out", logits)[:logits].view(shape)
    gates = [alloc("gate%d" % l, n * strands)[: n * strands].view(n, strands) for l in range(layers)]
    dout = alloc("dout", logits)[:logits].view(shape) if out_grad else None
    return ws, out, dout, gates


def model_struct(model: "ChromeGCN", *, graph: HiCGraph, strands: int, x_in: torch.Tensor,
                 x_in_grad: Optional[torch.Tensor] = None, params: Dict[str, torch.Tensor],
                 grads: Optional[Dict[str, torch.Tensor]] = None, out: torch.Tensor, gates: List[torch.Tensor],
                 out_grad: Optional[torch.Tensor] = None, workspace: torch.Tensor,
                 dropout_counter: Tuple[int, int]) -> _lib.Model:
    """The `cgcn_model` struct of one call of `model`.  Everything the module owns comes from it: d, nclass, layers,
    train / eval mode, dropout rate, `gate_off`, `gemm_impl` and the BatchNorm settings and running statistics.  The
    caller passes what belongs to the call: graph, strand count, tensors (buffers as `call_buffers` sizes them) and the
    dropout counter `(seed, step)` the call draws its masks from (`ChromeGCN._next_dropout_counter`)."""
    layers, bn = model.num_layers, model.batch_norm
    nclass = model.out.out_features
    seed, step = dropout_counter
    m = _lib.Model()
    m.out_ld = padded_classes(nclass)
    m.gate_off = 1 if model.gate_off else 0
    m.graph = graph.c_struct()
    m.d, m.nclass, m.layers, m.strands = model.GC1.in_features, nclass, layers, strands
    m.training = 1 if model.training else 0
    m.gemm_impl = model.gemm_impl
    m.need_input_grad = 1 if x_in_grad is not None else 0
    m.dropout_p, m.bn_momentum, m.bn_eps = float(model.dropout), bn_momentum(bn), float(bn.eps)
    m.seed, m.step = seed & 0xFFFFFFFFFFFFFFFF, step & 0xFFFFFFFFFFFFFFFF
    fill_params(m.params, params, layers)
    if grads is not None:
        fill_params(m.grads, grads, layers)
    m.bn_running_mean, m.bn_running_var = _lib.ptr(bn.running_mean), _lib.ptr(bn.running_var)
    m.bn_num_batches_tracked = _lib.ptr(bn.num_batches_tracked)
    m.x_in, m.x_in_grad, m.out = _lib.ptr(x_in), _lib.ptr(x_in_grad), _lib.ptr(out)
    for l in range(layers):
        m.gate[l] = _lib.ptr(gates[l])
    m.out_grad = _lib.ptr(out_grad)
    m.workspace, m.workspace_bytes = workspace.data_ptr(), workspace.numel() * workspace.element_size()
    m.stream = _lib.current_stream()
    return m


class _ChromeGCNFn(torch.autograd.Function):
    """One `ChromeGCN.forward` call (strands = 1) as cgcn_model_forward / cgcn_model_backward."""

    @staticmethod
    def forward(ctx, x_in, module, graph, *param_tensors):
        lib = _lib.load()
        names = module._param_names()
        params = {k: ops._f32c(t.detach()) for k, t in zip(names, param_tensors)}
        x = ops._f32c(x_in.detach())
        n, nclass, layers = x.shape[0], module.out.out_features, module.num_layers
        dev = x.device
        with torch.cuda.device(dev):
            # fresh buffers: the workspace and the logits are saved for the backward of this node
            ws, out, _, gates = call_buffers(module, n, 1, lambda name, numel: torch.empty(numel, dtype=torch.float32,
                                                                                          device=dev))
            counter = module._next_dropout_counter()
            m = model_struct(module, graph=graph, strands=1, x_in=x, params=params, out=out, gates=gates, workspace=ws,
                             dropout_counter=counter)
            _lib.check(lib.cgcn_model_forward(C.byref(m)), "cgcn_model_forward")
        ctx.module, ctx.graph, ctx.names = module, graph, names
        ctx.training, ctx.counter = module.training, counter
        ctx.save_for_backward(x, ws, out, *gates, *[params[k] for k in names])
        ctx.mark_non_differentiable(*gates)
        return (out[:, 0, :nclass], *gates)

    @staticmethod
    def backward(ctx, dout, *unused):
        lib = _lib.load()
        module, graph, names = ctx.module, ctx.graph, ctx.names
        layers = module.num_layers
        saved = ctx.saved_tensors
        x, ws, out = saved[0], saved[1], saved[2]
        gates = list(saved[3:3 + layers])
        params = dict(zip(names, saved[3 + layers:]))
        dev = x.device
        dpad = torch.zeros_like(out)
        dpad[:, 0, :dout.shape[1]] = dout
        with torch.cuda.device(dev):
            grads = {k: torch.empty_like(v) for k, v in params.items()}
            dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
            m = model_struct(module, graph=graph, strands=1, x_in=x, x_in_grad=dx, params=params, grads=grads, out=out,
                             gates=gates, out_grad=dpad, workspace=ws, dropout_counter=ctx.counter)
            m.training = 1 if ctx.training else 0            # the mode the forward ran in
            _lib.check(lib.cgcn_model_backward(C.byref(m)), "cgcn_model_backward")
        return (dx, None, None, *[grads[k] for k in names])


class ChromeGCN(nn.Module):
    """models/ChromeModels.py:21-52.  `gate` is accepted and ignored and `layers != 2` gives one
    layer, exactly like the reference (SURVEY.md F6, F7).

    `extended=True` (not in the reference; the variant sweep of BASELINE.json needs "gcn_layers 3" and "gate off",
    which the reference cannot express) honours both arguments: `layers` in 1..4 builds GC1..GC{layers} / W1..W{layers}
    with the same per-layer recipe (dropout between consecutive layers), and `gate=False` makes every layer
    `x <- tanh(A_hat x W + b)` (g == 1; the W{l} parameters stay in the state_dict and receive zero gradients).
    `forward` still returns `(x_in, out, (g, g2), None)`; further gates are in `self.last_gates`."""

    def __init__(self, nfeat, nhid, nclass, dropout, gate, layers, extended: bool = False):
        super().__init__()
        if nfeat != nhid:
            raise ValueError("ChromeGCN needs nhid == nfeat (W1 = Linear(nfeat, 1) is applied to an nhid-wide tensor, "
                             "models/ChromeModels.py:24-25)")
        self.extended = bool(extended)
        self.gate_off = self.extended and not bool(gate)
        if self.extended:
            if not 1 <= int(layers) <= MAX_LAYERS:
                raise ValueError("extended ChromeGCN supports 1..%d layers" % MAX_LAYERS)
            n_layers = int(layers)
        else:
            n_layers = 2 if layers == 2 else 1
        self.num_layers = n_layers
        self.GC1 = GraphConvolution(nfeat, nhid, bias=True, init="xavier")
        self.W1 = nn.Linear(nfeat, 1)
        for l in range(2, n_layers + 1):
            setattr(self, "GC%d" % l, GraphConvolution(nhid, nfeat, bias=True, init="xavier"))
            setattr(self, "W%d" % l, nn.Linear(nfeat, 1))
        self.last_gates: List[torch.Tensor] = []
        self.dropout = dropout
        self.batch_norm = nn.BatchNorm1d(nfeat)
        self.out = nn.Linear(nfeat, nclass)
        self.gemm_impl = ops.GEMM_AUTO
        self._graph_cache: Dict = {}
        self._drop_seed: Optional[int] = None
        self._drop_step = 0

    # -- helpers shared with the fused trainer
    def _param_names(self) -> List[str]:
        return param_order(self.num_layers)

    def _param_tensors(self) -> List[torch.Tensor]:
        sd = dict(self.named_parameters())
        return [sd[k] for k in self._param_names()]

    def _next_dropout_counter(self) -> Tuple[int, int]:
        """`(seed, step)` of the dropout masks of the next forward call: advances once per call in training mode,
        `(0, 0)` in eval mode (no dropout)."""
        if not self.training:
            return 0, 0
        if self._drop_seed is None:
            self._drop_seed = int(torch.randint(0, 2 ** 62, (1,)).item())     # follows torch.manual_seed
        self._drop_step += 1
        return self._drop_seed, self._drop_step

    def resolve_graph(self, adj) -> Optional[HiCGraph]:
        """The pattern graph behind `adj`, or None when `adj` needs the generic path (generic_adj.py)."""
        if isinstance(adj, torch.Tensor) and (adj.layout == torch.strided or adj.requires_grad):
            return None
        try:
            return _as_graph(adj, self._graph_cache)
        except NotImplementedError:
            if isinstance(adj, torch.Tensor):
                return None
            raise

    def forward(self, x_in, adj, deg=None, src_dict=None, return_gate=False):
        _lib.require_cuda()
        if not (isinstance(x_in, torch.Tensor) and x_in.is_cuda):
            raise _lib.ChromeGCNNativeError("ChromeGCN.forward needs CUDA inputs (no CPU fallback)")
        graph = self.resolve_graph(adj)
        if graph is None:
            # dense `adj`, `adj` that requires grad, or a sparse tensor that is not a symmetric mean-aggregation pattern
            # (scripts/visualize.py:30-45,103-111): the generic weighted-CSR path with d loss / d adj
            from .generic_adj import forward_generic
            out, gates = forward_generic(self, x_in, adj)
            self.last_gates = list(gates)
            return x_in, out, (gates[0], gates[1] if self.num_layers >= 2 else None), None
        res = _ChromeGCNFn.apply(x_in, self, graph, *self._param_tensors())
        out, g = res[0], res[1]
        g2 = res[2] if self.num_layers >= 2 else None
        self.last_gates = list(res[1:])
        return x_in, out, (g, g2), None
