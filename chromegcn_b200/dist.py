"""Multi-GPU plumbing for the chromosome model: one process per GPU, `torch.distributed` (NCCL on
the GPU box, gloo in CPU tests) for the exchange steps.

The reference trains on one GPU (README.md:45) and takes one optimiser step per chromosome
(finetune.py:39-49).  Two ways the path shards (SURVEY.md 8(e)):

* whole genome -- chromosomes are independent graphs that share only the 46 825 parameters, so
  they are bin-packed (LPT) onto ranks; the ranks walk their lists in lock-step "rounds", and each
  round ends with ONE all-reduce of the flat gradient buffer (~190 KB) and the same optimiser step
  on every rank.  Semantics: one step per round on the mean of that round's per-chromosome
  gradients (a grouped version of the reference's sequential steps; with world_size 1 it is
  exactly the reference's trajectory).
* one oversized graph -- contiguous row blocks per rank (`row_partition`); because the pattern is
  symmetric the same partition serves forward and backward, and the exchange step is an all-gather
  of the `[rows_local, width]` feature panel before each SpMM (`allgather_panel`).
"""
from __future__ import annotations

from typing import Dict, List, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist


def chromosome_cost(n: int, nnz: int, d: int = 128, strands: int = 2) -> float:
    """Bytes moved per train step, the LPT weight: 3 SpMM passes + ~40 streamed panels."""
    row = 4.0 * d * strands
    return 3.0 * nnz * (4.0 + row) + 40.0 * n * row


def lpt_shards(costs: Dict[str, float], world: int) -> List[List[str]]:
    """Longest-processing-time bin packing; deterministic (ties by name)."""
    bins: List[List[str]] = [[] for _ in range(world)]
    load = [0.0] * world
    for name in sorted(costs, key=lambda k: (-costs[k], k)):
        r = min(range(world), key=lambda i: (load[i], i))
        bins[r].append(name)
        load[r] += costs[name]
    return bins


def num_rounds(shards: Sequence[Sequence[str]]) -> int:
    return max((len(s) for s in shards), default=0)


def active_in_round(shards: Sequence[Sequence[str]], t: int) -> int:
    return sum(1 for s in shards if t < len(s))


def allreduce_gradients(t: torch.Tensor, group=None) -> None:
    """In-place sum over the ranks of `group` of the flat gradient buffer (or, in the row-partitioned step, of the
    BatchNorm column sums and the loss); nothing without an initialised process group of more than one rank."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)


class NativeComm:
    """The library's own NCCL communicator (`cgcn_comm_*`, include/chromegcn.h): the calls a host without Python makes
    for the exchanges above.  Here it is exercised next to torch.distributed (tests/test_gpu_sharded.py), not used
    by default: `id_bytes` comes from `NativeComm.unique_id()` on rank 0 and reaches the other ranks by any channel
    (the tests broadcast it with torch.distributed)."""

    def __init__(self, id_bytes: bytes, world: int, rank: int, device=None):
        import ctypes as C
        from . import _lib
        self._lib = _lib
        self._h = C.c_void_p()
        self.world, self.rank = int(world), int(rank)
        self.device = _lib.require_cuda(device)
        assert len(id_bytes) == 128
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().cgcn_comm_init(C.byref(self._h), bytes(id_bytes), self.world, self.rank), "cgcn_comm_init")

    @staticmethod
    def unique_id() -> bytes:
        import ctypes as C
        from . import _lib
        buf = C.create_string_buffer(128)
        _lib.check(_lib.load().cgcn_comm_unique_id(buf), "cgcn_comm_unique_id")
        return buf.raw

    def allreduce_sum(self, t: torch.Tensor) -> None:
        assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()
        with torch.cuda.device(self.device):
            self._lib.check(self._lib.load().cgcn_comm_allreduce_sum(self._h, t.data_ptr(), t.numel(), self._lib.current_stream()),
                            "cgcn_comm_allreduce_sum")

    def allgather(self, send: torch.Tensor, recv: torch.Tensor) -> None:
        nbytes = send.numel() * send.element_size()
        assert send.is_cuda and recv.is_cuda and send.is_contiguous() and recv.is_contiguous()
        assert recv.numel() * recv.element_size() == nbytes * self.world
        with torch.cuda.device(self.device):
            self._lib.check(self._lib.load().cgcn_comm_allgather(self._h, send.data_ptr(), recv.data_ptr(), nbytes,
                                                                 self._lib.current_stream()), "cgcn_comm_allgather")

    def close(self) -> None:
        if self._h:
            self._lib.check(self._lib.load().cgcn_comm_destroy(self._h), "cgcn_comm_destroy")
            self._h = None


def default_rounds(n_items: int, world: int) -> int:
    """Optimiser steps per pass over the chromosomes: one per chromosome on one rank (the reference,
    finetune.py:39-49); ONE on several ranks: every rank walks its LPT share of the chromosomes accumulating
    gradients, one all-reduce, one step on the mean gradient of the whole pass.  Lock-step rounds cost
    sum_r max_rank load(r, rank); with 23 chromosomes over 8 ranks the packing granularity makes that 0.89 of
    the balanced pass for 2 rounds, 0.84 for 3, against 0.955 for a single round (chr1 alone is 8.2 % of the genome),
    measured 0.84 / 0.9x on 8 B200 (profiles/).  `balanced_schedule(..., rounds=k)` / `bench.py --rounds k` give the
    grouped variants (k = n_items // world keeps "about `world` chromosomes per step")."""
    return n_items if world <= 1 else 1


def balanced_schedule(costs: Dict[str, float], world: int, rounds: int = None) -> List[List[List[str]]]:
    """`schedule[round][rank]` = chromosomes that rank processes (accumulating gradients) before the round's
    all-reduce + optimiser step.  Rounds are lock-step, so the pass costs sum_r max_rank load(r, rank); with one
    chromosome per cell that is 97 + 57 + 35 (k windows) on 8 ranks for the whole genome, 78 % efficient,
    because chr1 alone sets the first round's pace.  Packing small chromosomes next to it does better: each
    round gets a capacity (its largest item, or the even share of what is left) and is filled LPT-fashion;
    the last round takes the remainder.  Deterministic."""
    if rounds is None:
        rounds = default_rounds(len(costs), world)
    rounds = max(1, min(rounds, len(costs)))
    if world <= 1:
        order = sorted(costs, key=lambda k: (-costs[k], k))
        return [[[c]] for c in order] if rounds == len(order) else [[list(order[r::rounds])] for r in range(rounds)]
    remaining = sorted(costs, key=lambda k: (-costs[k], k))
    schedule: List[List[List[str]]] = []
    for r in range(rounds):
        cells: List[List[str]] = [[] for _ in range(world)]
        load = [0.0] * world
        later_rounds = rounds - r - 1
        if later_rounds == 0:                                   # last round: plain LPT of everything left
            for c in remaining:
                k = min(range(world), key=lambda i: (load[i], i))
                cells[k].append(c)
                load[k] += costs[c]
            remaining = []
        elif remaining:
            cap = max(costs[remaining[0]], sum(costs[c] for c in remaining) / (world * (later_rounds + 1)))
            kept: List[str] = []
            for idx, c in enumerate(remaining):
                k = min(range(world), key=lambda i: (load[i], i))
                still_available = (len(remaining) - idx - 1) + len(kept)
                if load[k] + costs[c] <= cap * 1.0001 and still_available >= later_rounds:
                    cells[k].append(c)
                    load[k] += costs[c]
                else:
                    kept.append(c)
            remaining = kept
        schedule.append(cells)
    return schedule


def schedule_cost(schedule: Sequence[Sequence[Sequence[str]]], costs: Dict[str, float]) -> float:
    return sum(max(sum(costs[c] for c in cell) for cell in rnd) for rnd in schedule)


def schedule_shards(schedule: Sequence[Sequence[Sequence[str]]], world: int) -> List[List[str]]:
    return [[c for rnd in schedule for c in rnd[r]] for r in range(world)]


def sharded_train_epoch(engine, optimizer, schedule, rank: int, graphs, panels, targets,
                        probs: Dict[str, torch.Tensor], losses: torch.Tensor, group=None) -> None:
    """One pass over all chromosomes.  `schedule` comes from `balanced_schedule` (or is a plain list of
    per-rank lists = one chromosome per rank per round, `lpt_shards`).  `graphs/panels/targets/probs` hold this
    rank's chromosomes (device resident).  `losses[i]` receives the loss of this rank's i-th chromosome.
    Every round ends with ONE all-reduce of the flat gradient buffer and the same optimiser step on every rank,
    on the mean gradient of the round's chromosomes."""
    if schedule and isinstance(schedule[0], (list, tuple)) and (not schedule[0] or isinstance(schedule[0][0], str)):
        shards = schedule                                        # per-rank lists: lock-step, one chromosome per cell
        schedule = [[[s[t]] if t < len(s) else [] for s in shards] for t in range(num_rounds(shards))]
    cells = [rnd[rank] for rnd in schedule]
    totals = [sum(len(cell) for cell in rnd) for rnd in schedule]
    for i, c in enumerate(sharded_rounds(engine.model, optimizer, cells, totals, group)):
        engine.run(graphs[c], panels[c], targets[c], probs[c], losses[i: i + 1], train=True)


def sharded_rounds(model, optimizer, cells, totals, group=None):
    """One rank's chromosome-sharded pass as an iterator: yields the chromosomes of `cells[r]` round by round, and the
    caller runs each one's train step before it asks for the next.  In between this does the rest of the round: a
    cell's gradients are summed (every backward overwrites the flat gradient buffer), an empty cell contributes zeros,
    and the round ends with one all-reduce of the flat gradient buffer and `step_on_mean` over the `totals[r]`
    chromosomes all ranks ran in round r.  The pass ends with `sync_batchnorm_buffers`."""
    from .engine import flat_params
    fp = flat_params(model, full=False)
    bn = model.batch_norm
    nbt_before = bn.num_batches_tracked.clone() if bn.num_batches_tracked is not None else None
    acc = None
    for mine, total in zip(cells, totals):
        if len(mine) == 0:
            fp.flat_grad.zero_()
        for j, c in enumerate(mine):
            yield c
            if len(mine) > 1:
                if j == 0:
                    acc = fp.flat_grad.clone() if acc is None else acc.copy_(fp.flat_grad)
                else:
                    acc.add_(fp.flat_grad)
        if len(mine) > 1:
            fp.flat_grad.copy_(acc)
        allreduce_gradients(fp.flat_grad, group)
        step_on_mean(optimizer, fp.flat_grad, 1.0 / max(total, 1))
    sync_batchnorm_buffers(model, group, nbt_before)


def step_on_mean(optimizer, flat_grad: torch.Tensor, scale: float) -> None:
    """One optimiser step on `scale * flat_grad` (the mean of a round's summed gradients).  The flat-buffer
    optimisers fold the factor into their kernel (`grad_scale`, restored afterwards so that it never leaks into a
    later single-GPU `finetune()`); any other `torch.optim.Optimizer` gets the buffer scaled in place."""
    if hasattr(optimizer, "grad_scale"):
        prev = optimizer.grad_scale
        optimizer.grad_scale = scale
        try:
            optimizer.step()
        finally:
            optimizer.grad_scale = prev
    else:
        if scale != 1.0:
            flat_grad.mul_(scale)
        optimizer.step()


def sync_batchnorm_buffers(model, group=None, nbt_before: torch.Tensor = None) -> None:
    """Make the BatchNorm running statistics identical on every rank after a chromosome-sharded pass.  The
    reference updates ONE model's `running_mean / running_var` once per strand call of every chromosome
    (models/ChromeModels.py:49, finetune.py:41-42); here each rank only saw its own chromosomes, so the replicas end a
    pass with different buffers and an eval pass or a checkpoint (`utils/evals.py:250-263` saves the whole
    state_dict) would depend on the rank.  The buffers become the rank average (every rank's exponential average
    started from the same value and has seen ~1/world of the batches), and `num_batches_tracked` the start value
    plus the calls of ALL ranks, as in a single-model pass."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return
    w = dist.get_world_size(group)
    bn = model.batch_norm
    for buf in (bn.running_mean, bn.running_var):
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
        buf.div_(w)
    if nbt_before is not None and bn.num_batches_tracked is not None:
        delta = (bn.num_batches_tracked - nbt_before).to(torch.int64)
        dist.all_reduce(delta, op=dist.ReduceOp.SUM, group=group)
        bn.num_batches_tracked.copy_(nbt_before + delta)


# ------------------------------------------------------------------ one oversized graph: row partition
def row_partition(n: int, world: int) -> List[Tuple[int, int]]:
    """Contiguous, nearly equal row blocks `[begin, end)` per rank."""
    base, extra = divmod(n, world)
    out, b = [], 0
    for r in range(world):
        e = b + base + (1 if r < extra else 0)
        out.append((b, e))
        b = e
    return out


def local_rows_csr(indptr: np.ndarray, indices: np.ndarray, begin: int, end: int) -> Tuple[np.ndarray, np.ndarray]:
    """CSR of rows `[begin, end)` with GLOBAL column indices (the gathered panel is global)."""
    ip = np.asarray(indptr, dtype=np.int64)
    lo, hi = ip[begin], ip[end]
    return (ip[begin: end + 1] - lo).astype(np.int32), np.asarray(indices[lo:hi], dtype=np.int32)


def allgather_panel(local: torch.Tensor, parts: Sequence[Tuple[int, int]], out: torch.Tensor = None, group=None) -> torch.Tensor:
    """Exchange step of the row-partitioned SpMM: every rank contributes its `[rows_local, width]`
    block, every rank ends with the full `[n, width]` panel.  Blocks may differ by one row."""
    world = len(parts)
    n = parts[-1][1]
    width = local.shape[1]
    if out is None:
        out = torch.empty(n, width, dtype=local.dtype, device=local.device)
    if world == 1:
        out.copy_(local)
        return out
    rows_max = max(e - b for b, e in parts)
    if all(e - b == rows_max for b, e in parts) and out.is_contiguous():
        dist.all_gather_into_tensor(out, local.contiguous(), group=group)     # equal blocks: gather in place
        return out
    # blocks differ by one row: gather fixed-size padded blocks, then drop the padding
    rank = dist.get_rank(group)
    b0, e0 = parts[rank]
    send = torch.zeros(rows_max, width, dtype=local.dtype, device=local.device)
    send[: e0 - b0] = local
    recv = torch.empty(world, rows_max, width, dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(recv.view(world * rows_max, width), send, group=group)
    for r, (b, e) in enumerate(parts):
        out[b:e] = recv[r, : e - b]
    return out


# ------------------------------------------------------------------ peer-memory exchange (NVLink loads, no all-gather)
class PeerExchange:
    """Exchange buffers of the peer-memory SpMM (`cgcn_spmm_peer`, include/chromegcn.h piece 2b).

    Every rank allocates two `[rows_max, width]` buffers with `cgcn_peer_alloc`, the 64-byte CUDA IPC handles
    travel through `torch.distributed.all_gather_object`, and every rank maps the others' buffers.  An exchange
    step is `publish(local_panel)`: a device copy into this rank's current buffer followed by a one-element
    all-reduce on the stream, which is the cross-rank barrier ("every rank's copy has landed").  The two buffers
    alternate, so a buffer is only overwritten two exchanges later, when every peer has provably finished reading
    it (it had to pass the barrier in between) -- one barrier per exchange is enough.  `panel()` is the
    `cgcn_peer_panel` the next SpMM stage reads.  With world_size 1 no IPC is involved."""

    def __init__(self, parts: Sequence[Tuple[int, int]], rank: int, width: int, device, group=None):
        import ctypes as C
        from . import _lib, ops
        self._lib, self._C = _lib, C
        lib = _lib.load()
        self.parts, self.rank, self.width, self.group, self.device = list(parts), rank, width, group, device
        self.world = len(parts)
        rows_max = max(e - b for b, e in parts)
        self.bytes = rows_max * width * 4
        self.own: List[int] = []
        self.mapped: List[List[int]] = [[], []]          # [buffer][rank] -> device address
        self._opened: List[int] = []
        handles = []
        with torch.cuda.device(device):
            for _ in range(2):
                p, h = C.c_void_p(0), C.create_string_buffer(64)
                _lib.check(lib.cgcn_peer_alloc(max(self.bytes, 256), C.byref(p), h), "cgcn_peer_alloc")
                self.own.append(p.value)
                handles.append(h.raw)
            if self.world > 1:
                gathered: List = [None] * self.world
                dist.all_gather_object(gathered, handles, group=group)
            else:
                gathered = [handles]
            for k in range(2):
                for r in range(self.world):
                    if r == rank:
                        self.mapped[k].append(self.own[k])
                    else:
                        p = C.c_void_p(0)
                        _lib.check(lib.cgcn_peer_open(gathered[r][k], C.byref(p)), "cgcn_peer_open(rank %d)" % r)
                        self.mapped[k].append(p.value)
                        self._opened.append(p.value)
        begins = [b for b, _ in parts] + [parts[-1][1]]
        self._panels = [ops.peer_panel(self.mapped[k], begins, rank) for k in range(2)]
        self._flag = torch.zeros(1, dtype=torch.float32, device=device)
        self.cur = 0
        self.exchanges = 0

    def publish(self, local_ptr: int, nbytes: int) -> None:
        lib = self._lib.load()
        self.cur ^= 1
        self._lib.check(lib.cgcn_peer_publish(self.own[self.cur], local_ptr, nbytes, self._lib.current_stream()),
                        "cgcn_peer_publish")
        if self.world > 1:
            dist.all_reduce(self._flag, group=self.group)            # stream-ordered cross-rank barrier
        self.exchanges += 1

    def panel(self):
        return self._panels[self.cur]

    def close(self) -> None:
        lib = self._lib.load()
        if self.world > 1 and dist.is_initialized():
            torch.cuda.synchronize(self.device)
            dist.barrier(group=self.group)                            # nobody unmaps / frees memory a peer still reads
        for p in self._opened:
            lib.cgcn_peer_close(p)
        self._opened = []
        if self.world > 1 and dist.is_initialized():
            dist.barrier(group=self.group)
        for p in self.own:
            lib.cgcn_peer_free(p)
        self.own = []


# ------------------------------------------------------------------ row-partitioned train step (one huge graph)
PHASE_FWD_LAYER, PHASE_FWD_HEAD, PHASE_BWD_HEAD, PHASE_BWD_LAYER, PHASE_BWD_INPUT = 0, 1, 2, 3, 4


class RowPartitionedStep:
    """One chromosome too large for (or simply spread over) several GPUs: rank r owns the contiguous row block
    `parts[r]` of every panel, its rows of the CSR pattern (global column indices) and a replica of the
    parameters.  `run()` drives `cgcn_model_phase` stage by stage and performs the exchange steps in between
    (SURVEY.md 8(e)): all-gather of the panel the next SpMM reads (L forward + L-1 backward, +1 with input
    gradients), all-reduce of the BatchNorm column sums (forward and backward), and one all-reduce of the flat
    gradient buffer + loss at the end.  With world_size 1 the collectives are identities and the result is the
    single-GPU step.

    `exchange="peer"` (the B200 path) replaces every panel all-gather by `PeerExchange.publish` + the peer-memory
    SpMM: neighbour rows are NVLink loads from the owner's exchange buffer inside the kernel, nothing is
    materialised.  `exchange="nccl"` is the all-gather formulation."""

    def __init__(self, model, graph_local, parts: Sequence[Tuple[int, int]], rank: int, strands: int = 2, group=None,
                 exchange: str = "nccl"):
        from .engine import ChromosomeEngine
        self.model, self.graph, self.parts, self.rank, self.S, self.group = model, graph_local, list(parts), rank, strands, group
        self.engine = ChromosomeEngine(model, strands)
        self.n_total = parts[-1][1]
        self.n_local = parts[rank][1] - parts[rank][0]
        assert graph_local.n == self.n_local
        if exchange not in ("nccl", "peer"):
            raise ValueError("exchange must be 'nccl' or 'peer'")
        self.exchange = exchange
        self.peer: PeerExchange = None
        self._x_full: torch.Tensor = None                    # all-gathered panel (nccl exchange)
        self._bn_sums: torch.Tensor = None                   # BatchNorm column sums, all-reduced

    def close(self) -> None:
        if self.peer is not None:
            self.peer.close()
            self.peer = None

    def _gather(self, local_panel: torch.Tensor, x_full: torch.Tensor) -> None:
        w = x_full.shape[1]
        allgather_panel(local_panel.reshape(self.n_local, w), self.parts, out=x_full, group=self.group)

    def run(self, panel_local: torch.Tensor, target_local: torch.Tensor, loss_out: torch.Tensor, train: bool = True,
            probs_out: torch.Tensor = None, input_grad: torch.Tensor = None):
        """panel_local `[n_local, S, d]`, target_local `[n_local, C]`; returns local logits `[n_local, S, C]`.
        `loss_out[0]` receives the GLOBAL mean loss (all-reduced); gradients (all-reduced) land in the model's
        flat gradient buffer."""
        import ctypes as C
        from . import _lib, ops
        from .chrome_models import model_struct
        from .engine import flat_params
        lib = _lib.load()
        model, S = self.model, self.S
        fp = flat_params(model, full=False)
        n, d, nclass, layers = self.n_local, model.GC1.in_features, model.out.out_features, model.num_layers
        dev = panel_local.device
        W = S * d
        with torch.cuda.device(dev):
            ws, out, dout, gates = self.engine.call_buffers(n, out_grad=train)
            use_peer = self.exchange == "peer"
            if use_peer and self.peer is None:
                self.peer = PeerExchange(self.parts, self.rank, W, dev, self.group)
            if not use_peer and self._x_full is None:
                self._x_full = torch.empty(self.n_total, W, dtype=torch.float32, device=dev)
            if self._bn_sums is None:
                self._bn_sums = torch.empty(2 * S * d, dtype=torch.float64, device=dev)
            x_full, bn_sums = self._x_full, self._bn_sums
            m = model_struct(model, graph=self.graph, strands=S, x_in=panel_local, x_in_grad=input_grad,
                             params=fp.views(fp.flat), grads=fp.views(fp.flat_grad) if train else None, out=out,
                             gates=gates, out_grad=dout, workspace=ws, dropout_counter=model._next_dropout_counter())
            m.n_total, m.row_begin = self.n_total, self.parts[self.rank][0]
            m.x_full, m.bn_sums = (None if use_peer else x_full.data_ptr()), bn_sums.data_ptr()
            pub = C.c_void_p(0)
            peer_ref = []                  # keeps the cgcn_peer_panel the struct points at alive

            def phase(kind, layer=0):
                m.stream = _lib.current_stream()
                if use_peer:
                    peer_ref[:] = [self.peer.panel()]
                    m.peer = C.cast(C.pointer(peer_ref[0]), C.c_void_p)
                _lib.check(lib.cgcn_model_phase(C.byref(m), kind, layer, C.byref(pub)), "cgcn_model_phase(%d,%d)" % (kind, layer))
                return pub.value

            def gather_ptr(ptr):          # the published panel lives in the workspace: wrap it without copying
                if use_peer:
                    self.peer.publish(ptr, n * W * 4)
                    return
                off = (ptr - ws.data_ptr()) // 4
                self._gather(ws[off: off + n * W], x_full)

            # ---- forward
            if use_peer:
                self.peer.publish(ops._f32c(panel_local).data_ptr(), n * W * 4)
            else:
                self._gather(panel_local, x_full)
            for l in range(layers):
                p = phase(PHASE_FWD_LAYER, l)
                if p:
                    gather_ptr(p)
            if model.training:
                allreduce_gradients(bn_sums, self.group)
            phase(PHASE_FWD_HEAD)
            loss_local = torch.zeros(1, dtype=torch.float32, device=dev)
            ops.bce_loss(out, target_local, S, loss_local, want_probs=False, want_grad=False, n_total=self.n_total,
                         nclass=nclass, probs_out=probs_out, grad_out=dout, workspace=self.engine.loss_workspace(n))
            allreduce_gradients(loss_local, self.group)
            loss_out += loss_local
            if not train:
                return out[:, :, :nclass], gates
            # ---- backward
            phase(PHASE_BWD_HEAD)
            allreduce_gradients(bn_sums, self.group)
            for l in range(layers - 1, -1, -1):
                p = phase(PHASE_BWD_LAYER, l)
                if p:
                    gather_ptr(p)
            if input_grad is not None:
                phase(PHASE_BWD_INPUT)
            allreduce_gradients(fp.flat_grad, self.group)
            fp.attach_grads()
        return out[:, :, :nclass], gates
