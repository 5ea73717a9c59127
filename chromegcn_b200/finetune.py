"""Drop-in `finetune(...)` (reference: finetune.py:9-67): one pass over the chromosomes of a split.

Same signature and return value `(all_preds, all_targets, total_loss)`.  What the reference does
per chromosome per epoch on the host -- unpickle the graphs, scipy `process_graph`, four pageable
H2D copies, `loss.item()`, `.cpu()` + quadratic `torch.cat` -- becomes:
  * graph pickles are read once and the `bin(A+I)` patterns stay on the GPU (cache keyed by file);
  * features / targets stream host -> device on a copy stream, one chromosome ahead of the compute
    stream (or stay resident when `opt.cache_features_on_device` is set); the 0/1 label matrix, the one
    input that never changes between epochs, is bit-packed on the host the first time it is seen
    (pinned, 16 B per window instead of 4*nclass) and consumed in that form by `cgcn_train_step_bits`;
  * the chromosome step is one `cgcn_train_step` call; losses go to a device array, probabilities
    into one preallocated `[sum N, nclass]` device buffer; one D2H copy and one sync per split.
"""
from __future__ import annotations

import os
import pickle
from typing import Dict, Optional

import torch

from . import _lib
from .engine import ChromosomeEngine
from .graph import HiCGraph, process_graph

_GRAPH_FILES: Dict = {}      # (path, mtime, device) -> {chrom: scipy csr}
_GRAPHS: Dict = {}           # (path, mtime, device, adj_type, chrom, n) -> HiCGraph
_ENGINES: Dict = {}          # id(model) -> ChromosomeEngine
_RESIDENT: Dict = {}         # (id(dict), chrom, device) -> (signature of the host tensors, panel, target)


def clear_caches() -> None:
    _GRAPH_FILES.clear()
    _GRAPHS.clear()
    _ENGINES.clear()
    _RESIDENT.clear()
    _TARGETS.clear()
    _STAGING.clear()
    _PACKED.clear()
    DEVICE_OUTPUTS.clear()


def _feature_signature(feats) -> tuple:
    """Identity of one chromosome's host tensors: object (weak reference), storage address, shape and in-place
    version of each.  A `_RESIDENT` entry is only reused while this is unchanged, so a new dict that happens to get a
    freed dict's `id()` (a second `run_model`, cross-validation folds) or features edited in place are re-uploaded."""
    import weakref
    sig = []
    for k in ("forward", "backward", "target"):
        t = feats[k]
        sig.append((weakref.ref(t), t.data_ptr(), tuple(t.shape), t._version))
    return tuple(sig)


def _signature_matches(sig, feats) -> bool:
    for (ref, ptr, shape, version), k in zip(sig, ("forward", "backward", "target")):
        t = feats[k]
        if ref() is not t or t.data_ptr() != ptr or tuple(t.shape) != shape or t._version != version:
            return False
    return True


def engine_for(model) -> ChromosomeEngine:
    e = _ENGINES.get(id(model))
    if e is None or e.model is not model:
        e = ChromosomeEngine(model, strands=2)
        _ENGINES[id(model)] = e
    return e


def graph_file(opt, split: str) -> str:
    return os.path.join(opt.graph_root, split + "_graphs_" + str(opt.hicsize) + "_" + opt.hicnorm + "norm.pkl")


def graphs_for(opt, split: str, chroms, sizes, device) -> Dict[str, HiCGraph]:
    """Device patterns for the chromosomes of a split (finetune.py:19-25,36), cached across epochs."""
    out = {}
    path, mtime, adj_dict = None, None, None
    if opt.adj_type in ("hic", "both"):
        path = graph_file(opt, split)
        mtime = os.path.getmtime(path)
    for chrom in chroms:
        key = (path, mtime, str(device), opt.adj_type, chrom, int(sizes[chrom]))
        g = _GRAPHS.get(key)
        if g is None:
            if path is not None and adj_dict is None:
                fkey = (path, mtime)
                adj_dict = _GRAPH_FILES.get(fkey)
                if adj_dict is None:
                    with open(path, "rb") as fp:
                        adj_dict = pickle.load(fp)
                    _GRAPH_FILES[fkey] = adj_dict
            g = process_graph(opt.adj_type, adj_dict, sizes[chrom], chrom, device)
            _GRAPHS[key] = g
        out[chrom] = g
    return out


_TARGETS: Dict = {}          # (id(dict), data_ptrs) -> concatenated CPU targets (they never change between epochs)
_STAGING: Dict = {}          # (device, slot) -> persistent device staging buffers of the H2D pipeline


def _staging(device, slot: int, n: int, d: int, nclass: int):
    """Device staging buffers of pipeline slot `slot`: x_f, x_r and (for soft labels only) float targets."""
    key = (str(device), slot)
    cur = _STAGING.get(key)
    if cur is None or cur[0].shape[0] < n or cur[0].shape[1] != d or cur[2].shape[1] != nclass:
        rows = max(n, cur[0].shape[0] if cur is not None and cur[0].shape[1] == d else 0)
        cur = (torch.empty(rows, d, dtype=torch.float32, device=device), torch.empty(rows, d, dtype=torch.float32, device=device),
               torch.empty(rows, nclass, dtype=torch.float32, device=device))
        _STAGING[key] = cur
    return cur[0][:n], cur[1][:n], cur[2][:n]


# What the last pass over a split left on the device: {split: (probabilities [sum N, nclass], label bit rows
# [sum N, ceil(nclass/32)] or None)}.  `runner.run_model` computes the split's AUROC / AUPR / FDR from these
# (cgcn_label_metrics) instead of from the CPU copies; valid until the next pass over the same split.
DEVICE_OUTPUTS: Dict = {}


_PACKED: Dict = {}           # id(target tensor) -> (weakref, version, pinned int32 bit rows | None for soft labels)


def packed_target(target: torch.Tensor):
    """The bit-packed pinned copy of a chromosome's 0/1 label matrix, built the first time the tensor is seen
    (`None` for soft labels, which keep the float path).  The entry is tied to the tensor object (weak reference)
    and its in-place version counter, so a recycled address or an edited matrix is packed again."""
    import weakref
    hit = _PACKED.get(id(target))
    if hit is not None and hit[0]() is target and hit[1] == target._version:
        return hit[2]
    from . import ops
    packed = ops.pack_targets(target, pin=True)
    if len(_PACKED) > 256:
        for k in [k for k, v in _PACKED.items() if v[0]() is None]:
            del _PACKED[k]
    _PACKED[id(target)] = (weakref.ref(target), target._version, packed)
    return packed


_STREAMS: Dict = {}          # device -> (h2d, d2h) copy streams, created once


def _copy_streams(device):
    key = str(device)
    st = _STREAMS.get(key)
    if st is None:
        st = (torch.cuda.Stream(device), torch.cuda.Stream(device))
        _STREAMS[key] = st
    return st


def _all_targets(chrom_feature_dict, chroms):
    key = (id(chrom_feature_dict), tuple(chrom_feature_dict[c]["target"].data_ptr() for c in chroms))
    t = _TARGETS.get(key)
    if t is None:
        t = (torch.cat([chrom_feature_dict[c]["target"].detach().cpu().float() for c in chroms], 0)
             if chroms else torch.Tensor())
        if len(_TARGETS) > 8:
            _TARGETS.clear()
        _TARGETS[key] = t
    return t


def finetune(WindowModel, ChromeModel, chrom_feature_dict, crit, optimizer, epoch, data_dict, opt, split):
    from . import ops
    from .engine import flat_params
    device = _lib.require_cuda(next(ChromeModel.parameters()).device)
    train = split == "train"
    ChromeModel.train() if train else ChromeModel.eval()
    engine = engine_for(ChromeModel)
    flat_params(ChromeModel, full=True)          # once per pass; the per-chromosome steps use the fast check
    chroms = list(chrom_feature_dict.keys())
    # Chromosome-sharded pass (one process per GPU, SURVEY.md 8(e)): `opt.shard = (schedule, rank, group)` with
    # `schedule[round][rank]` = chromosomes (dist.balanced_schedule).  This rank streams only ITS chromosomes, in
    # schedule order; in training `dist.sharded_rounds` accumulates the gradients over a round's cell and ends every
    # round with one all-reduce of the flat gradient buffer and the same optimiser step on every rank (mean gradient
    # of the round's chromosomes).
    shard = getattr(opt, "shard", None)
    if shard is not None:
        schedule, shard_rank, shard_group = shard
        cells = [[c for c in rnd[shard_rank] if c in chrom_feature_dict] for rnd in schedule]
        chroms = [c for cell in cells for c in cell]
    sizes = {c: chrom_feature_dict[c]["forward"].size(0) for c in chroms}
    nclass = ChromeModel.out.out_features
    graphs = graphs_for(opt, split, chroms, sizes, device)
    resident = bool(getattr(opt, "cache_features_on_device", False))
    pack_labels = bool(getattr(opt, "pack_labels", True))

    total_rows = sum(sizes.values())
    main = torch.cuda.current_stream(device)
    with torch.cuda.device(device):
        h2d, d2h = _copy_streams(device)
        all_preds_dev = torch.empty(total_rows, nclass, dtype=torch.float32, device=device)
        packed = ([packed_target(chrom_feature_dict[c]["target"]) for c in chroms]
                  if (pack_labels and not resident) else [None] * len(chroms))
        all_bits = all(p is not None for p in packed) and len(chroms) > 0
        # bit rows are 16 B per window: they go straight into one [sum N, words] device matrix (no staging slot)
        all_tbits_dev = (torch.empty(total_rows, (nclass + 31) // 32, dtype=torch.int32, device=device) if all_bits else None)
        offsets = [0]
        for c in chroms:
            offsets.append(offsets[-1] + sizes[c])
        all_preds = torch.empty(total_rows, nclass, dtype=torch.float32, pin_memory=True)
        losses_dev = torch.zeros(max(len(chroms), 1), dtype=torch.float32, device=device)
        # the copy streams write into buffers allocated (possibly from recycled blocks) under the compute stream:
        # order them after everything the compute stream has been given so far, and tell the allocator who else
        # touches them
        h2d.wait_stream(main)
        d2h.wait_stream(main)
        if all_tbits_dev is not None:
            all_tbits_dev.record_stream(h2d)
        all_preds_dev.record_stream(d2h)
        staged = [None, None]
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        consumed = [torch.cuda.Event(), torch.cuda.Event()]
        done = torch.cuda.Event()

        def stage(k: int):
            """Issue the H2D copies of chromosome k on the copy stream into staging slot k % 2."""
            chrom = chroms[k]
            feats = chrom_feature_dict[chrom]
            rkey = (id(chrom_feature_dict), chrom, str(device))
            if resident and rkey in _RESIDENT:
                if _signature_matches(_RESIDENT[rkey][0], feats):
                    staged[k % 2] = ("resident",) + _RESIDENT[rkey][1:]
                    return
                del _RESIDENT[rkey]                              # stale: another dict / edited features
            n, d = feats["forward"].shape
            x_f, x_r, tgt = _staging(device, k % 2, n, d, nclass)
            if all_bits:
                tgt = all_tbits_dev[offsets[k]: offsets[k + 1]]
            with torch.cuda.stream(h2d):
                if k >= 2:
                    h2d.wait_event(consumed[k % 2])          # the slot's previous tenant has been packed / consumed
                x_f.copy_(feats["forward"], non_blocking=True)
                x_r.copy_(feats["backward"], non_blocking=True)
                tgt.copy_(packed[k] if all_bits else feats["target"], non_blocking=True)
                ready[k % 2].record(h2d)
            staged[k % 2] = ("fresh", x_f, x_r, tgt)

        if chroms:
            stage(0)
        row = 0
        order = chroms
        if train and shard is not None:
            from . import dist as cdist
            totals = [sum(len(cell) for cell in rnd) for rnd in schedule]
            order = cdist.sharded_rounds(ChromeModel, optimizer, cells, totals, shard_group)
        for k, chrom in enumerate(order):
            if k + 1 < len(chroms):
                stage(k + 1)
            item = staged[k % 2]
            n = sizes[chrom]
            if item[0] == "resident":
                panel, tgt = item[1], item[2]
            else:
                main.wait_event(ready[k % 2])
                _, x_f, x_r, tgt = item
                if resident:
                    panel = ops.interleave_strands([x_f, x_r])
                    tgt = tgt.clone()
                    _RESIDENT[(id(chrom_feature_dict), chrom, str(device))] = (
                        _feature_signature(chrom_feature_dict[chrom]), panel, tgt)
                else:
                    panel = engine.pack(x_f, x_r)
            if train and shard is None:
                optimizer.zero_grad()                                    # finetune.py:39
            engine.run(graphs[chrom], panel, tgt, all_preds_dev[row: row + n], losses_dev[k: k + 1], train)
            if train and shard is None:
                optimizer.step()                                         # finetune.py:49
            consumed[k % 2].record(main)
            # predictions of this chromosome go home while the next one computes (finetune.py:52)
            d2h.wait_event(consumed[k % 2])
            with torch.cuda.stream(d2h):
                all_preds[row: row + n].copy_(all_preds_dev[row: row + n], non_blocking=True)
            row += n
        done.record(d2h)
        losses = losses_dev.cpu()                                            # the one sync of the split
        done.synchronize()
    DEVICE_OUTPUTS[split] = (all_preds_dev, all_tbits_dev)
    total_loss = float(losses.double().sum().item()) if chroms else 0
    return all_preds, _all_targets(chrom_feature_dict, chroms), total_loss
