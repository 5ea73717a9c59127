#!/usr/bin/env python
"""bench.py -- ChromeGCN chromosome-model hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload wg|c1|st] [--d-model 128|512] [--variant base|layers3|gateoff|normnone|hic1000000|hic125000]
                    [--rounds R] [--dump-outputs DIR]

Metric (BASELINE.json): "GCN train step edges/sec (GE/s)".  A step is one pass of the hot path over the workload: for
every chromosome graph, both strands through the gated GCN, BCE loss, backward, optimiser step (finetune.py:29-49).
Unit of work: one directed stored entry of A_hat = D^-1 bin(A+I), so  value = sum_c nnz(A_hat_c) / t_step / 1e9.

Workloads (BASELINE.json configs):
  wg   configs[1] / [2]: whole-genome synthetic GM12878-shaped, 23 chromosome graphs, chromosome-sharded over the ranks
       (one flat-gradient all-reduce + optimiser step per round);            <- the default, the line the metric is quoted on
  c1   configs[0]: the chr22-sized graph alone;
  st   configs[3]: ONE chromosome with 1e6 windows / ~51 M stored entries, d_model 128 or 512, row-partitioned over the
       ranks (neighbour rows over NVLink peer memory inside the kernels, BatchNorm sums and gradients all-reduced);
  --variant  configs[4]: gcn_layers 3, gate off, hicnorm '' (none), hicsize 1000000 / 125000 on the wg workload.

Keys of the JSON line beyond the base contract:
  value      inputs (graphs, feature panels, targets) resident in HBM when the timed region starts;
  e2e        the same metric through the drop-in `finetune()` with pinned HOST features: H2D of every chromosome's
             features / label bits and D2H of the predictions inside the timed region; at N > 1 the same lock-step
             rounds (all-reduce + step per round) as `value` (`opt.shard`);
  roofline   the dominant kernel (the fused GCN layer forward, cgcn_gcn_layer_fwd) timed alone with CUDA events against
             MEASURED_PEAKS.json's copy bandwidth on its ALGORITHMIC bytes, plus `time_bound_frac`: the larger of
             (compulsory bytes / HBM peak) and (algorithmic bytes / measured L2 read peak) over the launch time, and the
             standalone SpMM kernel the same way;
  cpu_baseline / --impl reference   the oracle port of the reference's PyTorch CPU path (oracle/gcn.py: torch.mm,
             torch.spmm on the un-coalesced COO tensor, host process_graph per chromosome per epoch) on the host cores;
  gpu_baseline   the same reference model with STOCK torch on this B200 (torch.spmm -> coalesce + cuSPARSE, torch.mm ->
             cuBLAS): `value` with tensors and adjacencies resident, `e2e` with the reference's own per-chromosome host
             work (process_graph, four H2D copies, loss.item(), .cpu()) -- the kernel-level bar of SURVEY.md 2b / 8(d).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "GCN train step edges/sec (GE/s)"
UNIT = "GE/s"
NCLASS = 103
DROPOUT, LR = 0.2, 0.25      # README.md:45 recipe: SGD lr 0.25, gcn_dropout 0.2
CPU_SAMPLE = ["chr19", "chr20", "chr21", "chr22"]
ST_ROWS, ST_PAIRS = 1_000_000, 25_000_000
VARIANTS = ("base", "layers3", "gateoff", "normnone", "hic1000000", "hic125000")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="wg", choices=["wg", "c1", "st"])
    # --d-model is the spelling to use under `python -m torch.distributed.run` (its own parser claims the prefix `--d`)
    ap.add_argument("--d", "--d-model", dest="d", type=int, default=128, choices=[128, 256, 512])
    ap.add_argument("--variant", default="base", choices=VARIANTS)
    ap.add_argument("--graph", default="synthetic", choices=["synthetic", "longrange", "permuted"],
                    help="locality sensitivity of the wg / c1 workloads: longrange = contact distances log-uniform over the "
                         "whole chromosome instead of <= 2000 bins; permuted = the synthetic graph with its windows "
                         "relabelled at random (same degrees, no locality at all)")
    ap.add_argument("--rounds", type=int, default=0, help="optimiser steps per pass at N > 1 (0 = default schedule)")
    ap.add_argument("--st-rows", type=int, default=ST_ROWS)
    ap.add_argument("--st-pairs", type=int, default=ST_PAIRS)
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--gemm-impl", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (probabilities of a fixed row sample, "
                         "losses, model state) as DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the GPU path; the reference arm has nothing to dump")
    return args


DUMP_PROB_BYTES = 32 << 20       # probabilities --dump-outputs writes per run, spread over the workload's graphs


def dump_rows(n, n_graphs, seed):
    """Sorted row indices of the fixed sample of an n-row probability matrix that --dump-outputs writes."""
    import numpy as np
    k = max(1, DUMP_PROB_BYTES // (4 * NCLASS * n_graphs))
    return np.arange(n) if n <= k else np.sort(np.random.default_rng(seed).choice(n, k, replace=False))


def dump_outputs(out_dir, torch, arrays):
    """Write host copies of the given tensors as out_dir/<name>.npy: float64 stays float64, the rest becomes float32."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().cpu()
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy() if t.dtype == torch.float64 else t.float().numpy())


def last_step_losses(acc):
    """--dump-outputs: the loss slots accumulate (`+=`) over every pass.  `before()` runs right before the last timed
    step and zeroes them; `after()` then returns exactly that step's losses and adds the earlier sum back (one fp32
    add per slot, so the running sum ends bit-identical to a run without the dump)."""
    prior = []

    def before():
        prior.append(acc.clone())
        acc.zero_()

    def after():
        last = acc.clone()
        acc.add_(prior[0])
        return last
    return before, after


def dump_model_state(out_dir, torch, model):
    dump_outputs(out_dir, torch, {"model." + k: v.double() if v.dtype == torch.int64 else v
                                  for k, v in model.state_dict().items()})


def variant_cfg(args):
    """(layers, gate, extended, hic_edges, use_norm) of a variant-sweep point (BASELINE.json configs[4])."""
    v = args.variant
    layers, gate, extended = (3, True, True) if v == "layers3" else ((2, False, True) if v == "gateoff" else (2, True, False))
    hic = 1000000 if v == "hic1000000" else (125000 if v == "hic125000" else 500000)
    return layers, gate, extended, hic, v != "normnone"


def workload_chroms(name):
    from chromegcn_b200 import synthetic
    return ["chr22"] if name == "c1" else list(synthetic.WHOLE_GENOME)


def permute_pattern(indptr, indices, seed):
    """P A P^T of a CSR pattern for a random relabelling P of the windows: degrees and entry count unchanged, every
    neighbour row a random one (the worst case for the gather kernels' cache reuse)."""
    import numpy as np
    from scipy import sparse
    n = indptr.shape[0] - 1
    a = sparse.csr_matrix((np.ones(indices.shape[0], dtype=np.float32), indices, indptr), shape=(n, n))
    p = np.random.default_rng(seed).permutation(n)
    a = a[p][:, p].tocsr()
    a.sort_indices()
    return a.indptr.astype(np.int32), a.indices.astype(np.int32)


def workload_name(args):
    if args.workload == "st":
        return ("ST: one synthetic chromosome, N=%d windows, %d undirected pairs (~%d M stored entries), d_model %d, "
                "row-partitioned" % (args.st_rows, args.st_pairs, (2 * args.st_pairs + args.st_rows) // 1000000, args.d))
    base = ("C1: one chr22-sized graph (N=20000)" if args.workload == "c1" else
            "WG: whole-genome synthetic GM12878-shaped, 23 chromosome graphs (sum N ~1.18M)")
    _, _, _, hic, use_norm = variant_cfg(args)
    graph = {"synthetic": "", "longrange": ", contact distances log-uniform over the whole chromosome",
             "permuted": ", windows relabelled at random (no locality)"}[args.graph]
    return "%s, hicsize %d, hicnorm %s, variant %s%s" % (base, hic, "SQRTVC" if use_norm else "'' (none)", args.variant, graph)


def build_inputs(chrom, hic_edges, use_norm, longrange=False):
    """Synthetic Hi-C inputs of one chromosome in the form the adjacency build takes.  hicnorm '' mode (--norm ''): no
    norm vector and the contact list pre-sorted by value, descending (data/extras/sort_hic.py:36-38; ties in file order)."""
    import numpy as np
    from chromegcn_b200 import synthetic
    if longrange:
        h = synthetic.make_hic(chrom, hic_edges=hic_edges, max_dist_bins=synthetic.HG19_LENGTHS[chrom] // synthetic.BIN_BP - 1)
    else:
        h = synthetic.make_hic(chrom, hic_edges=hic_edges)
    if use_norm:
        return h.window_starts, h.bin1, h.bin2, h.val, h.norm
    order = np.argsort(-h.val, kind="stable")
    return h.window_starts, h.bin1[order], h.bin2[order], h.val[order], None


# ---------------------------------------------------------------------------------------- CPU (oracle port)
def _oracle_model(args, torch, ogcn):
    layers, gate, extended, _, _ = variant_cfg(args)
    torch.manual_seed(0)
    if extended:
        return ogcn.ChromeGCNExtOracle(args.d, args.d, NCLASS, DROPOUT, gate, layers)
    return ogcn.ChromeGCNOracle(args.d, args.d, NCLASS, DROPOUT, True, layers)


def cpu_reference_run(args, chroms, steps, warmup, threads=None):
    """The reference's CPU path restated (oracle/gcn.py), timed on the host: per step one pass over `chroms`
    exactly as finetune.py does it (process_graph on the host for every chromosome every pass, two
    forward calls, BCE, backward, SGD)."""
    import torch
    from chromegcn_b200 import synthetic
    from oracle import adjacency as oadj
    from oracle import gcn as ogcn
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    _, _, _, hic, use_norm = variant_cfg(args)
    graphs, feats, edges = {}, {}, 0
    for c in chroms:
        w, b1, b2, v, nv = build_inputs(c, hic, use_norm)
        ip, ix = (oadj.build_adjacency_numpy(w, b1, b2, v, nv, 1, hic) if use_norm else
                  oadj.build_adjacency_numpy(w, b1, b2, v, None, 1, hic))
        graphs[c] = (ip, ix)
        feats[c] = synthetic.make_features(c, ip.shape[0] - 1, args.d, NCLASS)
        edges += int(ip[-1]) + ip.shape[0] - 1
    model = _oracle_model(args, torch, ogcn)
    opt = ogcn.make_optimizer(model, "sgd", LR)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        ogcn.finetune_epoch(model, feats, graphs, opt, "train")
        times.append(time.perf_counter() - t0)
    dt = sum(times[warmup:]) / max(steps, 1)
    return edges / dt / 1e9, dt, edges, threads


def run_reference_arm(args):
    """`--impl reference`: the reference's own CPU implementation of the path (the oracle port: the reference is a flat
    Python script repo, nothing to compile into oracle/_ref) on all host cores, on the SAME workload and variant as
    the GPU arm.  The whole-genome pass costs ~10 s per step on 16 threads; if one warm-up pass shows that K steps would
    not fit CGCN_REF_BUDGET_S (default 900 s) the arm falls back to the 4-chromosome sample and says so."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps
    chroms = ["chr22"] if args.workload == "c1" else (CPU_SAMPLE if args.workload == "st" else workload_chroms("wg"))
    budget = float(os.environ.get("CGCN_REF_BUDGET_S", "900"))
    same_config = args.workload != "st"
    warmup = 1                                    # a CPU pass has no clocks or caches worth more than one warm-up pass
    if args.workload == "wg":
        t0 = time.perf_counter()
        _, dt1, _, _ = cpu_reference_run(args, CPU_SAMPLE, 1, 0)
        est = dt1 * 8.0 * (steps + warmup) + 40.0  # the 4 smallest chromosomes are ~1/8 of the genome's stored entries + rows
        if est > budget:
            chroms, same_config = CPU_SAMPLE, False
    value, dt, edges, threads = cpu_reference_run(args, chroms, steps, warmup)
    sample = "one pass over %s (%d stored entries) per step, oracle port of the reference PyTorch CPU path incl. host " \
             "process_graph per chromosome" % ("all 23 chromosomes" if len(chroms) == 23 else "+".join(chroms), edges)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args), "sample": sample, "same_config": same_config, "d_model": args.d,
                       "nclass": NCLASS, "optim": "sgd", "variant": args.variant},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------- stock torch on the GPU
def gpu_stock_torch_run(args, chroms, dev, steps=5, warmup=2):
    """The reference model (oracle restatement: same torch calls as models/ChromeModels.py / models/SubLayers.py) on
    this GPU with stock PyTorch kernels.  Returns (resident GE/s, e2e GE/s, edges): `resident` keeps features and the
    sparse adjacency tensors on the device (kernels only: coalesce + cuSPARSE SpMM, cuBLAS, ATen element-wise);
    `e2e` is the reference's loop as written -- process_graph on the host, .cuda() copies, loss.item(), .cpu() per
    chromosome (finetune.py:29-53)."""
    import torch
    from chromegcn_b200 import synthetic
    from oracle import adjacency as oadj
    from oracle import gcn as ogcn
    _, _, _, hic, use_norm = variant_cfg(args)
    graphs, feats, edges = {}, {}, 0
    for c in chroms:
        w, b1, b2, v, nv = build_inputs(c, hic, use_norm)
        ip, ix = oadj.build_adjacency_numpy(w, b1, b2, v, nv, 1, hic)
        graphs[c] = (ip, ix)
        feats[c] = synthetic.make_features(c, ip.shape[0] - 1, args.d, NCLASS)
        edges += int(ip[-1]) + ip.shape[0] - 1
    model = _oracle_model(args, torch, ogcn).to(dev).train()
    opt = ogcn.make_optimizer(model, "sgd", LR)

    def pass_resident(adjs, fd):
        for c in chroms:
            f = fd[c]
            ogcn.chromosome_step(model, f["forward"], f["backward"], f["target"], adjs[c], opt, True, input_grads=True)

    def pass_e2e():
        for c in chroms:
            f = feats[c]
            adj = ogcn.coo_adjacency(*graphs[c]).to(dev)                               # finetune.py:36
            loss, prob, _, _ = ogcn.chromosome_step(model, f["forward"].to(dev), f["backward"].to(dev), f["target"].to(dev),
                                                    adj, opt, True, input_grads=True)  # .item() inside
            prob.cpu()                                                                 # finetune.py:52
    adjs = {c: ogcn.coo_adjacency(*graphs[c]).to(dev) for c in chroms}
    fd = {c: {k: v.to(dev) for k, v in feats[c].items()} for c in chroms}
    out = []
    for fn in (lambda: pass_resident(adjs, fd), pass_e2e):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        torch.cuda.synchronize(dev)
        out.append(edges / ((time.perf_counter() - t0) / steps) / 1e9)
    return out[0], out[1], edges


# ---------------------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None
        self.load0 = time.monotonic()

    def mark_begin(self):
        self.t0 = time.monotonic()

    def mark_end(self):
        self.t1 = time.monotonic()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.monotonic(), line.strip()))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        # nvidia-smi needs ~1 s to come up, so it is started before the data is built and its rows are
        # time-stamped: the reported samples are the ones that fall inside the timed region (plus one
        # sampling period of slack either side, the loop period being 20 ms).
        rows = self.rows
        window = "timed region"
        if self.t0 is not None and self.t1 is not None:
            rows = [(t, r) for t, r in self.rows if self.t0 - 0.02 <= t <= self.t1 + 0.02]
            if not rows:      # region shorter than one sampling period: fall back to the warm-up + timed load window
                rows = [(t, r) for t, r in self.rows if self.load0 - 0.02 <= t <= self.t1 + 0.02]
                window = "warm-up + timed region (timed region shorter than one 20 ms sample)"
        sm, mx, reasons = [], [], set()
        for _, r in rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        hbm, src = float(json.load(open(path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        hbm, src = 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"
    l2, l2src = None, None
    lp = os.path.join(ROOT, "profiles", "r02_l2_bw.json")
    if os.path.exists(lp):
        l2, l2src = float(json.load(open(lp))["l2_read_peak_GBs"]), "profiles/r02_l2_bw.json (tools/l2_bw.py, measured on this pool)"
    return hbm, src, l2, l2src


def time_launches(torch, fn, items, reps=5):
    """One CUDA-event pair around a back-to-back pass over `items` (no host round trip between launches)."""
    for _ in range(3):
        for it in items:
            fn(it)
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for it in items:
            fn(it)
        b.record()
        b.synchronize()
        tot += a.elapsed_time(b)
    return tot / reps * 1e-3 / len(items)          # seconds per launch


def roofline_block(args, torch, ops, graphs, panels, names, model):
    """The fused GCN layer forward (dominant kernel of the pass) and the standalone SpMM, each timed alone."""
    hbm, hbm_src, l2, l2_src = peaks()
    d = args.d
    W = 2 * d
    n_tot = sum(graphs[c].n for c in names)
    nnz_tot = sum(graphs[c].nnz for c in names)
    k = len(names)
    out = {"bound": "hbm", "peak": hbm, "unit": "GB/s", "peak_source": hbm_src, "l2_read_peak": l2, "l2_peak_source": l2_src}
    # ---- standalone SpMM (forward mean aggregation): nnz*(4+4W) + 4(N+1) + 4WN algorithmic, 4nnz + 4(N+1) + 8WN compulsory
    outs = {c: torch.empty_like(panels[c]) for c in names}
    t = time_launches(torch, lambda c: ops.spmm(graphs[c], panels[c].view(graphs[c].n, W), True, out=outs[c].view(graphs[c].n, W)), names)
    alg = (nnz_tot * (4 + 4 * W) + 4 * (n_tot + k) + 4 * W * n_tot) / k
    comp = (4 * nnz_tot + 4 * (n_tot + k) + 8 * W * n_tot) / k
    spmm = {"kernel": "spmm_pattern_kernel<%d> (width %d)" % (W // 128, W), "avg_launch_us": t * 1e6, "algorithmic_bytes_per_launch": alg,
            "compulsory_bytes_per_launch": comp, "achieved": alg / t / 1e9, "frac": alg / t / 1e9 / hbm,
            "compulsory_frac": comp / t / 1e9 / hbm}
    if l2:
        spmm["time_bound_frac"] = max(comp / (hbm * 1e9), alg / (l2 * 1e9)) / t
    del outs
    if d == 128:
        # ---- fused layer forward: gather (as the SpMM) + x re-read for the blend + three panels written (sx, z, x') + g
        p0 = dict(model.named_parameters())
        wts = (p0["GC1.weight"].detach(), p0["GC1.bias"].detach(), p0["W1.weight"].detach().reshape(-1), p0["W1.bias"].detach())
        t = time_launches(torch, lambda c: ops.gcn_layer_fwd(graphs[c], panels[c], wts[0], wts[1], wts[2], wts[3], dropout_p=DROPOUT,
                                                            seed=1, step=1, site=0), names)
        alg = (nnz_tot * (4 + 4 * W) + 4 * (n_tot + k) + 4 * 4 * W * n_tot + 8 * n_tot) / k
        comp = (4 * nnz_tot + 4 * (n_tot + k) + 4 * 4 * W * n_tot + 8 * n_tot) / k
        out.update({"kernel": "fused_layer_kernel<2, FWD> (cgcn_gcn_layer_fwd: gather + tcgen05 3xTF32 + gate epilogue, width %d)" % W,
                    "avg_launch_us": t * 1e6, "algorithmic_bytes_per_launch": alg, "compulsory_bytes_per_launch": comp,
                    "achieved": alg / t / 1e9, "frac": alg / t / 1e9 / hbm, "compulsory_frac": comp / t / 1e9 / hbm,
                    "includes": "3 output allocations per launch by the Python wrapper are outside the event pair's kernels"})
        if l2:
            out["time_bound_frac"] = max(comp / (hbm * 1e9), alg / (l2 * 1e9)) / t
    else:
        out.update({k2: spmm[k2] for k2 in ("kernel", "avg_launch_us", "algorithmic_bytes_per_launch", "compulsory_bytes_per_launch",
                                            "achieved", "frac", "compulsory_frac")})
        if "time_bound_frac" in spmm:
            out["time_bound_frac"] = spmm["time_bound_frac"]
    out["spmm"] = spmm
    traffic, tsrc = None, None
    tpath = os.path.join(ROOT, "profiles", "r02_fused_traffic.json")
    if args.workload == "wg" and args.variant == "base" and d == 128 and os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic, tsrc = tj["dram_bytes_per_launch"], "profiles/r02_fused_traffic.json (ncu dram__bytes_read.sum + dram__bytes_write.sum, mean of %d launches)" % tj["launches"]
    out["traffic"], out["traffic_source"] = traffic, tsrc
    out["note"] = ("algorithmic bytes: every gathered neighbour row counted (nnz*(4+4W)); compulsory bytes: every panel row once. "
                   "Hi-C graphs are near-diagonal, so most gathers are served by L1 / L2 and `frac` (algorithmic bytes over the "
                   "DRAM copy peak) can exceed 1; `compulsory_frac` is the DRAM-side fraction and `time_bound_frac` the fraction of "
                   "the L2 / HBM time bound -- the honest distance to the roofline")
    return out


# ---------------------------------------------------------------------------------------- GPU arm: wg / c1
def run_chromosomes(args, torch, dist, dev, world, rank, sampler):
    import numpy as np
    from chromegcn_b200 import _lib, ops, synthetic
    from chromegcn_b200 import dist as cdist
    from chromegcn_b200 import finetune as ft
    from chromegcn_b200.chrome_models import ChromeGCN
    from chromegcn_b200.engine import ChromosomeEngine
    from chromegcn_b200.graph import HiCGraph
    from chromegcn_b200.optim import FlatSGD
    steps, warmup = args.steps, max(args.warmup, 3)
    layers, gate, extended, hic, use_norm = variant_cfg(args)
    D = args.d
    chroms = workload_chroms(args.workload)
    sizes = {c: synthetic.num_windows(c) for c in chroms}
    costs = {c: cdist.chromosome_cost(sizes[c], hic + sizes[c]) for c in chroms}
    schedule = cdist.balanced_schedule(costs, world, args.rounds if args.rounds > 0 else None)
    shards = cdist.schedule_shards(schedule, world)
    mine = shards[rank]
    graphs, feats_host, panels, targets, probs = {}, {}, {}, {}, {}
    local_edges = 0
    for c in mine:
        w, b1, b2, v, nv = build_inputs(c, hic, use_norm, args.graph == "longrange")
        ip, ix = ops.adjacency_build(w, b1, b2, v, nv, 1, hic, dev)          # the product's own build (cgcn_adj_build)
        if args.graph == "permuted":
            ip, ix = permute_pattern(ip, ix, 4000 + synthetic.chrom_index(c))
        graphs[c] = HiCGraph.from_csr_pattern(ip, ix, dev, name=c)
        n = graphs[c].n
        f = synthetic.make_features(c, n, D, NCLASS)
        feats_host[c] = {k: t.pin_memory() for k, t in f.items()}
        panels[c] = ops.interleave_strands([f["forward"].to(dev), f["backward"].to(dev)])
        targets[c] = ops.pack_targets(f["target"]).to(dev)      # label bit rows, the form finetune() feeds the loss kernel
        probs[c] = torch.empty(n, NCLASS, device=dev)
        local_edges += graphs[c].nnz
    edges_t = torch.tensor([local_edges], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(edges_t)
    total_edges = float(edges_t.item())

    torch.manual_seed(0)
    model = ChromeGCN(D, D, NCLASS, DROPOUT, gate, layers, extended=extended).to(dev)
    model.gemm_impl = args.gemm_impl
    model.train()
    if world > 1:
        for p in model.parameters():
            dist.broadcast(p.data, 0)
    engine = ChromosomeEngine(model, 2)
    optimizer = FlatSGD(model, lr=LR)
    losses = torch.zeros(max(len(mine), 1), device=dev)

    def one_step():
        cdist.sharded_train_epoch(engine, optimizer, schedule, rank, graphs, panels, targets, probs, losses)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    before_last, after_last = last_step_losses(losses)
    ms_per_step, launches = timed_region(torch, dist, dev, world, sampler, one_step, barrier, steps, warmup, _lib,
                                         before_last if args.dump_outputs else None)
    value = total_edges / (ms_per_step * 1e-3) / 1e9
    last_losses = after_last() if args.dump_outputs else None
    final_loss = float(losses.sum().item())
    if args.dump_outputs:
        # before the e2e passes below train the model further; each rank writes its own chromosomes
        order = [c for rnd in schedule for c in rnd[rank]]          # losses[i] belongs to order[i]
        out = {}
        for i, c in enumerate(order):
            rows = torch.from_numpy(dump_rows(graphs[c].n, len(chroms), synthetic.chrom_index(c))).to(dev)
            out["probs." + c] = probs[c].index_select(0, rows)
            out["loss." + c] = last_losses[i: i + 1]
        dump_outputs(args.dump_outputs, torch, out)
        if rank == 0:
            dump_model_state(args.dump_outputs, torch, model)

    # ---- e2e: drop-in finetune() with pinned host features, H2D/D2H inside the timed region, the same rounds at N > 1
    e2e = None
    if not args.no_e2e:
        import pickle
        import tempfile
        from scipy import sparse
        tmp = tempfile.mkdtemp(prefix="cgcn_bench_")
        gdict = {}
        for c in mine:
            rp, ci = graphs[c].csr_numpy()
            n = graphs[c].n
            rows = np.repeat(np.arange(n), np.diff(rp))
            keep = rows != ci                                  # the pickles hold A without self loops
            gdict[c] = sparse.csr_matrix((np.ones(int(keep.sum())), (rows[keep], ci[keep])), shape=(n, n))
        norm_tag = "SQRTVC" if use_norm else ""
        with open(os.path.join(tmp, "train_graphs_%d_%snorm.pkl" % (hic, norm_tag)), "wb") as fp:
            pickle.dump(gdict, fp)
        opt_ns = argparse.Namespace(adj_type="hic", graph_root=tmp, hicsize=str(hic), hicnorm=norm_tag)
        if world > 1:
            opt_ns.shard = (schedule, rank, None)
        # per pass: both strands' fp32 features + the labels as bit rows (16 B per window; finetune() packs the 0/1
        # label matrix once, on first sight, during the untimed warm-up passes)
        h2d = sum(2 * sizes[c] * D * 4 + sizes[c] * ((NCLASS + 31) // 32) * 4 for c in mine)
        d2h = sum(sizes[c] * NCLASS * 4 for c in mine) + 4 * len(mine)
        for _ in range(2):
            ft.finetune(None, model, feats_host, None, optimizer, 0, None, opt_ns, "train")
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            ft.finetune(None, model, feats_host, None, optimizer, 0, None, opt_ns, "train")
        barrier()
        dt = torch.tensor([(time.perf_counter() - t0) / steps], dtype=torch.float64, device=dev)
        bytes_t = torch.tensor([h2d, d2h], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            dist.all_reduce(bytes_t)
        e2e = {"value": total_edges / float(dt.item()) / 1e9, "unit": UNIT, "h2d_bytes_per_step": int(bytes_t[0].item()),
               "d2h_bytes_per_step": int(bytes_t[1].item()), "ms_per_step": float(dt.item()) * 1e3,
               "note": "finetune() drop-in, pinned host features (fp32) and bit-packed 0/1 labels copied H2D every pass, predictions "
                       "copied D2H every pass; " + ("one optimiser step per chromosome" if world == 1 else
                                                     "the same lock-step rounds as `value`: gradient all-reduce + optimiser step per "
                                                     "round, BatchNorm buffers synchronised per pass (opt.shard)")}

    roofline = None
    if rank == 0 and not args.no_roofline:
        try:
            roofline = roofline_block(args, torch, ops, graphs, panels, mine, model)
        except Exception as exc:      # rank-0-only, no collective inside: a failure here must not cost the main line
            import traceback
            traceback.print_exc()
            roofline = {"bound": "hbm", "error": "%s: %s" % (type(exc).__name__, exc)}
    config = {"workload": workload_name(args), "d_model": D, "gcn_layers": layers, "nclass": NCLASS, "gate": gate, "adj_type": "hic",
              "hicnorm": "SQRTVC" if use_norm else "", "hicsize": hic, "variant": args.variant, "graph": args.graph, "optim": "sgd", "gcn_dropout": DROPOUT,
              "strands": 2, "total_stored_entries": total_edges,
              "parallelism": "chromosome-sharded x%d, %d lock-step round(s) per pass (balanced packing, gradient accumulation inside "
                             "a rank's cell), one flat-gradient allreduce + optimiser step per round" % (world, len(schedule)),
              "l2": "inputs larger than L2 (126 MB): %.2f GB of resident feature panels + targets cycled per step" % (
                  sum(sizes[c] for c in chroms) * (2 * D * 4 + NCLASS * 4) / 1e9),
              "gemm_impl": args.gemm_impl, "fused_layers": os.environ.get("CGCN_NO_FUSED") is None and D == 128,
              "final_loss_sum": final_loss}
    return value, ms_per_step, launches, e2e, roofline, config, "strong"


def timed_region(torch, dist, dev, world, sampler, one_step, barrier, steps, warmup, _lib, before_last=None):
    sampler.load0 = time.monotonic()
    for _ in range(warmup):
        one_step()
    barrier()
    launches0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.mark_begin()
    ev0.record()
    torch.cuda.nvtx.range_push("timed")
    for i in range(steps):
        if before_last is not None and i == steps - 1:
            before_last()
        one_step()
    torch.cuda.nvtx.range_pop()
    ev1.record()
    barrier()
    sampler.mark_end()
    ms = ev0.elapsed_time(ev1)
    launches = _lib.launch_count() - launches0
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    lt = torch.tensor([launches], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
    return float(t.item()) / steps, int(lt.item())


# ---------------------------------------------------------------------------------------- GPU arm: st (row-partitioned)
def run_stress(args, torch, dist, dev, world, rank, sampler):
    from scipy import sparse
    from chromegcn_b200 import _lib, ops, synthetic
    from chromegcn_b200 import dist as cdist
    from chromegcn_b200.chrome_models import ChromeGCN
    from chromegcn_b200.graph import HiCGraph
    from chromegcn_b200.optim import FlatSGD
    steps, warmup = args.steps, max(args.warmup, 3)
    D, n = args.d, args.st_rows
    a = synthetic.make_pattern_direct(n, args.st_pairs, seed=77)
    a = (a + sparse.eye(n, format="csr")).tocsr()
    a.sort_indices()
    parts = cdist.row_partition(n, world)
    b, e = parts[rank]
    lp, lc = cdist.local_rows_csr(a.indptr, a.indices, b, e)
    total_edges = float(a.nnz)
    g = HiCGraph.from_csr_pattern(lp, lc, dev, add_selfloops=False)
    del a
    torch.manual_seed(0)
    model = ChromeGCN(D, D, NCLASS, DROPOUT, True, 2).to(dev).train()
    model.gemm_impl = args.gemm_impl
    if world > 1:
        for p in model.parameters():
            dist.broadcast(p.data, 0)
    opt = FlatSGD(model, lr=LR)
    step = cdist.RowPartitionedStep(model, g, parts, rank, 2, exchange=args.exchange)
    gen = torch.Generator().manual_seed(100 + rank)
    host = {"forward": torch.randn(e - b, D, generator=gen).pin_memory(), "backward": torch.randn(e - b, D, generator=gen).pin_memory(),
            "target": (torch.rand(e - b, NCLASS, generator=gen) < 0.05).float().pin_memory()}
    panel = ops.interleave_strands([host["forward"].to(dev), host["backward"].to(dev)])
    tgt = host["target"].to(dev)
    probs = torch.empty(e - b, NCLASS, device=dev)
    loss = torch.zeros(1, device=dev)

    def one_step():
        step.run(panel, tgt, loss, train=True, probs_out=probs)
        opt.step()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    before_last, after_last = last_step_losses(loss)
    ms_per_step, launches = timed_region(torch, dist, dev, world, sampler, one_step, barrier, steps, warmup, _lib,
                                         before_last if args.dump_outputs else None)
    value = total_edges / (ms_per_step * 1e-3) / 1e9
    if args.dump_outputs:
        # before the e2e steps below; the loss and the model state are the same on every rank, the probability budget
        # is split over the ranks' row blocks
        last_loss = after_last()
        name = "probs.st" if world == 1 else "probs.st.rank%d" % rank
        rows = torch.from_numpy(dump_rows(e - b, world, rank)).to(dev)
        dump_outputs(args.dump_outputs, torch, {name: probs.index_select(0, rows)})
        if rank == 0:
            dump_outputs(args.dump_outputs, torch, {"loss.st": last_loss})
            dump_model_state(args.dump_outputs, torch, model)

    e2e = None
    if not args.no_e2e:
        xf, xr, tg = torch.empty(e - b, D, device=dev), torch.empty(e - b, D, device=dev), torch.empty(e - b, NCLASS, device=dev)
        probs_host = torch.empty(e - b, NCLASS).pin_memory()

        def e2e_step():
            xf.copy_(host["forward"], non_blocking=True)
            xr.copy_(host["backward"], non_blocking=True)
            tg.copy_(host["target"], non_blocking=True)
            p = ops.interleave_strands([xf, xr], out=panel)
            step.run(p, tg, loss, train=True, probs_out=probs)
            opt.step()
            probs_host.copy_(probs, non_blocking=True)
        for _ in range(2):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            e2e_step()
        barrier()
        dt = torch.tensor([(time.perf_counter() - t0) / steps], dtype=torch.float64, device=dev)
        bytes_t = torch.tensor([(e - b) * (2 * D + NCLASS) * 4, (e - b) * NCLASS * 4 + 4], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            dist.all_reduce(bytes_t)
        e2e = {"value": total_edges / float(dt.item()) / 1e9, "unit": UNIT, "h2d_bytes_per_step": int(bytes_t[0].item()),
               "d2h_bytes_per_step": int(bytes_t[1].item()), "ms_per_step": float(dt.item()) * 1e3,
               "note": "RowPartitionedStep.run with this rank's pinned host feature rows / float labels copied H2D and its "
                       "probabilities copied D2H every step"}
    roofline = None
    if rank == 0 and not args.no_roofline:
        try:
            roofline = roofline_block(args, torch, ops, {"st": g}, {"st": panel}, ["st"], model) if world == 1 else None
        except Exception as exc:
            import traceback
            traceback.print_exc()
            roofline = {"bound": "hbm", "error": "%s: %s" % (type(exc).__name__, exc)}
    final_loss = float(loss.item())
    step.close()
    config = {"workload": workload_name(args), "d_model": D, "gcn_layers": 2, "nclass": NCLASS, "gate": True, "optim": "sgd",
              "gcn_dropout": DROPOUT, "strands": 2, "total_stored_entries": total_edges,
              "parallelism": "one graph row-partitioned x%d (contiguous row blocks), exchange=%s: %s; BatchNorm column sums, loss and "
                             "the flat gradient buffer all-reduced over NCCL" % (
                                 world, args.exchange, "neighbour rows loaded over NVLink from the owners' exchange buffers inside "
                                 "the gather kernels" if args.exchange == "peer" else "NCCL all-gather of the gathered panel per layer"),
              "l2": "inputs larger than L2: %.2f GB feature panel per rank" % ((e - b) * 2 * D * 4 / 1e9),
              "gemm_impl": args.gemm_impl, "fused_layers": os.environ.get("CGCN_NO_FUSED") is None and D == 128,
              "accumulated_loss": final_loss}
    return value, ms_per_step, launches, e2e, roofline, config, "strong"


# ---------------------------------------------------------------------------------------- main
def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return
    import torch
    import torch.distributed as dist
    from chromegcn_b200 import _lib, hostbind

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    _lib.require_cuda()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    binding = hostbind.bind_to_gpu(local_rank)      # before any pinned allocation (first touch decides the NUMA node)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()            # started here so that nvidia-smi is already looping when the timed region begins
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    runner = run_stress if args.workload == "st" else run_chromosomes
    value, ms_per_step, launches, e2e, roofline, config, scaling = runner(args, torch, dist, dev, world, rank, sampler)
    clocks = sampler.stop() if rank == 0 else None
    config["host_binding_rank0"] = binding
    hostbind.unbind(binding)       # the CPU baseline gets every host core back
    cpu_baseline = gpu_baseline = None
    if rank == 0 and not args.no_gpu_baseline:
        try:
            names = ["chr22"] if args.workload != "wg" else CPU_SAMPLE
            res, ee, edges = gpu_stock_torch_run(args, names, dev)
            gpu_baseline = {"value": res, "e2e": ee, "unit": UNIT, "kind": "port",
                            "sample": "%s (%d stored entries): the reference model (oracle restatement, same torch calls) with stock "
                                      "torch %s kernels on this GPU -- torch.spmm (coalesce + cuSPARSE) / torch.mm (cuBLAS); `value` "
                                      "with tensors and adjacencies resident, `e2e` the reference loop as written (host process_graph, "
                                      ".cuda() copies, loss.item(), .cpu() per chromosome)" % ("+".join(names), edges, torch.__version__)}
        except Exception as exc:
            gpu_baseline = {"error": "%s: %s" % (type(exc).__name__, exc)}
    if rank == 0 and not args.no_cpu_baseline:
        v, dt_cpu, e_cpu, threads = cpu_reference_run(args, ["chr22"], steps=10, warmup=2)
        cpu_baseline = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": "10 train steps on the chr22-sized graph (N=20000, %d stored entries), %.3f s/step; "
                                  "oracle port of the reference PyTorch CPU path incl. host process_graph" % (e_cpu, dt_cpu)}
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling,
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config, "e2e": e2e,
                "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline,
                "gpu_baseline": gpu_baseline}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
