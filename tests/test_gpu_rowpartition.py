"""GPU: one graph row-partitioned over ranks (cgcn_model_phase + exchange steps) equals the single-GPU step.

* world_size 1 (always runs): the stage-by-stage path with identity collectives must reproduce
  `ChromosomeEngine.run` bit for bit -- it is the same kernels in the same order;
* world_size 2 (needs two GPUs, NCCL): contiguous row blocks, all-gather of the SpMM input panels, all-reduce of
  the BatchNorm sums and of the flat gradient buffer; logits, loss and every gradient within 1e-5 of the
  single-GPU result (only summation order differs)."""
import os
import socket

import numpy as np
import pytest
import torch

from oracle import adjacency as oadj
from oracle import gcn as ogcn

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _case(device, dropout=0.0):
    from chromegcn_b200.chrome_models import ChromeGCN
    z = np.load(os.path.join(GOLDEN, "model_l2_stress.npz"))
    sd = {k[4:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd0.")}
    m = ChromeGCN(128, 128, sd["out.weight"].shape[0], dropout, True, 2)
    m.load_state_dict(sd)
    m = m.to(device).train()
    rp, ci = oadj.pattern_with_selfloops(z["indptr"], z["indices"])
    return z, m, rp, ci


def _single_gpu_reference(device, dropout=0.0, input_grad=True):
    from chromegcn_b200.engine import ChromosomeEngine
    from chromegcn_b200.graph import HiCGraph
    z, m, rp, ci = _case(device, dropout)
    g = HiCGraph.from_csr_pattern(rp, ci, device, add_selfloops=False)
    eng = ChromosomeEngine(m, 2)
    panel = eng.pack(torch.from_numpy(z["x_f"]).to(device), torch.from_numpy(z["x_r"]).to(device)).clone()
    loss = torch.zeros(1, device=device)
    xg = torch.empty_like(panel) if input_grad else None
    out, _ = eng.run(g, panel, torch.from_numpy(z["target"]).to(device), None, loss, train=True, input_grad=xg)
    return (out.clone(), loss.clone(), {k: p.grad.clone() for k, p in m.named_parameters()}, xg,
            m.batch_norm.running_var.clone())


def _partitioned(device, rank, world, dropout=0.0, input_grad=True, group=None, exchange="nccl"):
    from chromegcn_b200 import dist as cdist
    from chromegcn_b200.graph import HiCGraph
    from chromegcn_b200 import ops
    z, m, rp, ci = _case(device, dropout)
    n = rp.shape[0] - 1
    parts = cdist.row_partition(n, world)
    b, e = parts[rank]
    lp, lc = cdist.local_rows_csr(rp, ci, b, e)
    g = HiCGraph.from_csr_pattern(lp, lc, device, add_selfloops=False)
    step = cdist.RowPartitionedStep(m, g, parts, rank, 2, group, exchange=exchange)
    panel = ops.interleave_strands([torch.from_numpy(z["x_f"][b:e]).to(device), torch.from_numpy(z["x_r"][b:e]).to(device)])
    loss = torch.zeros(1, device=device)
    xg = torch.empty_like(panel) if input_grad else None
    out, _ = step.run(panel, torch.from_numpy(z["target"][b:e]).to(device), loss, train=True, input_grad=xg)
    if exchange == "peer":
        assert step.peer.exchanges == 4          # x_in, layer-1 output, t of layer 2, t of layer 1 (input gradients)
        out = out.clone()
        torch.cuda.synchronize(device)
        step.close()
    return out, loss, {k: p.grad for k, p in m.named_parameters()}, xg, m.batch_norm.running_var, (b, e)


def _hub_graph(n=3000, hub_row=1500, hub_deg=700):
    """Near-diagonal pattern of bin(A + I) in which row `hub_row` has `hub_deg` neighbours drawn from all rows."""
    rng = np.random.default_rng(11)
    i = rng.integers(0, n, n * 8)
    j = np.clip(i + rng.integers(-30, 31, n * 8), 0, n - 1)
    i = np.concatenate([i, np.full(hub_deg, hub_row)])
    j = np.concatenate([j, rng.choice(n, hub_deg, replace=False)])
    keep = i != j
    return oadj.pattern_with_selfloops(*oadj._pairs_to_csr(n, i[keep], j[keep]))


@pytest.mark.parametrize("width", [128, 256, 512, 1024])
@pytest.mark.parametrize("mean", [True, False])
def test_spmm_peer_blocks_on_one_device_match_spmm(width, mean):
    """The peer-memory SpMM with the panel split into 3 uneven blocks (three separate allocations on one GPU stand
    in for three ranks' exchange buffers) is bit-identical to the single-panel SpMM on every block's rows.  Two graphs:
    the golden stress graph, and one whose middle block holds a hub row (> LONG_ROW = 512 entries, split over the
    CTA's warps) with neighbours in all three blocks."""
    from chromegcn_b200 import dist as cdist, ops
    from chromegcn_b200.graph import HiCGraph
    dev = torch.device("cuda", 0)
    z = np.load(os.path.join(GOLDEN, "model_l2_stress.npz"))
    hub_rp, hub_ci = _hub_graph()
    hub = hub_ci[hub_rp[1500]: hub_rp[1501]]                   # row 1500 of block [600, 2100)
    assert hub.shape[0] > 512 and all(((hub >= b) & (hub < e)).any() for b, e in ((0, 600), (600, 2100), (2100, 3000)))
    for rp, ci in (oadj.pattern_with_selfloops(z["indptr"], z["indices"]), (hub_rp, hub_ci)):
        n = rp.shape[0] - 1
        cuts = [0, n // 5, n // 5 + n // 2, n]
        gen = torch.Generator(device=dev).manual_seed(5)
        x = torch.randn(n, width, device=dev, generator=gen)
        res = torch.randn(n, width, device=dev, generator=gen)
        full = ops.spmm(HiCGraph.from_csr_pattern(rp, ci, dev, add_selfloops=False), x, mean=mean, residual=res)
        blocks = [x[cuts[r]: cuts[r + 1]].clone() for r in range(3)]
        for r in range(3):
            lp, lc = cdist.local_rows_csr(rp, ci, cuts[r], cuts[r + 1])
            g = HiCGraph.from_csr_pattern(lp, lc, dev, add_selfloops=False)
            got = ops.spmm_peer(g, blocks, r, mean=mean, residual=res[cuts[r]: cuts[r + 1]])
            assert torch.equal(got, full[cuts[r]: cuts[r + 1]]), (n, r)


def test_spmm_peer_rejects_invalid_panel():
    """cgcn_spmm_peer checks the peer panel on the host: each malformed panel, an output that is one of the blocks
    and a width the peer entry point has no kernel for (384) return CGCN_ERR_INVALID before anything is launched."""
    import ctypes as C
    from chromegcn_b200 import _lib, dist as cdist, ops
    from chromegcn_b200.graph import HiCGraph
    dev = torch.device("cuda", 0)
    lib = _lib.load()
    n, cuts = 3000, [0, 600, 2100, 3000]
    rp, ci = _hub_graph(n)
    lp, lc = cdist.local_rows_csr(rp, ci, cuts[1], cuts[2])
    g = HiCGraph.from_csr_pattern(lp, lc, dev, add_selfloops=False)
    x = {w: torch.randn(n, w, device=dev) for w in (128, 384)}
    out = {w: torch.empty(g.n, w, device=dev) for w in (128, 384)}

    def call(width=128, world=3, rank=1, begins=cuts, bases=None, o=None):
        pp = ops.peer_panel([x[width][cuts[r]].data_ptr() for r in range(3)], begins, rank)
        pp.world = world
        for r, b in enumerate(bases or []):
            pp.base[r] = b
        o = out[width].data_ptr() if o is None else o
        return lib.cgcn_spmm_peer(C.byref(g.c_struct()), C.byref(pp), o, width, 1, None, _lib.current_stream())

    assert call() == 0                                    # the panel the bad cases below are derived from
    torch.cuda.synchronize()
    bad = [dict(world=0), dict(world=9), dict(rank=3), dict(rank=-1), dict(bases=[x[128][0].data_ptr(), None]),
           dict(begins=[0, 2100, 600, 3000]), dict(begins=[0, 600, 2101, 3000]), dict(o=x[128][cuts[2]].data_ptr()),
           dict(width=384)]
    before = _lib.launch_count()
    for kw in bad:
        assert call(**kw) == -1, kw                       # CGCN_ERR_INVALID
    assert _lib.launch_count() == before


@pytest.mark.parametrize("exchange", ["nccl", "peer"])
def test_phase_api_world1_is_bit_identical(exchange):
    dev = torch.device("cuda", 0)
    os.environ["CGCN_NO_SIDE_STREAM"] = "1"      # same stream order in both runs (fixed-order reductions either way)
    ref = _single_gpu_reference(dev)
    got = _partitioned(dev, 0, 1, exchange=exchange)
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    for k in ref[2]:
        assert torch.equal(got[2][k], ref[2][k]), k
    assert torch.equal(got[3], ref[3]) and torch.equal(got[4], ref[4])


def _worker(rank, world, port, ret, exchange="nccl"):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        ref = _single_gpu_reference(dev)
        out, loss, grads, xg, rv, (b, e) = _partitioned(dev, rank, world, exchange=exchange)
        errs = {"out": ogcn.max_rel(out.cpu(), ref[0][b:e].cpu()), "loss": abs(loss.item() - ref[1].item()) / abs(ref[1].item()),
                "xgrad": ogcn.max_rel(xg.cpu(), ref[3][b:e].cpu()), "running_var": ogcn.max_rel(rv.cpu(), ref[4].cpu())}
        for k in ref[2]:
            errs["grad." + k] = ogcn.max_rel(grads[k].cpu(), ref[2][k].cpu())
        ret[rank] = errs
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("exchange", ["nccl", "peer"])
def test_row_partition_two_gpus_matches_single_gpu(exchange):
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, ret, exchange)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        assert p.exitcode == 0
    for r in (0, 1):
        for k, v in ret[r].items():
            assert v <= (1e-5 if not k.startswith("grad.") else 2e-5), (r, k, v)


@pytest.mark.parametrize("exchange", ["nccl", "peer"])
def test_phase_api_world1_d512_is_bit_identical(exchange):
    """d_model 512 (BASELINE.json's stress configuration, width-1024 panels): the stage-by-stage path with identity
    collectives reproduces the fused single-GPU step bit for bit."""
    from chromegcn_b200 import dist as cdist, synthetic
    from chromegcn_b200.chrome_models import ChromeGCN
    from chromegcn_b200.engine import ChromosomeEngine
    from chromegcn_b200.graph import HiCGraph
    dev = torch.device("cuda", 0)
    os.environ["CGCN_NO_SIDE_STREAM"] = "1"
    d, nclass = 512, 11
    h = synthetic.make_hic("chr21", hic_edges=5000, n_windows=700, n_bins=1900)
    ip, ix = oadj.build_adjacency_numpy(h.window_starts, h.bin1, h.bin2, h.val, h.norm, 1, 5000)
    rp, ci = oadj.pattern_with_selfloops(ip, ix)
    n = rp.shape[0] - 1
    gen = torch.Generator().manual_seed(9)
    panel = torch.randn(n, 2, d, generator=gen).to(dev)
    tgt = (torch.rand(n, nclass, generator=gen) < 0.3).float().to(dev)
    runs = []
    for mode in ("fused", exchange):
        torch.manual_seed(4)
        m = ogcn.stress_init_(ChromeGCN(d, d, nclass, 0.0, True, 2)).to(dev).train()
        g = HiCGraph.from_csr_pattern(rp, ci, dev, add_selfloops=False)
        loss = torch.zeros(1, device=dev)
        if mode == "fused":
            out, _ = ChromosomeEngine(m, 2).run(g, panel, tgt, None, loss, train=True)
        else:
            step = cdist.RowPartitionedStep(m, g, cdist.row_partition(n, 1), 0, 2, None, exchange=mode)
            out, _ = step.run(panel, tgt, loss, train=True)
            out = out.clone()
            torch.cuda.synchronize(dev)
            step.close()
        runs.append((out.clone(), loss.clone(), {k: p.grad.clone() for k, p in m.named_parameters()}))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    for k in runs[0][2]:
        assert torch.equal(runs[0][2][k], runs[1][2][k]), k
