"""GPU parity: each C-ABI kernel against the CPU oracle / fp64 torch on the same seeded inputs.

Tolerances (max-norm relative, `oracle.gcn.max_rel`):
  * integer work (adjacency, patterns): bit-exact;
  * SpMM: 2e-6 (same fp32 summation order as the reference's per-row accumulation);
  * fp32 FFMA contractions: 2e-6 against fp64;
  * tcgen05 3xTF32 contractions: 1e-5 against fp64 (north_star budget), and reported.
"""
import functools
import os

import numpy as np
import pytest
import torch

from oracle import adjacency as oadj
from oracle import gcn as ogcn

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
CHROMS = ["chr1", "chr2", "chr3", "chr22"]


def _dev():
    return torch.device("cuda", 0)


def _random_pattern(n, avg_deg, seed, hub=None):
    rng = np.random.default_rng(seed)
    m = n * avg_deg // 2
    i = rng.integers(0, n, m)
    j = np.clip(i + rng.integers(1, 200, m), 0, n - 1)
    if hub is not None:
        hi = np.full(hub, 7)
        hj = rng.choice(n, hub, replace=False)
        i, j = np.concatenate([i, hi]), np.concatenate([j, hj])
    keep = i != j
    ip, ix = oadj._pairs_to_csr(n, i[keep], j[keep])
    return ip, ix


def _graph(ip, ix):
    from chromegcn_b200.graph import HiCGraph
    return HiCGraph.from_csr_pattern(ip, ix, _dev(), add_selfloops=True)


@pytest.mark.parametrize("width", [128, 256, 512, 1024])
@pytest.mark.parametrize("mean", [True, False])
def test_spmm_matches_oracle(width, mean):
    from chromegcn_b200 import ops
    n = 3001
    ip, ix = _random_pattern(n, 12, 5, hub=1500)          # row 7 is a hub (> LONG_ROW): block-cooperative path
    g = _graph(ip, ix)
    rp, ci = oadj.pattern_with_selfloops(ip, ix)
    assert np.array_equal(g.csr_numpy()[0], rp) and np.array_equal(g.csr_numpy()[1], ci)
    gen = torch.Generator().manual_seed(1)
    x = torch.randn(n, width, generator=gen)
    res = torch.randn(n, width, generator=gen)
    a = ogcn.coo_adjacency(ip, ix, torch.float64).coalesce()
    if not mean:
        a = torch.sparse_coo_tensor(a.indices(), torch.ones_like(a.values()), a.shape)
    want = torch.sparse.mm(a, x.double())
    got = ops.spmm(g, x.to(_dev()), mean=mean).cpu()
    assert ogcn.max_rel(got, want) <= 2e-6
    got2 = ops.spmm(g, x.to(_dev()), mean=mean, residual=res.to(_dev())).cpu()
    assert ogcn.max_rel(got2, want + res.double()) <= 2e-6


@pytest.mark.parametrize("width", [128, 256])
@pytest.mark.parametrize("n", [1013, 37, 4500])
def test_spmm_near_diagonal_graph_matches_oracle_and_peer_kernel(width, n):
    """Near-diagonal (Hi-C-like) graphs: short-range pairs, 5 % long-range pairs, one hub row, isolated rows, n not
    a multiple of the CTA's row count.  Checked against the fp64 oracle and, bit for bit, against the peer-memory
    kernel with one block (both kernels sum a row's neighbours in CSR order)."""
    from chromegcn_b200 import ops
    rng = np.random.default_rng(n + width)
    m = n * 8
    i = rng.integers(0, n, m)
    j = np.clip(i + rng.integers(-20, 21, m), 0, n - 1)
    far = rng.random(m) < 0.05
    j[far] = rng.integers(0, n, int(far.sum()))
    if n > 800:                                                           # row 5: hub (> LONG_ROW entries)
        hj = rng.choice(n, 700, replace=False)
        i, j = np.concatenate([i, np.full(700, 5)]), np.concatenate([j, hj])
    keep = (i != j) & (i % 97 != 3)                                       # rows 3, 100, 197, ... keep only their self loop
    ip, ix = oadj._pairs_to_csr(n, i[keep], j[keep])
    g = _graph(ip, ix)
    gen = torch.Generator().manual_seed(n)
    x = torch.randn(n, width, generator=gen)
    res = torch.randn(n, width, generator=gen)
    a = ogcn.coo_adjacency(ip, ix, torch.float64).coalesce()
    want = torch.sparse.mm(a, x.double())
    got = ops.spmm(g, x.to(_dev()), mean=True, residual=res.to(_dev()))
    assert ogcn.max_rel(got.cpu(), want + res.double()) <= 2e-6
    same_order = ops.spmm_peer(g, [x.to(_dev())], 0, mean=True, residual=res.to(_dev()))
    assert torch.equal(got, same_order)
    plain = ops.spmm(g, x.to(_dev()), mean=False)
    assert torch.equal(plain, ops.spmm_peer(g, [x.to(_dev())], 0, mean=False))


def test_spmm_isolated_rows_and_tiny_graph():
    from chromegcn_b200 import ops
    ip = np.array([0, 0, 1, 2, 2], dtype=np.int32)        # rows 0 and 3 isolated -> self loop only
    ix = np.array([2, 1], dtype=np.int32)
    g = _graph(ip, ix)
    x = torch.arange(4 * 128, dtype=torch.float32).view(4, 128)
    got = ops.spmm(g, x.to(_dev())).cpu()
    want = torch.stack([x[0], (x[1] + x[2]) / 2, (x[1] + x[2]) / 2, x[3]])
    assert torch.equal(got, want)


@pytest.mark.parametrize("impl", [1, 0])
@pytest.mark.parametrize("m,k,n,bt,bias,scale", [(1000, 128, 128, False, True, False), (777, 128, 103, True, True, False),
                                                  (515, 103, 128, False, False, False), (4099, 128, 128, True, False, True),
                                                  (130, 128, 128, False, False, False), (64, 37, 5, True, True, False),
                                                  # weight operands wider than one 128 x 128 block (d_model 256 / 512)
                                                  (1000, 512, 512, False, True, False), (777, 512, 103, True, True, False),
                                                  (515, 103, 512, False, False, False), (600, 256, 256, True, False, True),
                                                  (300, 200, 300, False, True, False)])
def test_gemm_rowpanel(impl, m, k, n, bt, bias, scale):
    from chromegcn_b200 import ops
    gen = torch.Generator().manual_seed(m)
    a = torch.randn(m, k, generator=gen)
    b = torch.randn(n, k, generator=gen) if bt else torch.randn(k, n, generator=gen)
    bi = torch.randn(n, generator=gen) if bias else None
    want = a.double() @ (b.double().t() if bt else b.double())
    g = None
    if scale:
        ip, ix = _random_pattern(m, 6, 3)
        g = _graph(ip, ix)
        deg = torch.from_numpy(np.diff(oadj.pattern_with_selfloops(ip, ix)[0])).double()
        want = want / deg[:, None]
    if bias:
        want = want + bi.double()
    got = ops.gemm_rowpanel(a.to(_dev()), b.to(_dev()), bt, bi.to(_dev()) if bias else None, g, 1, impl).cpu()
    tol = 2e-6 if impl == 1 else 1e-5
    err = ogcn.max_rel(got, want)
    print("rowpanel impl=%d m=%d k=%d n=%d err=%.2e" % (impl, m, k, n, err))
    assert err <= tol


@pytest.mark.parametrize("impl", [1, 0])
@pytest.mark.parametrize("m,ka,nb", [(5000, 128, 128), (70001, 103, 128), (33, 128, 128), (2049, 128, 128),
                                     (5000, 512, 512), (3000, 103, 512), (2000, 256, 128), (700, 300, 200)])
def test_gemm_gram(impl, m, ka, nb):
    from chromegcn_b200 import ops
    gen = torch.Generator().manual_seed(m)
    a = torch.randn(m, ka, generator=gen)
    b = torch.randn(m, nb, generator=gen)
    want = a.double().t() @ b.double()
    got = ops.gemm_gram(a.to(_dev()), b.to(_dev()), impl).cpu()
    tol = 2e-6 if impl == 1 else 1e-5
    # reduction over m signed terms: scale by the no-cancellation magnitude sqrt(m)
    err = float((got.double() - want).abs().max()) / float(want.abs().max())
    print("gram impl=%d m=%d err=%.2e" % (impl, m, err))
    assert err <= tol * 4


def test_bce_loss_and_gradient():
    from chromegcn_b200 import ops
    gen = torch.Generator().manual_seed(2)
    n, c, s = 1001, 103, 2
    out = torch.randn(n, s, c, generator=gen) * 3
    out[0, :, 0] = 40.0
    out[1, :, 1] = -40.0
    tgt = (torch.rand(n, c, generator=gen) < 0.2).float()
    o64 = out.double().requires_grad_(True)
    pred = o64.mean(1)
    loss = torch.nn.functional.binary_cross_entropy_with_logits(pred, tgt.double())
    loss.backward()
    acc = torch.zeros(1, device=_dev())
    probs, grad = ops.bce_loss(out.to(_dev()), tgt.to(_dev()), s, acc)
    assert abs(acc.item() - loss.item()) <= 2e-6 * abs(loss.item())
    assert ogcn.max_rel(probs.cpu(), torch.sigmoid(pred)) <= 2e-6
    assert ogcn.max_rel(grad.cpu(), o64.grad) <= 2e-6
    ops.bce_loss(out.to(_dev()), tgt.to(_dev()), s, acc, want_probs=False, want_grad=False)   # accumulates
    assert abs(acc.item() - 2 * loss.item()) <= 4e-6 * abs(loss.item())


@pytest.mark.parametrize("c", [103, 1, 32, 33, 128, 200])
def test_bce_loss_bit_packed_labels_identical_to_float(c):
    """`cgcn_bce_loss_bits` (labels as bit rows) must reproduce `cgcn_bce_loss` bit for bit."""
    from chromegcn_b200 import ops
    gen = torch.Generator().manual_seed(20 + c)
    n, s = 777, 2
    ld = (c + 3) // 4 * 4
    out = torch.zeros(n, s, ld)
    out[:, :, :c] = torch.randn(n, s, c, generator=gen) * 3
    tgt = (torch.rand(n, c, generator=gen) < 0.3).float()
    bits = ops.pack_targets(tgt)
    assert bits is not None and bits.dtype == torch.int32 and tuple(bits.shape) == (n, (c + 31) // 32)
    a0, a1 = torch.zeros(1, device=_dev()), torch.zeros(1, device=_dev())
    p0, g0 = ops.bce_loss(out.to(_dev()), tgt.to(_dev()), s, a0)
    p1, g1 = ops.bce_loss(out.to(_dev()), bits.to(_dev()), s, a1, nclass=c)
    assert torch.equal(p0, p1) and torch.equal(g0, g1) and a0.item() == a1.item()
    soft = tgt.clone()
    soft[3, 0] = 0.5
    assert ops.pack_targets(soft) is None                      # soft labels keep the float path


@pytest.mark.parametrize("kind", ["sgd", "adam"])
def test_optimizer_kernels_match_torch(kind):
    from chromegcn_b200 import ops
    gen = torch.Generator().manual_seed(3)
    p0 = torch.randn(5000, generator=gen)
    ref = torch.nn.Parameter(p0.clone().double())
    opt = (torch.optim.SGD([ref], lr=0.25, momentum=0.9, weight_decay=1e-6) if kind == "sgd"
           else torch.optim.Adam([ref], lr=2e-3, betas=(0.9, 0.98)))
    p = p0.clone().to(_dev())
    b1 = torch.zeros_like(p)
    b2 = torch.zeros_like(p)
    for step in range(1, 6):
        g = torch.randn(5000, generator=gen)
        ref.grad = g.double()
        opt.step()
        if kind == "sgd":
            ops.sgd_step(p, g.to(_dev()), b1, 0.25)
        else:
            ops.adam_step(p, g.to(_dev()), b1, b2, 2e-3, step)
    assert ogcn.max_rel(p.cpu(), ref.data) <= 2e-6


def test_interleave_roundtrip_and_dropout_mask():
    from chromegcn_b200 import ops
    gen = torch.Generator().manual_seed(4)
    a, b = torch.randn(333, 128, generator=gen), torch.randn(333, 128, generator=gen)
    panel = ops.interleave_strands([a.to(_dev()), b.to(_dev())])
    assert torch.equal(panel.cpu(), torch.stack([a, b], 1))
    ra, rb = ops.deinterleave_strands(panel)
    assert torch.equal(ra.cpu(), a) and torch.equal(rb.cpu(), b)
    m1 = ops.dropout_mask(4000, 2, 128, 0.2, 123, 5, 0)
    m2 = ops.dropout_mask(4000, 2, 128, 0.2, 123, 5, 0)
    m3 = ops.dropout_mask(4000, 2, 128, 0.2, 123, 6, 0)
    m4 = ops.dropout_mask(4000, 2, 128, 0.2, 123, 5, 1)
    assert torch.equal(m1, m2) and not torch.equal(m1, m3) and not torch.equal(m1, m4)
    vals = torch.unique(m1).cpu().tolist()
    assert len(vals) == 2 and vals[0] == 0.0 and abs(vals[1] - 1.25) < 1e-6
    keep = float((m1 > 0).float().mean())
    assert abs(keep - 0.8) < 3e-3                       # 1.0e6 draws: sigma = 4e-4


# ------------------------------------------------------------------------------ adjacency (bit-exact)
@pytest.mark.parametrize("fname", ["adjacency_SQRTVC_1200.npz", "adjacency_none_1200.npz", "adjacency_SQRTVC_41.npz",
                                   "adjacency_SQRTVC_1000000.npz"])
def test_adjacency_build_golden(fname):
    from chromegcn_b200 import ops
    z = np.load(os.path.join(GOLDEN, fname))
    use_norm = str(z["norm_name"]) != ""
    for c in CHROMS:
        ip, ix = ops.adjacency_build(z[c + "_windows"], z[c + "_bin1"], z[c + "_bin2"], z[c + "_val"],
                                     z[c + "_norm"] if use_norm else None, 1, int(z["hic_edges"]))
        assert ip.dtype == np.int32 and ix.dtype == np.int32
        assert np.array_equal(ip, z[c + "_indptr"]), (fname, c)
        assert np.array_equal(ix, z[c + "_indices"]), (fname, c)


@pytest.mark.parametrize("chrom,hic_edges,use_norm", [("chr22", 500000, True), ("chr22", 125000, True),
                                                      ("chr20", 1000000, True), ("chr21", 250000, False)])
def test_adjacency_build_full_size_vs_oracle(chrom, hic_edges, use_norm):
    """Config-1 sized input (1.5 M contact rows, 20 k windows): byte-identical CSR + structural properties."""
    from chromegcn_b200 import ops, synthetic
    h = synthetic.make_hic(chrom, hic_edges=hic_edges)
    b1, b2, v = h.bin1, h.bin2, h.val
    if not use_norm:
        order = np.argsort(-v, kind="stable")
        b1, b2, v = b1[order], b2[order], v[order]
    norm = h.norm if use_norm else None
    ip, ix = ops.adjacency_build(h.window_starts, b1, b2, v, norm, 1, hic_edges)
    wp, wx = oadj.build_adjacency_numpy(h.window_starts, b1, b2, v, norm, 1, hic_edges)
    assert np.array_equal(ip, wp) and np.array_equal(ix, wx)
    n = ip.shape[0] - 1
    rows = np.repeat(np.arange(n), np.diff(ip))
    assert not np.any(rows == ix)
    assert ip[-1] <= hic_edges
    fwd = rows.astype(np.int64) * n + ix
    bwd = ix.astype(np.int64) * n + rows
    assert np.array_equal(np.sort(fwd), np.sort(bwd))          # symmetric
    assert np.all(np.diff(fwd) > 0)                            # sorted, unique


def test_adjacency_edge_cases():
    from chromegcn_b200 import ops, _lib
    w = np.array([0, 1000, 2000, 5000], dtype=np.int64)
    norm = np.ones(6)
    # no acceptable contact at all
    ip, ix = ops.adjacency_build(w, np.array([3000, 0]), np.array([4000, 0]), np.array([1.0, 9.0]), norm, 1, 10)
    assert np.array_equal(ip, np.zeros(5, dtype=np.int32)) and ix.shape[0] == 0
    # empty contact list
    ip, ix = ops.adjacency_build(w, np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0), norm, 1, 10)
    assert np.array_equal(ip, np.zeros(5, dtype=np.int32)) and ix.shape[0] == 0
    # (a,b) and (b,a) selected together collapse; K larger than the candidates keeps everything
    ip, ix = ops.adjacency_build(w, np.array([0, 1000, 2000]), np.array([1000, 0, 5000]), np.array([3.0, 2.0, 1.0]),
                                 norm, 1, 100)
    wp, wx = oadj.build_adjacency_loops(w, np.array([0, 1000, 2000]), np.array([1000, 0, 5000]),
                                        np.array([3.0, 2.0, 1.0]), norm, 1, 100)
    assert np.array_equal(ip, wp) and np.array_equal(ix, wx) and ip[-1] == 4
    # a bin beyond the norm vector is the reference's IndexError
    with pytest.raises(_lib.ChromeGCNNativeError):
        ops.adjacency_build(w, np.array([0]), np.array([5000]), np.array([1.0]), np.ones(3), 1, 10)
    # NaN contact value: undefined order in the reference -> rejected
    with pytest.raises(_lib.ChromeGCNNativeError):
        ops.adjacency_build(w, np.array([0]), np.array([5000]), np.array([np.nan]), norm, 1, 10)


def test_adjacency_build_random_small_cases_vs_loop_oracle():
    """150 seeded adversarial cases (heavy value ties, duplicate and reversed keys, NaN / 0 norm entries, diagonal and
    non-window rows, K from 0 to more than the candidates, with and without the norm vector) through cgcn_adj_build,
    byte-compared with the record-at-a-time restatement of data/7create_graph_new.py:67-120."""
    from chromegcn_b200 import ops
    rng = np.random.default_rng(2024)
    vals_pool = np.array([0.0, 1.0, 2.0, 2.0, 3.0, 5.5, 7.0])
    norm_pool = np.array([1.0, 0.5, 2.0, np.nan, 0.0, 1.25])
    for case in range(150):
        n_bins = int(rng.integers(4, 60))
        starts = np.sort(rng.choice(n_bins, int(rng.integers(1, n_bins + 1)), replace=False)).astype(np.int64) * 1000
        m = int(rng.integers(0, 200))
        b1 = rng.integers(0, n_bins, m).astype(np.int64) * 1000
        b2 = rng.integers(0, n_bins, m).astype(np.int64) * 1000
        v = vals_pool[rng.integers(0, len(vals_pool), m)]
        norm = norm_pool[rng.integers(0, len(norm_pool), n_bins)] if case % 3 else None
        hic_edges = int(rng.integers(0, 2 * m + 5))
        want = oadj.build_adjacency_loops(starts, b1, b2, v, norm, 1, hic_edges)
        got = ops.adjacency_build(starts, b1, b2, v, norm, 1, hic_edges, _dev())
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), (case, n_bins, m, hic_edges)


def test_process_graph_golden():
    from scipy import sparse
    from chromegcn_b200.graph import process_graph, HiCGraph
    z = np.load(os.path.join(GOLDEN, "process_graph.npz"))
    for c in CHROMS:
        ip, ix = z[c + "_indptr"], z[c + "_indices"]
        n = ip.shape[0] - 1
        csr = sparse.csr_matrix((np.ones(ix.shape[0]), ix, ip), shape=(n, n))
        g = process_graph("hic", {c: csr}, n, c)
        assert isinstance(g, HiCGraph) and g.cuda() is g
        rp, ci = g.csr_numpy()
        wrp, wci = oadj.pattern_with_selfloops(ip, ix)
        assert np.array_equal(rp, wrp) and np.array_equal(ci, wci)
        coo = g.to_sparse_coo()
        assert not coo.is_coalesced()
        assert np.array_equal(coo._indices()[0].cpu().numpy(), z[c + "_coo_rows"])
        assert np.array_equal(coo._indices()[1].cpu().numpy(), z[c + "_coo_cols"])
        assert np.array_equal(coo._values().cpu().numpy(), z[c + "_coo_vals"])        # bit-exact fp32 1/deg
        # and back: the reference's tensor -> pattern
        g2 = HiCGraph.from_torch_coo(coo)
        assert np.array_equal(g2.csr_numpy()[0], wrp) and np.array_equal(g2.csr_numpy()[1], wci)


def test_process_graph_other_adj_types():
    """adj_type constant / none (pattern kernels) and both (weighted kernels) against the reference's tensors."""
    from scipy import sparse
    from chromegcn_b200.graph import process_graph
    from chromegcn_b200 import ops
    z = np.load(os.path.join(GOLDEN, "adj_types.npz"))
    n = int(z["n"])
    csr = sparse.csr_matrix((np.ones(z["indices"].shape[0]), z["indices"], z["indptr"]), shape=(n, n))
    gen = torch.Generator().manual_seed(9)
    x = torch.randn(n, 256, generator=gen)
    for t in ("constant", "both", "none"):
        g = process_graph(t, {"chrZ": csr}, n, "chrZ")
        coo = g.to_sparse_coo().coalesce()
        assert np.array_equal(coo.indices()[0].cpu().numpy(), z[t + "_rows"])
        assert np.array_equal(coo.indices()[1].cpu().numpy(), z[t + "_cols"])
        assert np.allclose(coo.values().cpu().numpy(), z[t + "_vals"], rtol=2e-7, atol=0)
        assert (g.vals is not None) == (t == "both")
        ref = torch.sparse_coo_tensor(torch.from_numpy(np.vstack((z[t + "_rows"], z[t + "_cols"]))),
                                      torch.from_numpy(z[t + "_vals"]).double(), (n, n))
        want = torch.sparse.mm(ref, x.double())
        assert ogcn.max_rel(ops.spmm(g, x.to(_dev()), mean=True).cpu(), want) <= 2e-6
        # backward operator: A_hat^T G = A (row_inv .* G)
        wantT = ref.to_dense().t() @ x.double()
        if g.vals is None:
            scaled = x / g.degrees().cpu().float()[:, None]
        else:
            scaled = x * g.row_inv.cpu()[:, None]
        assert ogcn.max_rel(ops.spmm(g, scaled.to(_dev()), mean=False).cpu(), wantT) <= 2e-6


def test_model_on_weighted_graph_matches_reference():
    """ChromeGCN step with adj_type 'both' (weighted SpMM, row_inv row scaling in the backward GEMM)."""
    from scipy import sparse
    from chromegcn_b200.chrome_models import ChromeGCN
    from chromegcn_b200.engine import ChromosomeEngine
    from chromegcn_b200.graph import process_graph
    z = np.load(os.path.join(GOLDEN, "adj_types.npz"))
    n = int(z["n"])
    csr = sparse.csr_matrix((np.ones(z["indices"].shape[0]), z["indices"], z["indptr"]), shape=(n, n))
    g = process_graph("both", {"c": csr}, n, "c")
    sd = {k[4:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd0.")}
    nclass = sd["out.weight"].shape[0]
    for impl in (1, 0):
        m = ChromeGCN(128, 128, nclass, 0.0, True, 2)
        m.load_state_dict(sd)
        m = m.to(_dev()).train()
        m.gemm_impl = impl
        eng = ChromosomeEngine(m, 2)
        loss = torch.zeros(1, device=_dev())
        xg = torch.empty(n, 2, 128, device=_dev())
        out, _ = eng.run(g, eng.pack(torch.from_numpy(z["x_f"]).to(_dev()), torch.from_numpy(z["x_r"]).to(_dev())),
                         torch.from_numpy(z["target"]).to(_dev()), None, loss, train=True, input_grad=xg)
        assert ogcn.max_rel(out.mean(1).cpu(), torch.from_numpy(z["f32.pred"])) <= 1e-5
        assert abs(loss.item() - float(z["f32.loss"])) <= 1e-5 * abs(float(z["f32.loss"]))
        for k, p in m.named_parameters():
            ref64 = torch.from_numpy(z["f64.grad." + k])
            own = ogcn.max_rel(torch.from_numpy(z["f32.grad." + k]), ref64)
            assert ogcn.max_rel(p.grad.cpu(), ref64) <= max(1e-5, 3 * own), (impl, k)


def _elementwise_rel(got, ref, floor):
    """max over elements of |got - ref| / max(|ref|, floor * max|ref|): the element-wise companion of `max_rel` (VERDICT
    r01: max-norm alone hides errors on small entries).  The floor is needed because every output here is a 128-term
    fp32 dot product: its absolute rounding error (~1e-6 of the row's scale, the fp32 reference's as much as ours) is
    unrelated to how close to zero the sum happens to land."""
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    denom = torch.clamp(ref.abs(), min=floor * float(ref.abs().max()))
    return float(((got - ref).abs() / denom).max())


# ------------------------------------------------------------------------------ fused layer kernel (csrc/fused_layer.cu)
def _cdiv(a, b):
    return -(-a // b)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _fused_grid(n, strands, sms):
    """Python copy of fused_layer_grid (csrc/fused_layer.cu): `(CTAs, window rows per CTA)`.  A CTA runs its rows as
    tiles of 64 / strands window rows; the tests below pick their sizes and place their edge-case rows with it, and
    check the kernel's CTA count against it, so a change of the rule fails them instead of moving them to another
    regime unnoticed."""
    grid = max(min(_cdiv(n, 64 // strands), sms), 1)
    rows = max(_cdiv(_cdiv(n, grid), 4) * 4, 4)
    return max(_cdiv(n, rows), 1), rows


# "one_tile": 2777 rows are one tile per CTA on 148 SMs (44 CTAs x 64 rows with one strand, 87 x 32 with two).
# "multi_tile": every CTA but the last runs >= 3 tiles and the last of them is partly filled: on 148 SMs, one strand
# 31 111 rows = 147 CTAs x 212 (4 tiles, the last holding 20), two strands 15 557 = 145 x 108 (4 tiles, the last
# holding 12).  Other SM counts scale n and take the next n with these properties.
_ONE_TILE_N = 2777
_MULTI_TILE_N_148 = {1: 31111, 2: 15557}


def _layer_n(strands, size):
    if size == "one_tile":
        return _ONE_TILE_N
    sms, tg = _sms(), 64 // strands
    n0 = _MULTI_TILE_N_148[strands] * sms // 148
    for n in range(n0, 2 * n0):
        grid, rows = _fused_grid(n, strands, sms)
        if grid >= 10 and rows % tg != 0 and _cdiv(rows, tg) >= 3:
            return n
    raise AssertionError("no multi-tile size for %d SMs" % sms)


_HUB = 913      # stored entries of a hub row, self loop included: 29 segments of <= 32 column indices


def _edge_case_graph(n, strands, seed=11):
    """A near-diagonal Hi-C-like symmetric pattern (mean degree ~13 with the self loops) in which rows at positions
    taken from the grid have exactly 1 (self loop only), 32, 33, 64, 65 (the segment and batch edges of the gather for
    U = 3 and 6) or _HUB stored entries: at the first and last row of a CTA, at a tile's first or last row and in the
    middle of a tile.  Edges of these rows lead to other rows only, so the counts are exact.  Returns
    `(indptr, indices, graph)`, the CSR without the self loops the graph adds."""
    grid, rows = _fused_grid(n, strands, _sms())
    tg = 64 // strands
    ntile = _cdiv(rows, tg)
    last = (ntile - 1) * tg                      # offset of a CTA's last tile
    cta = lambda c: c * rows
    assert grid >= 10
    want = {cta(1): 1, cta(3) - 1: 1,            # self loop only: first row of one CTA, last row of another
            cta(4) - 1: _HUB,                    # hub: last row of a CTA ...
            cta(5) + min(2, ntile - 1) * tg: _HUB,   # ... and first row of a tile inside one (its third, if it has one)
            cta(6) + min(tg, rows) - 1: 32,      # last row of a CTA's first tile
            cta(7) + last: 33,                   # first row of a CTA's last tile
            cta(8) + last + 1: 64, cta(9) - 1: 65,   # inside and at the end of a CTA's last tile
            cta(9) + 4: 32, cta(9) + 5: 33, cta(9) + 6: 64, cta(9) + 7: 65}
    rng = np.random.default_rng(seed)
    m = n * 6
    i = rng.integers(0, n, m)
    j = np.clip(i + rng.integers(1, 200, m), 0, n - 1)
    special = np.zeros(n, dtype=bool)
    special[list(want)] = True
    keep = (i != j) & ~special[i] & ~special[j]
    pi, pj = [i[keep]], [j[keep]]
    free = np.flatnonzero(~special)
    for r, k in want.items():
        if k == _HUB:
            partners = rng.choice(free, k - 1, replace=False)
        else:                                    # the nearest ordinary rows: a near-diagonal band
            partners = free[np.argsort(np.abs(free - r), kind="stable")[: k - 1]]
        pi.append(np.full(k - 1, r))
        pj.append(partners)
    ip, ix = oadj._pairs_to_csr(n, np.concatenate(pi), np.concatenate(pj))
    g = _graph(ip, ix)
    deg = np.diff(g.csr_numpy()[0])
    assert all(deg[r] == k for r, k in want.items()), {r: (k, deg[r]) for r, k in want.items()}
    assert 10 <= g.nnz / n <= 15
    return ip, ix, g


_FWD_CASES = ([pytest.param(m, "one_tile", id=m) for m in ("plain", "gate_off", "dropout", "stats", "hubs")] +
              [pytest.param(m, "multi_tile", id=m + "-multi_tile") for m in ("plain", "gate_off", "dropout", "stats")])


@pytest.mark.parametrize("strands", [1, 2])
@pytest.mark.parametrize("mode,size", _FWD_CASES)
def test_fused_layer_fwd_matches_fp64(strands, mode, size):
    """cgcn_gcn_layer_fwd (one kernel: gather -> tcgen05 3xTF32 -> gate epilogue) against the layer of
    models/ChromeModels.py:37-40 + models/SubLayers.py:42-52 in fp64 torch on the same inputs; the dropout case feeds
    the oracle the kernel's own keep-mask (cgcn_dropout_mask).  The multi-tile cases run several tiles per CTA on the
    edge-case graph; their stats case checks column partials accumulated over several tiles."""
    from chromegcn_b200 import ops
    if size == "multi_tile":
        n = _layer_n(strands, size)
        ip, ix, g = _edge_case_graph(n, strands)
    else:
        n = _ONE_TILE_N if mode != "hubs" else 1500      # not a multiple of the 64-row tile; several CTAs
        ip, ix = _random_pattern(n, 14, 11, hub=900 if mode == "hubs" else None)     # row 7 of "hubs" spans 29 segments
        g = _graph(ip, ix)
    gen = torch.Generator().manual_seed(3)
    shape = (n, 128) if strands == 1 else (n, 2, 128)
    x = torch.randn(*shape, generator=gen)
    w = torch.randn(128, 128, generator=gen) * 0.12
    b = torch.randn(128, generator=gen) * 0.1
    wg = torch.randn(128, generator=gen) * 0.3
    bg = torch.randn(1, generator=gen) * 0.1
    p = 0.3 if mode == "dropout" else 0.0
    seed, step, site = 1234567, 9, 0
    xo, z, gate, sx, stats = ops.gcn_layer_fwd(g, x.to(_dev()), w.to(_dev()), b.to(_dev()), wg.to(_dev()), bg.to(_dev()),
                                               gate_off=(mode == "gate_off"), dropout_p=p, seed=seed, step=step, site=site,
                                               with_stats=(mode == "stats"))
    a = ogcn.coo_adjacency(ip, ix, torch.float64).coalesce()
    xd = x.double().reshape(n, -1)
    pat = torch.sparse_coo_tensor(a.indices(), torch.ones_like(a.values()), a.shape)
    sx_ref = torch.sparse.mm(pat, xd).reshape(shape)
    ax = torch.sparse.mm(a, xd).reshape(shape)
    z_ref = torch.tanh(ax @ w.double() + b.double())
    g_ref = torch.ones(*shape[:-1], 1, dtype=torch.float64) if mode == "gate_off" else torch.sigmoid(z_ref @ wg.double()[:, None] + bg.double())
    xo_ref = (1 - g_ref) * x.double() + g_ref * z_ref
    if p > 0:
        mask = ops.dropout_mask(n, strands, 128, p, seed, step, site, _dev()).cpu().double().reshape(shape)
        assert 0.6 < float((mask > 0).double().mean()) < 0.8
        xo_ref = xo_ref * mask
    assert ogcn.max_rel(sx.cpu(), sx_ref) <= 2e-6
    report = {"z": _panel_errors(z.cpu(), z_ref)}
    assert ogcn.max_rel(gate.cpu().reshape(g_ref.shape), g_ref) <= 1e-5
    report["x_out"] = _panel_errors(xo.cpu(), xo_ref)
    grid, rows = _fused_grid(n, strands, _sms())
    stats_err = ""
    if mode == "stats":
        assert stats.shape[0] == grid
        r = torch.relu(xo_ref).reshape(n, strands, 128)
        got = stats.double().sum(0).cpu().reshape(2, strands, 128)
        e = (ogcn.max_rel(got[0], r.sum(0)), ogcn.max_rel(got[1], (r * r).sum(0)))
        assert max(e) <= 1e-5
        stats_err = " | stats max_rel %.2e %.2e" % e
    print("fwd S=%d %s %s: %d CTAs, %d rows / CTA, %d tiles / CTA | %s%s"
          % (strands, size, mode, grid, rows, _cdiv(rows, 64 // strands),
             " | ".join("%s max_rel %.2e elementwise %.2e" % (k, *v) for k, v in report.items()), stats_err))


# The backward twin (cgcn_gcn_layer_bwd).  Its panels are the forward's error structure (a CSR gather of fp32 values, then
# a 3xTF32 128-term contraction) and get the forward test's bounds.  A column partial is a sum of signed terms over the
# rows of a CTA: it is held to 1e-5 of the no-cancellation magnitude sum_rows |term| of its own CTA and, summed over the
# CTAs in fp64, of the whole column.  A plain max-norm would be loose or fail on cancelling columns such as d b_g; this
# bound catches one dropped row slot or CTA.
_SEED, _STEP, _SITE = 1234567, 9, 0
_NAN_BITS = 0x7FC00000                          # torch.full(..., nan)


def _panel_errors(got, ref):
    """The bounds of the forward's z and x_out: max-norm relative <= 1e-5, element-wise <= 1e-4."""
    mr, er = ogcn.max_rel(got, ref), _elementwise_rel(got, ref, 0.05)
    assert mr <= 1e-5 and er <= 1e-4, (mr, er)
    return mr, er


def _guarded(shape):
    """A NaN-filled buffer with two guard rows on each side of `shape`: `(buffer, output view)`."""
    buf = torch.full((shape[0] + 4, *shape[1:]), float("nan"), device=_dev())
    return buf, buf[2:2 + shape[0]]


def _guards_intact(buf, rows):
    """The buffer's rows outside [2, 2 + rows) still hold their NaN, bit for bit."""
    outside = torch.cat([buf[:2].reshape(-1), buf[2 + rows:].reshape(-1)])
    return bool((outside.view(torch.int32) == _NAN_BITS).all())


def _bits_equal(a, b):
    return torch.equal(a.view(torch.int32), b.view(torch.int32))


@functools.lru_cache(maxsize=4)
def _bwd_inputs(strands, size):
    """Edge-case graph and fp32 inputs of one (strands, size), shared by the backward cases."""
    n = _layer_n(strands, size)
    _, _, g = _edge_case_graph(n, strands)
    gen = torch.Generator().manual_seed(17 + strands)
    shape = (n, 128) if strands == 1 else (n, 2, 128)
    inp = {k: torch.randn(*shape, generator=gen) for k in ("dys", "dxd", "y_prev", "x_prev")}
    inp["w"] = torch.randn(128, 128, generator=gen) * 0.12
    inp["wg"] = torch.randn(128, generator=gen) * 0.3
    inp["bg"] = torch.randn(1, generator=gen) * 0.1
    return n, g, inp


def _layer_above(g, inp, x):
    """`<G, (A_hat x) W> + <dxd, x>` with G = D dys: its gradient in x, A_hat^T G W^T + dxd, is what the kernel computes as
    (P dys) W^T + dxd.  A_hat = D^-1 P is written out per strand from the graph's CSR on the window index, so the
    reference does not rely on the pattern being symmetric; the kernel does."""
    rp, ci = g.csr_numpy()
    n, s = x.shape[0], x.shape[1]
    deg = torch.from_numpy(np.diff(rp)).double()
    rows = torch.repeat_interleave(torch.arange(n), deg.long())
    a_hat = torch.sparse_coo_tensor(torch.stack([rows, torch.from_numpy(ci).long()]), 1.0 / deg[rows], (n, n)).coalesce()
    ax = torch.sparse.mm(a_hat, x.reshape(n, s * 128)).reshape(n, s, 128)
    G = deg[:, None, None] * inp["dys"].double().reshape(n, s, 128)
    return (G * (ax @ inp["w"].double())).sum() + (inp["dxd"].double().reshape(n, s, 128) * x).sum()


@functools.lru_cache(maxsize=3)
def _bwd_mid_reference(strands, size, gate_off, p):
    """fp64 autograd of the layer below (tanh, gate, blend, dropout with the kernel's own keep-mask) under the layer
    above, from the fp32 values handed to the kernel.  Returns the kernel's z_prev = fp32(z) and g_prev = fp32(g), and
    the expected dy = y_prev.grad, dxd_out = x_prev.grad, dgp = d loss / d(z . wg + bg) and z."""
    from chromegcn_b200 import ops
    n, g, inp = _bwd_inputs(strands, size)
    y_prev = inp["y_prev"].double().reshape(n, strands, 128).requires_grad_(True)
    x_prev = inp["x_prev"].double().reshape(n, strands, 128).requires_grad_(True)
    wg = inp["wg"].double().requires_grad_(True)
    bg = inp["bg"].double().requires_grad_(True)
    z = torch.tanh(y_prev)
    a = z @ wg + bg
    a.retain_grad()
    gate = torch.ones_like(a) if gate_off else torch.sigmoid(a)
    x_l = (1 - gate)[..., None] * x_prev + gate[..., None] * z
    if p > 0:
        mask = ops.dropout_mask(n, strands, 128, p, _SEED, _STEP, _SITE, _dev()).cpu().double()
        assert 0.6 < float((mask > 0).double().mean()) < 0.8
        x_l = x_l * mask
    _layer_above(g, inp, x_l).backward()
    if gate_off:
        assert a.grad is None and wg.grad is None and bg.grad is None
    dgp = torch.zeros(n, strands, dtype=torch.float64) if gate_off else a.grad
    return {"z_prev": z.detach().float(), "g_prev": gate.detach().float(), "dy": y_prev.grad, "dxd": x_prev.grad,
            "dgp": dgp, "z": z.detach()}


def _run_bwd_mid(strands, size, gate_off, p, dxd_out):
    """cgcn_gcn_layer_bwd with the layer below, every output inside NaN guard rows (the partials inside a buffer of one
    row per SM, more than the kernel has CTAs).  `dxd_out`: "new" (a panel of its own), "in_place" (the dxd panel
    itself, as the model runs it) or None.  Returns host copies of (dys_out, dxd_out, partial)."""
    from chromegcn_b200 import ops
    n, g, inp = _bwd_inputs(strands, size)
    ref = _bwd_mid_reference(strands, size, gate_off, p)
    d = {k: v.to(_dev()) for k, v in inp.items()}
    shape = d["dys"].shape
    dys_buf, dys_out = _guarded(shape)
    part_buf, part_out = _guarded((_sms(), 2 * 128 + 4))
    dxd, dxd_buf, dxd_o = d["dxd"], None, None
    if dxd_out == "new":
        dxd_buf, dxd_o = _guarded(shape)
    elif dxd_out == "in_place":
        dxd_buf, dxd = _guarded(shape)
        dxd.copy_(d["dxd"])
        dxd_o = dxd
    got = ops.gcn_layer_bwd(g, d["dys"], dxd, d["w"], ref["z_prev"].reshape(shape).to(_dev()), d["x_prev"],
                            ref["g_prev"].to(_dev()), d["wg"], gate_off, p, _SEED, _STEP, _SITE,
                            dys_out=dys_out, dxd_out=dxd_o, partial=part_out)
    assert got[0] is dys_out and got[1] is dxd_o
    parts = got[2].shape[0]
    torch.cuda.synchronize()
    assert _guards_intact(dys_buf, n) and _guards_intact(part_buf, parts)
    assert dxd_buf is None or _guards_intact(dxd_buf, n)
    return dys_out.cpu(), (None if dxd_o is None else dxd_o.cpu()), got[2].cpu()


@pytest.mark.parametrize("mode", ["plain", "gate_off", "dropout", "in_place", "no_dxd_out"])
@pytest.mark.parametrize("strands", [1, 2])
@pytest.mark.parametrize("size", ["one_tile", "multi_tile"])
def test_fused_layer_bwd_mid_matches_fp64(size, strands, mode):
    """cgcn_gcn_layer_bwd with the layer below (fused_layer_kernel<S, BWD_MID>: gather u = P dys, u W^T on the tensor
    cores, + dxd, then the dropout / gate / tanh backward of the layer below and its column partials for d b, d w_g,
    d b_g) against fp64 autograd, on the edge-case graph with one and with several tiles per CTA.  The kernel must write
    nothing outside its outputs, repeat itself bit for bit (CSR-order gathers, fixed-order partials), and give the same
    bits when dxd_out is the dxd panel itself or absent."""
    gate_off, p = mode == "gate_off", (0.3 if mode == "dropout" else 0.0)
    dxd_mode = {"in_place": "in_place", "no_dxd_out": None}.get(mode, "new")
    n, g, _ = _bwd_inputs(strands, size)
    ref = _bwd_mid_reference(strands, size, gate_off, p)
    grid, rows = _fused_grid(n, strands, _sms())
    dys, dxd, part = _run_bwd_mid(strands, size, gate_off, p, dxd_mode)
    again = _run_bwd_mid(strands, size, gate_off, p, dxd_mode)
    assert _bits_equal(dys, again[0]) and _bits_equal(part, again[2]) and (dxd is None or _bits_equal(dxd, again[1]))
    if dxd_mode != "new":
        plain = _run_bwd_mid(strands, size, gate_off, p, "new")
        assert _bits_equal(dys, plain[0]) and _bits_equal(part, plain[2]) and (dxd is None or _bits_equal(dxd, plain[1]))
    assert part.shape[0] == grid
    # dys_out = D^-1 dy, compared as D dys_out against dy: rows with few entries (large 1/D) would otherwise set the
    # max-norm and the element-wise floor for all the others
    deg = torch.from_numpy(np.diff(g.csr_numpy()[0])).double()
    report = {"dys_out": _panel_errors(dys.double().reshape(n, strands, 128) * deg[:, None, None], ref["dy"])}
    if dxd is not None:
        if gate_off:
            assert bool((dxd == 0).all())
        else:
            report["dxd_out"] = _panel_errors(dxd.reshape(n, strands, 128), ref["dxd"])
    # partial columns d b | d w_g | d b_g, then 3 zeros; per CTA (its window rows, both strands) and in total
    dgp = ref["dgp"]
    terms = torch.cat([ref["dy"], dgp[..., None] * ref["z"], dgp[..., None]], -1)
    cta = torch.arange(n) // rows
    want = torch.zeros(grid, 257, dtype=torch.float64).index_add_(0, cta, terms.sum(1))
    bound = 1e-5 * torch.zeros(grid, 257, dtype=torch.float64).index_add_(0, cta, terms.abs().sum(1))
    got = part.double()
    assert bool((got[:, 257:] == 0).all())
    if gate_off:
        assert bool((got[:, 128:257] == 0).all())
    worst = []
    for diff, bnd in (((got[:, :257] - want).abs(), bound), ((got[:, :257].sum(0) - want.sum(0)).abs(), bound.sum(0))):
        assert bool((diff <= bnd).all()), (diff - bnd).max()
        worst.append(float((diff / bnd)[bnd > 0].max()))
    print("bwd_mid S=%d %s %s: parts %d, %d rows / CTA, %d tiles / CTA | %s | partials err/bound: per CTA %.3f, total %.3f"
          % (strands, size, mode, grid, rows, _cdiv(rows, 64 // strands),
             " | ".join("%s max_rel %.2e elementwise %.2e" % (k, *v) for k, v in report.items()), *worst))


@pytest.mark.parametrize("strands", [1, 2])
@pytest.mark.parametrize("size", ["one_tile", "multi_tile"])
def test_fused_layer_bwd_input_matches_fp64(size, strands):
    """cgcn_gcn_layer_bwd without the layer below (fused_layer_kernel<S, BWD_INPUT>): dx_out = (P dys) W^T + dxd is
    d loss / d x of the layer above, against fp64 autograd; nothing written outside dx_out, bit-identical when repeated."""
    from chromegcn_b200 import ops
    n, g, inp = _bwd_inputs(strands, size)
    x = torch.zeros(n, strands, 128, dtype=torch.float64, requires_grad=True)
    _layer_above(g, inp, x).backward()
    d = {k: v.to(_dev()) for k, v in inp.items()}
    outs = []
    for _ in range(2):
        buf, dx = _guarded(d["dys"].shape)
        assert ops.gcn_layer_bwd(g, d["dys"], d["dxd"], d["w"], dx_out=dx) is dx
        torch.cuda.synchronize()
        assert _guards_intact(buf, n)
        outs.append(dx.cpu())
    assert _bits_equal(outs[0], outs[1])
    grid, rows = _fused_grid(n, strands, _sms())
    print("bwd_input S=%d %s: %d CTAs, %d rows / CTA, %d tiles / CTA | dx_out max_rel %.2e elementwise %.2e"
          % (strands, size, grid, rows, _cdiv(rows, 64 // strands), *_panel_errors(outs[0].reshape(n, strands, 128), x.grad)))


def test_fused_layer_bwd_rejects_invalid_arguments():
    """cgcn_gcn_layer_bwd refuses, before it launches anything, a dys_out that aliases the gathered panel, a missing
    layer-below tensor, a weighted graph and a dropout probability outside [0, 1) -- NaN included, which would otherwise
    switch dropout off without a word."""
    from chromegcn_b200 import _lib, ops
    from chromegcn_b200.graph import HiCGraph
    n, g, inp = _bwd_inputs(2, "one_tile")
    ref = _bwd_mid_reference(2, "one_tile", False, 0.0)
    d = {k: v.to(_dev()) for k, v in inp.items()}
    below = dict(z_prev=ref["z_prev"].to(_dev()), x_prev=d["x_prev"], g_prev=ref["g_prev"].to(_dev()), wg_prev=d["wg"])
    bad = [dict(below, dys_out=d["dys"])] + [dict(below, **{k: None}) for k in ("x_prev", "g_prev", "wg_prev")]
    bad += [dict(below, dropout_p=p) for p in (-0.1, 1.0, 1.5, float("nan"))]
    weighted = HiCGraph(g.rowptr, g.colidx, n, g.nnz, vals=torch.ones(g.nnz, device=_dev()),
                        row_inv=torch.ones(n, device=_dev()))
    before = _lib.launch_count()
    for graph, kw in [(g, k) for k in bad] + [(weighted, below), (weighted, {})]:
        with pytest.raises(_lib.ChromeGCNNativeError):
            ops.gcn_layer_bwd(graph, d["dys"], d["dxd"], d["w"], **kw)
    assert _lib.launch_count() == before
