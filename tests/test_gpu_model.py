"""GPU parity of the model path against the golden vectors minted from the live reference
(tests/golden/make_golden.py) and against the CPU oracle on larger seeded inputs.

Tolerance rule (stated once, used everywhere):
  * forward quantities (logits, gates, loss, probabilities, BatchNorm running stats):
        max|a-b| / max|b|  <=  1e-5   against the reference's fp32 output;
  * gradients: error against the reference's fp64 output <= max(1e-5, 3 x the fp32 reference's own
    error against fp64) -- sums of signed terms over all rows (bias / gate-bias gradients) cancel,
    and the fp32 reference itself is only 1e-5 .. 2e-3 accurate there (tests/test_oracle_golden.py);
  * per-label AUROC / AUPR: <= 1e-4 absolute.
"""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import adjacency as oadj
from oracle import gcn as ogcn

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
FWD_TOL = 1e-5


def _dev():
    return torch.device("cuda", 0)


def _grad_ok(name, got, z, prefix="grad."):
    ref64 = torch.from_numpy(z["f64." + prefix + name])
    own = ogcn.max_rel(torch.from_numpy(z["f32." + prefix + name]), ref64)
    err = ogcn.max_rel(got.detach().cpu(), ref64)
    assert err <= max(1e-5, 3 * own), "%s: err %.3e (fp32 reference's own %.3e)" % (name, err, own)
    return err


def _load(z, layers, dropout=0.0):
    from chromegcn_b200.chrome_models import ChromeGCN
    sd = {k[4:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd0.")}
    m = ChromeGCN(128, 128, sd["out.weight"].shape[0], dropout, True, layers)
    missing = m.load_state_dict(sd)          # the reference's state_dict loads as is
    assert not missing.missing_keys and not missing.unexpected_keys
    return m.to(_dev())


def _graph(z):
    from chromegcn_b200.graph import HiCGraph
    return HiCGraph.from_csr_pattern(z["indptr"], z["indices"], _dev())


@pytest.mark.parametrize("tag", ["l2_ref", "l2_stress", "l1_stress"])
def test_module_api_matches_reference(tag):
    """ChromeGCN.forward called exactly like finetune.py:41-45 (two calls, torch loss, autograd)."""
    z = np.load(os.path.join(GOLDEN, "model_%s.npz" % tag))
    layers = int(z["layers"])
    m = _load(z, layers)
    g = _graph(z)
    x_f = torch.from_numpy(z["x_f"]).to(_dev())
    x_r = torch.from_numpy(z["x_r"]).to(_dev())
    tgt = torch.from_numpy(z["target"]).to(_dev())

    m.eval()
    with torch.no_grad():
        xin, out, (g1, g2), last = m(x_f, g, None)
    assert xin is x_f and last is None
    assert ogcn.max_rel(out.cpu(), torch.from_numpy(z["f32.eval.out_f"])) <= FWD_TOL
    assert ogcn.max_rel(g1.cpu(), torch.from_numpy(z["f32.eval.g1_f"])) <= FWD_TOL
    assert g1.shape == (x_f.shape[0], 1)
    if layers == 2:
        assert ogcn.max_rel(g2.cpu(), torch.from_numpy(z["f32.eval.g2_f"])) <= FWD_TOL
    else:
        assert g2 is None

    m.train()
    x_f.requires_grad_(True)
    x_r.requires_grad_(True)
    _, pf, (g1f, g2f), _ = m(x_f, g, None)
    _, pr, (g1r, g2r), _ = m(x_r, g, None)
    pred = (pf + pr) / 2
    loss = F.binary_cross_entropy_with_logits(pred, tgt)
    loss.backward()
    assert ogcn.max_rel(pred.detach().cpu(), torch.from_numpy(z["f32.train.pred"])) <= FWD_TOL
    assert abs(loss.item() - float(z["f32.train.loss"])) <= FWD_TOL * abs(float(z["f32.train.loss"]))
    assert ogcn.max_rel(g1r.cpu(), torch.from_numpy(z["f32.train.g1_r"])) <= FWD_TOL
    for k, p in m.named_parameters():
        _grad_ok(k, p.grad, z)
    _grad_ok("xgrad_f", x_f.grad, z, prefix="train.")
    _grad_ok("xgrad_r", x_r.grad, z, prefix="train.")
    bn = m.batch_norm
    assert ogcn.max_rel(bn.running_mean.cpu(), torch.from_numpy(z["f32.after.batch_norm.running_mean"])) <= FWD_TOL
    assert ogcn.max_rel(bn.running_var.cpu(), torch.from_numpy(z["f32.after.batch_norm.running_var"])) <= FWD_TOL
    assert int(bn.num_batches_tracked) == 2


@pytest.mark.parametrize("tag", ["l2_ref", "l2_stress", "l1_stress"])
def test_fused_engine_matches_reference(tag):
    """Both strands batched in one cgcn_train_step call (what finetune() uses)."""
    from chromegcn_b200.engine import ChromosomeEngine, flat_params
    z = np.load(os.path.join(GOLDEN, "model_%s.npz" % tag))
    layers = int(z["layers"])
    m = _load(z, layers)
    m.train()
    g = _graph(z)
    eng = ChromosomeEngine(m, 2)
    panel = eng.pack(torch.from_numpy(z["x_f"]).to(_dev()), torch.from_numpy(z["x_r"]).to(_dev()))
    tgt = torch.from_numpy(z["target"]).to(_dev())
    n, c = tgt.shape
    probs = torch.empty(n, c, device=_dev())
    loss = torch.zeros(1, device=_dev())
    xg = torch.empty_like(panel)
    out, gates = eng.run(g, panel, tgt, probs, loss, train=True, input_grad=xg)
    pred = out.mean(1)
    assert ogcn.max_rel(pred.cpu(), torch.from_numpy(z["f32.train.pred"])) <= FWD_TOL
    assert ogcn.max_rel(probs.cpu(), torch.sigmoid(torch.from_numpy(z["f32.train.pred"]))) <= FWD_TOL
    assert abs(loss.item() - float(z["f32.train.loss"])) <= FWD_TOL * abs(float(z["f32.train.loss"]))
    assert ogcn.max_rel(gates[0][:, 0].cpu(), torch.from_numpy(z["f32.train.g1_f"])[:, 0]) <= FWD_TOL
    assert ogcn.max_rel(gates[0][:, 1].cpu(), torch.from_numpy(z["f32.train.g1_r"])[:, 0]) <= FWD_TOL
    if layers == 2:
        assert ogcn.max_rel(gates[1][:, 1].cpu(), torch.from_numpy(z["f32.train.g2_r"])[:, 0]) <= FWD_TOL
    for k, p in m.named_parameters():
        _grad_ok(k, p.grad, z)
    _grad_ok("xgrad_f", xg[:, 0], z, prefix="train.")
    _grad_ok("xgrad_r", xg[:, 1], z, prefix="train.")
    assert ogcn.max_rel(m.batch_norm.running_var.cpu(), torch.from_numpy(z["f32.after.batch_norm.running_var"])) <= FWD_TOL
    assert int(m.batch_norm.num_batches_tracked) == 2
    # parameters are views of one flat buffer and .grad of one flat gradient buffer
    fp = flat_params(m)
    assert all(p.data_ptr() >= fp.flat.data_ptr() and p.data_ptr() < fp.flat.data_ptr() + 4 * fp.total
               for p in m.parameters())
    # without input gradients the result is the same (first-layer backward SpMM skipped)
    m2 = _load(z, layers)
    m2.train()
    eng2 = ChromosomeEngine(m2, 2)
    loss2 = torch.zeros(1, device=_dev())
    eng2.run(g, eng2.pack(torch.from_numpy(z["x_f"]).to(_dev()), torch.from_numpy(z["x_r"]).to(_dev())), tgt, None, loss2,
             train=True)
    for (k, p), (_, q) in zip(m.named_parameters(), m2.named_parameters()):
        assert torch.equal(p.grad, q.grad), k


@pytest.mark.parametrize("d,gemm_impl", [(256, 0), (512, 0), (512, 1)])
def test_wide_model_matches_fp64_oracle(d, gemm_impl):
    """d_model 256 / 512 (BASELINE.json's stress configuration; the reference class is generic in nfeat,
    models/ChromeModels.py:24-31): the fused step -- width-2d SpMM, weight operands cut into 128 x 128 blocks on
    the tensor cores, DV = d/128 row kernels -- against the fp64 oracle on the same inputs."""
    from chromegcn_b200 import synthetic
    from chromegcn_b200.chrome_models import ChromeGCN
    from chromegcn_b200.engine import ChromosomeEngine
    from chromegcn_b200.graph import HiCGraph
    from oracle import adjacency as oadj
    h = synthetic.make_hic("chr22", hic_edges=8000, n_windows=900, n_bins=2400)
    ip, ix = oadj.build_adjacency_numpy(h.window_starts, h.bin1, h.bin2, h.val, h.norm, 1, 8000)
    n, nclass = ip.shape[0] - 1, 19
    gen = torch.Generator().manual_seed(d)
    xf, xr = torch.randn(n, d, generator=gen), torch.randn(n, d, generator=gen)
    tgt = (torch.rand(n, nclass, generator=gen) < 0.2).float()
    torch.manual_seed(3)
    om = ogcn.stress_init_(ogcn.ChromeGCNOracle(d, d, nclass, 0.0, True, 2))
    m = ChromeGCN(d, d, nclass, 0.0, True, 2)
    m.load_state_dict(om.state_dict())
    m = m.to(_dev()).train()
    m.gemm_impl = gemm_impl
    g = HiCGraph.from_csr_pattern(ip, ix, _dev())
    eng = ChromosomeEngine(m, 2)
    probs, loss = torch.empty(n, nclass, device=_dev()), torch.zeros(1, device=_dev())
    xg = torch.empty(n, 2, d, device=_dev())
    out, gates = eng.run(g, eng.pack(xf.to(_dev()), xr.to(_dev())), tgt.to(_dev()), probs, loss, train=True, input_grad=xg)
    grads = {k: p.grad.detach().cpu().clone() for k, p in m.named_parameters()}
    om = om.double().train()
    lo, prob_o, pred_o, ex = ogcn.chromosome_step(om, xf.double(), xr.double(), tgt.double(),
                                                  ogcn.coo_adjacency(ip, ix, torch.float64), None, True, input_grads=True)
    xf64, xr64 = ex["x_f"], ex["x_r"]
    assert ogcn.max_rel(out.mean(1).cpu(), pred_o) <= FWD_TOL
    assert ogcn.max_rel(probs.cpu(), prob_o) <= FWD_TOL
    assert abs(loss.item() - lo) <= FWD_TOL * abs(lo)
    for k, q in om.named_parameters():
        err = ogcn.max_rel(grads[k], q.grad)
        assert err <= 5e-5, (k, err)
    assert ogcn.max_rel(xg[:, 0].cpu(), xf64.grad) <= 5e-5 and ogcn.max_rel(xg[:, 1].cpu(), xr64.grad) <= 5e-5
    # eval mode through the module API (one strand per call, models/ChromeModels.py:34-52)
    m.eval()
    om.eval()
    with torch.no_grad():
        _, o1, (g1, g2), _ = m(xf.to(_dev()), g, None)
        _, o2, (h1, h2), _ = om(xf.double(), ogcn.coo_adjacency(ip, ix, torch.float64), None)
    assert ogcn.max_rel(o1.cpu(), o2) <= FWD_TOL and ogcn.max_rel(g2.cpu(), h2) <= FWD_TOL


def test_reference_sparse_tensor_is_accepted():
    """The adjacency the reference's own process_graph returns (torch sparse COO) drops in."""
    z = np.load(os.path.join(GOLDEN, "model_l2_stress.npz"))
    m = _load(z, 2).eval()
    coo = ogcn.coo_adjacency(z["indptr"], z["indices"]).to(_dev())
    x = torch.from_numpy(z["x_f"]).to(_dev())
    with torch.no_grad():
        _, a, _, _ = m(x, coo, None)
        _, b, _, _ = m(x, _graph(z), None)
    assert torch.equal(a, b)
    assert ogcn.max_rel(a.cpu(), torch.from_numpy(z["f32.eval.out_f"])) <= FWD_TOL
    with pytest.raises(Exception):
        m(x.cpu(), coo, None)                      # no CPU fallback


def test_dropout_training_matches_oracle_with_injected_masks():
    """Train mode with gcn_dropout 0.2: the oracle is fed the keep-masks the CUDA path drew."""
    from chromegcn_b200 import ops
    from chromegcn_b200.engine import ChromosomeEngine
    z = np.load(os.path.join(GOLDEN, "model_l2_stress.npz"))
    p = 0.2
    # The dropout seed is drawn from torch's generator: seed it so that the masks do not depend on which tests ran
    # before in this process.  Bias gradients are single sums over all rows and cancel more for some masks than for
    # others: unseeded, one draw left W2.bias 1.8e-4 (max-rel) from the fp64 oracle, and on such masks the fp32
    # oracle itself reaches 5e-5 on W1.bias.  With this seed the fp32 oracle stays within 7e-6 on every bias.
    torch.manual_seed(0)
    m = _load(z, 2, dropout=p)
    m.train()
    g = _graph(z)
    eng = ChromosomeEngine(m, 2)
    x_f, x_r, tgt = (torch.from_numpy(z[k]) for k in ("x_f", "x_r", "target"))
    n = x_f.shape[0]
    probs = torch.empty(n, tgt.shape[1], device=_dev())
    loss = torch.zeros(1, device=_dev())
    out, _ = eng.run(g, eng.pack(x_f.to(_dev()), x_r.to(_dev())), tgt.to(_dev()), probs, loss, train=True)
    seed, step = m._drop_seed, m._drop_step
    mid = ops.dropout_mask(n, 2, 128, p, seed, step, 0).cpu()
    head = ops.dropout_mask(n, 2, 128, p, seed, step, 1).cpu()
    assert 0.15 < float((mid == 0).float().mean()) < 0.25
    om = ogcn.ChromeGCNOracle(128, 128, tgt.shape[1], p, True, 2).double()
    om.load_state_dict({k[4:]: torch.from_numpy(z[k]).double() for k in z.files if k.startswith("sd0.")})
    om.train()
    adj = ogcn.coo_adjacency(z["indptr"], z["indices"], torch.float64)
    lo, prob_o, pred_o, _ = ogcn.chromosome_step(om, x_f.double(), x_r.double(), tgt.double(), adj, None, True,
                                                 masks_f=(mid[:, 0].double(), head[:, 0].double()),
                                                 masks_r=(mid[:, 1].double(), head[:, 1].double()))
    assert ogcn.max_rel(out.mean(1).cpu(), pred_o) <= FWD_TOL
    assert abs(loss.item() - lo) <= FWD_TOL * abs(lo)
    for (k, pp), (_, q) in zip(m.named_parameters(), om.named_parameters()):
        err = ogcn.max_rel(pp.grad.cpu(), q.grad)
        assert err <= 5e-5, (k, err)              # fp32 vs fp64 oracle, cancellation-prone sums included


def test_large_graph_against_oracle():
    """Config-1 sized chromosomes (N = 20 000) vs the CPU oracle in fp64, through both entry points: the fused step (both
    strands in one cgcn_train_step) and the module API (finetune.py:41-48: one strand per call, BCE on the mean,
    backward).  With 500 k Hi-C edges (520 k stored entries, mean degree 26) every layer runs as three kernels.  With
    400 k (mean degree 21) every layer runs as the fused layer kernel, and on 148 SMs each CTA of it runs several tiles:
    136 rows = 3 tiles of 64 with one strand, 5 of 32 with two, the last tile holding 8 rows."""
    from chromegcn_b200 import synthetic
    from chromegcn_b200.chrome_models import ChromeGCN
    from chromegcn_b200.engine import ChromosomeEngine
    from chromegcn_b200.graph import HiCGraph
    from oracle import adjacency as oadj
    for hic_edges, fused in ((500000, False), (400000, True)):
        h = synthetic.make_hic("chr22", hic_edges=hic_edges)
        ip, ix = oadj.build_adjacency_numpy(h.window_starts, h.bin1, h.bin2, h.val, h.norm, 1, hic_edges)
        n = ip.shape[0] - 1
        feats = synthetic.make_features("chr22", n)
        torch.manual_seed(0)
        om = ogcn.ChromeGCNOracle(128, 128, synthetic.NCLASS, 0.0, True, 2)
        ogcn.stress_init_(om)
        sd = {k: v.clone() for k, v in om.state_dict().items()}
        m = ChromeGCN(128, 128, synthetic.NCLASS, 0.0, True, 2)
        m.load_state_dict(sd)
        m = m.to(_dev()).train()
        om = om.double().train()
        adj = ogcn.coo_adjacency(ip, ix, torch.float64)
        lo, prob_o, pred_o, _ = ogcn.chromosome_step(om, feats["forward"].double(), feats["backward"].double(),
                                                     feats["target"].double(), adj, None, True)
        g = HiCGraph.from_csr_pattern(ip, ix, _dev())
        assert g.nnz == ip[-1] + n
        assert (g.nnz <= 24 * n) == fused          # FUSED_MAX_DEGREE (csrc/model.cu) selects the layer path
        eng = ChromosomeEngine(m, 2)
        probs = torch.empty(n, synthetic.NCLASS, device=_dev())
        loss = torch.zeros(1, device=_dev())
        out, _ = eng.run(g, eng.pack(feats["forward"].to(_dev()), feats["backward"].to(_dev())), feats["target"].to(_dev()),
                         probs, loss, train=True)
        # the module API on the same model and inputs
        m1 = ChromeGCN(128, 128, synthetic.NCLASS, 0.0, True, 2)
        m1.load_state_dict(sd)
        m1 = m1.to(_dev()).train()
        _, pf, _, _ = m1(feats["forward"].to(_dev()), g, None)
        _, pr, _, _ = m1(feats["backward"].to(_dev()), g, None)
        pred1 = (pf + pr) / 2
        loss1 = F.binary_cross_entropy_with_logits(pred1, feats["target"].to(_dev()))
        loss1.backward()
        for arm, model, pred, prob, l in (("engine", m, out.mean(1), probs, loss.item()),
                                          ("module", m1, pred1.detach(), torch.sigmoid(pred1.detach()), loss1.item())):
            errs = [ogcn.max_rel(pred.cpu(), pred_o), ogcn.max_rel(prob.cpu(), prob_o), abs(l - lo) / abs(lo)]
            assert max(errs) <= FWD_TOL, (hic_edges, arm, errs)
            for (k, p), (_, q) in zip(model.named_parameters(), om.named_parameters()):
                err = ogcn.max_rel(p.grad.cpu(), q.grad)
                assert err <= 5e-5, (hic_edges, arm, k, err)
                errs.append(err)
            print("large graph, %d Hi-C edges, %s: pred %.2e prob %.2e loss %.2e, worst gradient %.2e"
                  % (hic_edges, arm, *errs[:3], max(errs[3:])))


def _auc_aupr(targets, preds):
    from sklearn import metrics as skm
    aucs, auprs = [], []
    for i in range(targets.shape[1]):
        if targets[:, i].min() == targets[:, i].max():
            continue
        aucs.append(skm.roc_auc_score(targets[:, i], preds[:, i]))                     # utils/metrics.py:244
        pr, rc, _ = skm.precision_recall_curve(targets[:, i], preds[:, i], pos_label=1)  # utils/metrics.py:172-173
        auprs.append(skm.auc(rc, pr))
    return np.array(aucs), np.array(auprs)


@pytest.mark.parametrize("optim_kind,gemm_impl", [("flat", 1), ("torch", 1), ("flat", 0)])
def test_finetune_matches_reference(tmp_path, optim_kind, gemm_impl):
    """Three epochs of finetune() (train on 2 chromosomes, validate on 1) against the reference's own
    finetune.py run: losses, probabilities, per-label AUROC / AUPR, final state_dict.

    gemm_impl 1 (exact-fp32 FFMA contractions) must track the fp64 trajectory as tightly as the fp32
    reference does.  gemm_impl 0 (tcgen05 3xTF32, ~1e-6 per contraction) is checked more loosely over
    the trajectory (loss 2e-3 relative, probabilities 2e-2 absolute, mean AUROC / AUPR 2e-3): a 1e-6
    perturbation can put a pre-ReLU activation on the other side of zero (|h| < 2e-6; observed on chr2,
    row 12 strand 0 column 33), which switches that element's gradient on or off.  On these 157-row
    chromosomes with lr 0.25 and weight gradients that cancel to ~1e-3, one such element moves a step by
    ~1e-4 and six steps compound it; either side of the kink is a valid fp32 evaluation (the fp32
    reference sits on one of them by the same chance).  Same-weights parity of the tcgen05 path (1e-5,
    per-label AUROC / AUPR 1e-4) is asserted in test_eval_from_reference_weights_auroc_aupr."""
    import argparse
    import pickle
    from scipy import sparse
    from chromegcn_b200.chrome_models import ChromeGCN
    from chromegcn_b200 import finetune as ft
    from chromegcn_b200.optim import get_optimizer
    z = np.load(os.path.join(GOLDEN, "finetune.npz"))
    nclass = int(z["nclass"])
    sd = {k[4:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd0.")}
    m = ChromeGCN(128, 128, nclass, 0.0, True, 2)
    m.load_state_dict(sd)
    m = m.to(_dev())
    m.gemm_impl = gemm_impl
    strict = gemm_impl == 1
    graphs = {}
    for c in ("chr1", "chr2", "chr3"):
        ip, ix = z[c + ".indptr"], z[c + ".indices"]
        n = ip.shape[0] - 1
        graphs[c] = sparse.csr_matrix((np.ones(ix.shape[0]), ix, ip), shape=(n, n))
    with open(tmp_path / "train_graphs_1200_SQRTVCnorm.pkl", "wb") as fp:
        pickle.dump({c: graphs[c] for c in ("chr1", "chr2")}, fp)
    with open(tmp_path / "valid_graphs_1200_SQRTVCnorm.pkl", "wb") as fp:
        pickle.dump({"chr3": graphs["chr3"]}, fp)
    opt = argparse.Namespace(adj_type="hic", graph_root=str(tmp_path), hicsize="1200", hicnorm="SQRTVC", optim="sgd", lr=0.25)
    optimizer = (get_optimizer(m, opt) if optim_kind == "flat"
                 else torch.optim.SGD(m.parameters(), lr=0.25, weight_decay=1e-6, momentum=0.9))
    feats = lambda cs: {c: {k: torch.from_numpy(z["%s.%s" % (c, k)]) for k in ("forward", "backward", "target")} for c in cs}
    train_d, valid_d = feats(["chr1", "chr2"]), feats(["chr3"])
    ft.clear_caches()
    # fp64 trajectory of the same recipe (CPU oracle): the yardstick.  Rule: error against fp64 <=
    # max(2e-5, 3 x the fp32 reference's own error against fp64) -- six SGD steps at lr 0.25 amplify the
    # reference's own fp32 rounding (its bias gradients are only 1e-5..2e-3 accurate) by about that much.
    o64 = ogcn.ChromeGCNOracle(128, 128, nclass, 0.0, True, 2)
    o64.load_state_dict(sd)
    o64 = o64.double()
    oopt = ogcn.make_optimizer(o64, "sgd", 0.25)
    og = {c: (z[c + ".indptr"], z[c + ".indices"]) for c in ("chr1", "chr2", "chr3")}
    dbl = lambda d: {c: {k: v.double() for k, v in f.items()} for c, f in d.items()}

    def close(ours, ref32, ref64, what):
        own = ogcn.max_rel(torch.as_tensor(ref32), ref64)
        err = ogcn.max_rel(torch.as_tensor(ours), ref64)
        tol = max(2e-5, 3 * own) if strict else 2e-2
        assert err <= tol, "%s: err %.2e, fp32 reference's own %.2e" % (what, err, own)

    for epoch in (1, 2, 3):
        p, t, l = ft.finetune(None, m, train_d, None, optimizer, epoch, None, opt, "train")
        pv, tv, lv = ft.finetune(None, m, valid_d, None, optimizer, epoch, None, opt, "valid")
        p64, _, l64 = ogcn.finetune_epoch(o64, dbl(train_d), og, oopt, "train")
        pv64, _, lv64 = ogcn.finetune_epoch(o64, dbl(valid_d), og, oopt, "valid")
        assert not p.is_cuda and p.shape == (t.shape[0], nclass)
        gp, gpv = z["epoch%d.train_preds" % epoch], z["epoch%d.valid_preds" % epoch]
        close(p, gp, p64, "train preds epoch %d" % epoch)
        close(pv, gpv, pv64, "valid preds epoch %d" % epoch)
        close([l], [float(z["epoch%d.train_loss" % epoch])], torch.tensor([l64]), "train loss")
        close([lv], [float(z["epoch%d.valid_loss" % epoch])], torch.tensor([lv64]), "valid loss")
        ltol = 1e-4 if strict else 2e-3
        assert abs(l - l64) <= ltol * abs(l64) and abs(lv - lv64) <= ltol * abs(lv64)
        for ours, ref, targ in ((p.numpy(), gp, t.numpy()), (pv.numpy(), gpv, tv.numpy())):
            a1, r1 = _auc_aupr(targ, ours)
            a2, r2 = _auc_aupr(targ, ref)
            if strict:
                assert np.abs(a1 - a2).max() <= 1e-4 and np.abs(r1 - r2).max() <= 1e-4
            else:
                assert abs(a1.mean() - a2.mean()) <= 2e-3 and abs(r1.mean() - r2.mean()) <= 2e-3
    for k, v in m.state_dict().items():
        if "num_batches" in k:
            assert int(v) == int(z["sd3." + k])
            continue
        close(v.float().cpu(), z["sd3." + k], o64.state_dict()[k], "state_dict " + k)


def test_finetune_bit_packed_labels_identical_to_float_labels(tmp_path):
    """finetune() moves the 0/1 label matrix host -> device as bit rows (cgcn_train_step_bits / cgcn_bce_loss_bits);
    `opt.pack_labels = False` keeps the float matrix of finetune.py:32.  Same kernels, same order of operations:
    predictions, losses and the trained weights must be bit-identical.  Soft labels fall back to the float path."""
    import argparse
    import pickle
    from scipy import sparse
    from chromegcn_b200.chrome_models import ChromeGCN
    from chromegcn_b200 import finetune as ft
    from chromegcn_b200.optim import get_optimizer
    z = np.load(os.path.join(GOLDEN, "finetune.npz"))
    nclass = int(z["nclass"])
    sd = {k[4:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd0.")}
    graphs = {}
    for c in ("chr1", "chr2"):
        ip, ix = z[c + ".indptr"], z[c + ".indices"]
        graphs[c] = sparse.csr_matrix((np.ones(ix.shape[0]), ix, ip), shape=(ip.shape[0] - 1,) * 2)
    for split in ("train", "valid"):
        with open(tmp_path / ("%s_graphs_1200_SQRTVCnorm.pkl" % split), "wb") as fp:
            pickle.dump(graphs, fp)
    feats = {c: {k: torch.from_numpy(z["%s.%s" % (c, k)]) for k in ("forward", "backward", "target")} for c in ("chr1", "chr2")}
    assert all(ft.packed_target(f["target"]) is not None for f in feats.values())
    results = []
    for pack in (True, False):
        ft.clear_caches()
        torch.manual_seed(7)                                   # the dropout stream's seed is drawn from torch's generator
        m = ChromeGCN(128, 128, nclass, 0.2, True, 2)
        m.load_state_dict(sd)
        m = m.to(_dev())
        opt = argparse.Namespace(adj_type="hic", graph_root=str(tmp_path), hicsize="1200", hicnorm="SQRTVC", optim="sgd", lr=0.25,
                                 pack_labels=pack)
        optimizer = get_optimizer(m, opt)
        run = []
        for epoch in (1, 2):
            p, t, l = ft.finetune(None, m, feats, None, optimizer, epoch, None, opt, "train")
            pv, _, lv = ft.finetune(None, m, feats, None, optimizer, epoch, None, opt, "valid")
            run += [p.clone(), torch.tensor(l), pv.clone(), torch.tensor(lv)]
        run += [v.detach().cpu().clone() for v in m.state_dict().values()]
        results.append(run)
    for a, b in zip(*results):
        assert torch.equal(a, b)
    soft = {c: dict(f) for c, f in feats.items()}
    soft["chr1"]["target"] = soft["chr1"]["target"] * 0.75
    assert ft.packed_target(soft["chr1"]["target"]) is None
    p, _, l = ft.finetune(None, m, soft, None, optimizer, 3, None, opt, "valid")
    assert np.isfinite(l) and torch.isfinite(p).all()


@pytest.mark.parametrize("gemm_impl", [0, 1])
def test_eval_from_reference_weights_auroc_aupr(gemm_impl):
    """The reference's trained weights (state_dict after its own 3 epochs) evaluated on the CUDA path:
    probabilities within 1e-5 of the reference's, per-label AUROC / AUPR within 1e-4 (north-star criteria)."""
    from chromegcn_b200.chrome_models import ChromeGCN
    from chromegcn_b200.engine import ChromosomeEngine
    from chromegcn_b200.graph import HiCGraph
    z = np.load(os.path.join(GOLDEN, "finetune.npz"))
    nclass = int(z["nclass"])
    sd = {k[4:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd3.")}
    m = ChromeGCN(128, 128, nclass, 0.0, True, 2)
    m.load_state_dict(sd)
    m = m.to(_dev()).eval()
    m.gemm_impl = gemm_impl
    eng = ChromosomeEngine(m, 2)
    c = "chr3"
    g = HiCGraph.from_csr_pattern(z[c + ".indptr"], z[c + ".indices"], _dev())
    xf, xr, t = (torch.from_numpy(z["%s.%s" % (c, k)]) for k in ("forward", "backward", "target"))
    probs = torch.empty(xf.shape[0], nclass, device=_dev())
    loss = torch.zeros(1, device=_dev())
    eng.run(g, eng.pack(xf.to(_dev()), xr.to(_dev())), t.to(_dev()), probs, loss, train=False)
    ref = z["epoch3.valid_preds"]                       # the reference's own validation pass after epoch 3
    assert ogcn.max_rel(probs.cpu(), torch.from_numpy(ref)) <= FWD_TOL
    assert abs(loss.item() - float(z["epoch3.valid_loss"])) <= FWD_TOL * abs(float(z["epoch3.valid_loss"]))
    a1, r1 = _auc_aupr(t.numpy(), probs.cpu().numpy())
    a2, r2 = _auc_aupr(t.numpy(), ref)
    assert np.abs(a1 - a2).max() <= 1e-4 and np.abs(r1 - r2).max() <= 1e-4


@pytest.mark.parametrize("layers,gate", [(3, True), (2, False), (3, False), (4, True), (1, False)])
def test_extension_variants_match_oracle(layers, gate):
    """Variant sweep of BASELINE.json ("gcn_layers 3", "gate off"): `ChromeGCN(..., extended=True)` against the
    extension oracle in fp64, train mode with dropout (keep-masks injected), fused two-strand step with input
    gradients.  Same tolerances as the reference-pinned tests."""
    from chromegcn_b200 import ops
    from chromegcn_b200.chrome_models import ChromeGCN
    from chromegcn_b200.engine import ChromosomeEngine
    z = np.load(os.path.join(GOLDEN, "model_l2_stress.npz"))
    x_f, x_r, tgt = (torch.from_numpy(z[k]) for k in ("x_f", "x_r", "target"))
    n, c = tgt.shape
    p = 0.2
    torch.manual_seed(11)
    om = ogcn.stress_init_(ogcn.ChromeGCNExtOracle(128, 128, c, p, gate, layers), seed=5)
    m = ChromeGCN(128, 128, c, p, gate, layers, extended=True)
    missing = m.load_state_dict(om.state_dict())
    assert not missing.missing_keys and not missing.unexpected_keys
    assert m.num_layers == layers and m.gate_off == (not gate)
    m = m.to(_dev()).train()
    g = _graph(z)
    eng = ChromosomeEngine(m, 2)
    probs = torch.empty(n, c, device=_dev())
    loss = torch.zeros(1, device=_dev())
    panel = eng.pack(x_f.to(_dev()), x_r.to(_dev()))
    xg = torch.empty_like(panel)
    out, gates = eng.run(g, panel, tgt.to(_dev()), probs, loss, train=True, input_grad=xg)
    seed, step = m._drop_seed, m._drop_step
    sites = [0 if l == 0 else l + 1 for l in range(layers - 1)] + [1]  # after layer 1, after layer l+1 ..., after BatchNorm
    masks = [ops.dropout_mask(n, 2, 128, p, seed, step, s).cpu().double() for s in sites]
    if layers >= 3:
        assert not torch.equal(masks[0], masks[1])                     # every site draws its own mask
    om = om.double().train()
    adj = ogcn.coo_adjacency(z["indptr"], z["indices"], torch.float64)
    lo, prob_o, pred_o, ex = ogcn.chromosome_step(om, x_f.double(), x_r.double(), tgt.double(), adj, None, True,
                                                  masks_f=[mk[:, 0] for mk in masks], masks_r=[mk[:, 1] for mk in masks],
                                                  input_grads=True)
    assert ogcn.max_rel(out.mean(1).cpu(), pred_o) <= FWD_TOL
    assert ogcn.max_rel(probs.cpu(), prob_o) <= FWD_TOL
    assert abs(loss.item() - lo) <= FWD_TOL * abs(lo)
    assert len(gates) == layers
    for l in range(layers):
        assert ogcn.max_rel(gates[l][:, 0].cpu(), ex["gates_f"][l][:, 0]) <= FWD_TOL
    for (k, pp), (_, q) in zip(m.named_parameters(), om.named_parameters()):
        if q.grad is None:                                             # gate parameters of a gate-off model
            assert float(pp.grad.abs().max()) == 0.0, k
            continue
        err = ogcn.max_rel(pp.grad.cpu(), q.grad)
        assert err <= 5e-5, (k, err)
    assert ogcn.max_rel(xg[:, 0].cpu(), ex["x_f"].grad) <= 5e-5
    assert ogcn.max_rel(xg[:, 1].cpu(), ex["x_r"].grad) <= 5e-5
    # module API (one strand, autograd) agrees with the fused step's forward in eval mode
    m.eval()
    om.eval()
    with torch.no_grad():
        _, o1, (g1, g2), _ = m(x_f.to(_dev()), g, None)
        _, o2, og, _ = om(x_f.double(), adj)
    assert ogcn.max_rel(o1.cpu(), o2) <= FWD_TOL
    assert (g2 is None) == (layers == 1) and len(m.last_gates) == layers


def test_sharded_epoch_round_is_one_step_on_the_mean_gradient():
    """Chromosome-sharded data parallelism (SURVEY.md F11 / 8(e)): a round = the chromosomes the ranks process at the
    same weights, ONE optimiser step on the mean of their gradients.  On one rank a cell holding several chromosomes
    goes through the same accumulate / scale / step code as the all-reduce path; the result must equal the oracle's
    per-chromosome gradients (finetune.py:39-48 at fixed weights) averaged and applied by SGD
    (utils/util_methods.py:18-19)."""
    from chromegcn_b200 import dist as cdist, synthetic, ops
    from chromegcn_b200.chrome_models import ChromeGCN
    from chromegcn_b200.engine import ChromosomeEngine
    from chromegcn_b200.graph import HiCGraph
    from chromegcn_b200.optim import FlatSGD
    from oracle import adjacency as oadj
    nclass, chroms = 9, ["chr20", "chr21", "chr22"]
    graphs, og, feats, panels, targets, probs = {}, {}, {}, {}, {}, {}
    for i, c in enumerate(chroms):
        h = synthetic.make_hic(c, hic_edges=3000, n_windows=300 + 40 * i, n_bins=900)
        ip, ix = oadj.build_adjacency_numpy(h.window_starts, h.bin1, h.bin2, h.val, h.norm, 1, 3000)
        n = ip.shape[0] - 1
        og[c] = ogcn.coo_adjacency(ip, ix, torch.float64)
        graphs[c] = HiCGraph.from_csr_pattern(ip, ix, _dev())
        feats[c] = synthetic.make_features(c, n, 128, nclass)
        panels[c] = ops.interleave_strands([feats[c]["forward"].to(_dev()), feats[c]["backward"].to(_dev())])
        targets[c] = feats[c]["target"].to(_dev())
        probs[c] = torch.empty(n, nclass, device=_dev())
    torch.manual_seed(2)
    om = ogcn.stress_init_(ogcn.ChromeGCNOracle(128, 128, nclass, 0.0, True, 2))
    m = ChromeGCN(128, 128, nclass, 0.0, True, 2)
    m.load_state_dict(om.state_dict())
    m = m.to(_dev()).train()
    m.gemm_impl = 1
    om = om.double().train()
    schedule = [[["chr20", "chr22"]], [["chr21"]]]                 # round 1: two chromosomes at the same weights
    losses = torch.zeros(3, device=_dev())
    opt = FlatSGD(m, lr=0.25)
    cdist.sharded_train_epoch(ChromosomeEngine(m, 2), opt, schedule, 0, graphs, panels, targets, probs, losses)
    oopt = ogcn.make_optimizer(om, "sgd", 0.25)
    want_losses = []
    for rnd in schedule:
        acc = None
        for c in rnd[0]:
            oopt.zero_grad()
            lo, _, _, _ = ogcn.chromosome_step(om, feats[c]["forward"].double(), feats[c]["backward"].double(),
                                               feats[c]["target"].double(), og[c], None, True)
            want_losses.append(lo)
            g = [p.grad.clone() for p in om.parameters()]
            acc = g if acc is None else [a + b for a, b in zip(acc, g)]
        for p, a in zip(om.parameters(), acc):
            p.grad = a / len(rnd[0])
        oopt.step()
    assert ogcn.max_rel(losses.cpu(), torch.tensor(want_losses)) <= FWD_TOL
    for (k, p), (_, q) in zip(m.named_parameters(), om.named_parameters()):
        assert ogcn.max_rel(p.detach().cpu(), q.detach()) <= 2e-5, k


def test_module_api_training_loop_with_flat_optimizer_matches_oracle():
    """The reference's own loop -- optimizer.zero_grad(); forward x2 through the module API; loss.backward();
    optimizer.step() (finetune.py:39-49) -- for several steps with this package's ChromeGCN and get_optimizer().  After the
    first step every p.grad is a view of the flat gradient buffer and autograd ACCUMULATES into it, so zero_grad() must
    really clear it (ADVICE r01): the trajectory has to follow the oracle's, not the running sum of gradients."""
    import argparse
    from chromegcn_b200 import synthetic
    from chromegcn_b200.chrome_models import ChromeGCN
    from chromegcn_b200.graph import HiCGraph
    from chromegcn_b200.optim import get_optimizer
    h = synthetic.make_hic("chr21", hic_edges=4000, n_windows=500, n_bins=1400)
    ip, ix = oadj.build_adjacency_numpy(h.window_starts, h.bin1, h.bin2, h.val, h.norm, 1, 4000)
    n = ip.shape[0] - 1
    f = synthetic.make_features("chr21", n, 128, 9)
    for kind in ("sgd", "adam"):
        torch.manual_seed(11)
        om = ogcn.stress_init_(ogcn.ChromeGCNOracle(128, 128, 9, 0.0, True, 2))
        m = ChromeGCN(128, 128, 9, 0.0, True, 2)
        m.load_state_dict(om.state_dict())
        m = m.to(_dev()).train()
        lr = 0.05 if kind == "sgd" else 1e-3
        opt = get_optimizer(m, argparse.Namespace(optim=kind, lr=lr))
        oopt = ogcn.make_optimizer(om, kind, lr)
        g = HiCGraph.from_csr_pattern(ip, ix, _dev())
        adj = ogcn.coo_adjacency(ip, ix)
        xf, xr, tg = f["forward"].to(_dev()), f["backward"].to(_dev()), f["target"].to(_dev())
        for step in range(4):
            opt.zero_grad()
            _, pf, _, _ = m(xf, g, None)
            _, pr, _, _ = m(xr, g, None)
            loss = torch.nn.functional.binary_cross_entropy_with_logits((pf + pr) / 2, tg)
            loss.backward()
            opt.step()
            lo, _, _, _ = ogcn.chromosome_step(om, f["forward"], f["backward"], f["target"], adj, oopt, True)
            assert abs(loss.item() - lo) <= 2e-5 * abs(lo), (kind, step, loss.item(), lo)
        for k, v in om.state_dict().items():
            if "num_batches" in k:
                continue
            assert ogcn.max_rel(m.state_dict()[k].cpu(), v) <= 1e-4, (kind, k)


def test_three_epoch_trajectory_on_a_chr22_sized_graph_keeps_per_label_auroc_aupr():
    """VERDICT r01 item 4: on the DEFAULT path (fused layer kernels, tcgen05 3xTF32 contractions) a three-epoch
    finetune() trajectory on a C1-sized graph (N = 20 000: one ReLU sign flip cannot move a step by 1e-4 there) ends
    with per-label AUROC / AUPR within 1e-4 of the fp64 oracle's trajectory, probabilities within 1e-4."""
    import argparse
    import pickle
    from scipy import sparse
    from sklearn.metrics import average_precision_score, roc_auc_score
    from chromegcn_b200 import finetune as ft, synthetic
    from chromegcn_b200.chrome_models import ChromeGCN
    from chromegcn_b200.optim import get_optimizer
    import tempfile
    nclass = 12
    h = synthetic.make_hic("chr22", hic_edges=200000)
    ip, ix = oadj.build_adjacency_numpy(h.window_starts, h.bin1, h.bin2, h.val, h.norm, 1, 200000)
    n = ip.shape[0] - 1
    gen = torch.Generator().manual_seed(5)
    xf = torch.randn(n, 128, generator=gen)
    xr = xf + 0.2 * torch.randn(n, 128, generator=gen)
    wtrue = torch.randn(128, nclass, generator=gen)
    tgt = ((xf @ wtrue) > 8.0).float()                       # learnable labels, a few per cent positives
    feats = {"chr22": {"forward": xf, "backward": xr, "target": tgt}}
    tmp = tempfile.mkdtemp()
    for split in ("train", "valid"):
        with open(os.path.join(tmp, "%s_graphs_200000_SQRTVCnorm.pkl" % split), "wb") as fp:
            pickle.dump({"chr22": sparse.csr_matrix((np.ones(ix.shape[0]), ix, ip), shape=(n, n))}, fp)
    opt = argparse.Namespace(adj_type="hic", graph_root=tmp, hicsize="200000", hicnorm="SQRTVC", optim="sgd", lr=0.25)
    torch.manual_seed(2)
    o64 = ogcn.ChromeGCNOracle(128, 128, nclass, 0.0, True, 2)
    m = ChromeGCN(128, 128, nclass, 0.0, True, 2)
    m.load_state_dict(o64.state_dict())
    m = m.to(_dev())
    assert m.gemm_impl == 0
    optimizer = get_optimizer(m, opt)
    o64 = o64.double()
    oopt = ogcn.make_optimizer(o64, "sgd", 0.25)
    f64 = {"chr22": {k: v.double() for k, v in feats["chr22"].items()}}
    ft.clear_caches()
    for epoch in (1, 2, 3):
        _, _, l = ft.finetune(None, m, feats, None, optimizer, epoch, None, opt, "train")
        _, _, l64 = ogcn.finetune_epoch(o64, f64, {"chr22": (ip, ix)}, oopt, "train")
        assert abs(l - l64) <= 1e-5 * abs(l64), (epoch, l, l64)
    pv, _, _ = ft.finetune(None, m, feats, None, optimizer, 3, None, opt, "valid")
    pv64, _, _ = ogcn.finetune_epoch(o64, f64, {"chr22": (ip, ix)}, oopt, "valid")
    assert float((pv.double() - pv64).abs().max()) <= 1e-4
    t = tgt.numpy()
    for c in range(nclass):
        if 0 < t[:, c].sum() < n:
            assert abs(roc_auc_score(t[:, c], pv[:, c].numpy()) - roc_auc_score(t[:, c], pv64[:, c].numpy())) <= 1e-4, c
            assert abs(average_precision_score(t[:, c], pv[:, c].numpy()) - average_precision_score(t[:, c], pv64[:, c].numpy())) <= 1e-4, c


@pytest.mark.parametrize("env", [{"CGCN_NO_FUSED": "1"}], ids=["unfused"])
def test_alternative_kernel_paths_keep_parity(env):
    """The library runs each layer either as the all-in-one fused kernel (the default at Hi-C degrees) or as three
    kernels (SpMM, row-panel contraction, gate kernel: d != 128, weighted graphs, the FFMA contractions, mean degree
    above 24).  CGCN_NO_FUSED, read once per process, forces the three kernels on graphs that would take the fused
    kernel: the model parity tests re-run in a subprocess under it."""
    import subprocess
    import sys
    e = dict(os.environ)
    e.update(env)
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-m", "gpu", "-q", "-x", "-k",
                        "fused_engine_matches_reference or module_api_matches_reference or extension_variants or dropout_training"],
                       capture_output=True, text=True, timeout=900, env=e, cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-1000:]


def test_dense_and_asymmetric_adjacency_with_adjacency_gradient():
    """scripts/visualize.py:30-45 hands the model a DENSE `adj` that requires grad and reads `|adj * adj.grad|`;
    :103-111 hands it re-normalised sparse tensors with masked entries (arbitrary values, asymmetric pattern).  Both run
    on the generic weighted-CSR path (cgcn_spmm with values, its transpose, cgcn_sddmm for d loss / d adj) and must
    match the reference model (oracle restatement, fp64 CPU) on outputs, parameter gradients and the adjacency
    gradient on the non-zero support."""
    from chromegcn_b200.chrome_models import ChromeGCN
    n, nclass = 300, 7
    gen = torch.Generator().manual_seed(8)
    dense = (torch.rand(n, n, generator=gen) < 0.03).float() * torch.rand(n, n, generator=gen)      # asymmetric, weighted
    dense = dense + torch.eye(n)
    dense = dense / dense.sum(1, keepdim=True)
    x = torch.randn(n, 128, generator=gen)
    tgt = (torch.rand(n, nclass, generator=gen) < 0.2).double()
    torch.manual_seed(3)
    om = ogcn.stress_init_(ogcn.ChromeGCNOracle(128, 128, nclass, 0.0, True, 2)).double().train()
    m = ChromeGCN(128, 128, nclass, 0.0, True, 2)
    m.load_state_dict({k: v.float() for k, v in om.state_dict().items()})
    m = m.to(_dev()).train()
    # ---- dense adj with requires_grad
    a_ref = dense.double().clone().requires_grad_(True)
    _, out_ref, gates_ref, _ = om(x.double(), a_ref, None)
    torch.sigmoid(out_ref).backward(gradient=tgt)
    a = dense.to(_dev()).clone().requires_grad_(True)
    _, out, gates, _ = m(x.to(_dev()), a, None)
    torch.sigmoid(out).backward(gradient=tgt.float().to(_dev()))
    assert ogcn.max_rel(out.cpu(), out_ref) <= 1e-5
    assert ogcn.max_rel(gates[0].cpu(), gates_ref[0]) <= 1e-5 and ogcn.max_rel(gates[1].cpu(), gates_ref[1]) <= 1e-5
    support = dense != 0
    assert ogcn.max_rel(a.grad.cpu()[support], a_ref.grad[support]) <= 2e-5
    assert float(a.grad.cpu()[~support].abs().max()) == 0.0              # gradient on the support only (|adj * adj.grad|)
    sal = (a * a.grad).abs().cpu()
    assert ogcn.max_rel(sal, (a_ref * a_ref.grad).abs().detach()) <= 2e-5
    for k, p in om.named_parameters():
        assert ogcn.max_rel(dict(m.named_parameters())[k].grad.cpu(), p.grad) <= 5e-5, k
    # ---- asymmetric re-normalised sparse tensor, forward only (eval mode)
    om.eval()
    m.eval()
    idx = torch.nonzero(dense).t()
    sp = torch.sparse_coo_tensor(idx, dense[idx[0], idx[1]], dense.shape)
    with torch.no_grad():
        _, o_ref, _, _ = om(x.double(), sp.double(), None)
        _, o, _, _ = m(x.to(_dev()), sp.to(_dev()), None)
    assert ogcn.max_rel(o.cpu(), o_ref) <= 1e-5
