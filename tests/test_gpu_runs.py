"""Batched independent runs on the GPU: the segmented AUC and loss kernels against their one-list forms, one
union step against R separate steps from identical Z, and examples/train_link.py's run_batched against run()."""
import argparse
import math
import os
import sys

import numpy as np
import pytest
import torch

from conftest import load_golden
from disenlink_b200 import ops
from disenlink_b200.model import Disentangle
from disenlink_b200.runs import RunSet

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples"))


def _ptr(sizes):
    return torch.tensor(np.concatenate([[0], np.cumsum(sizes)]), dtype=torch.int64, device=DEV)


def _check_auc_segments(score, labels, sizes, sklearn_check=True):
    seg = _ptr(sizes)
    out = ops.roc_auc_segments(score, labels, seg).cpu()
    assert out.shape == (len(sizes), 5)
    bounds = seg.tolist()
    for r in range(len(sizes)):
        lo, hi = bounds[r], bounds[r + 1]
        ref = ops.roc_auc_stats(score[lo:hi], labels[lo:hi]).cpu()
        assert np.array_equal(out[r].numpy().view(np.uint64), ref.numpy().view(np.uint64)), (r, out[r], ref)
        if sklearn_check and hi - lo > 0 and 0 < ref[1] and 0 < ref[2] and ref[3] == 0:
            from sklearn.metrics import roc_auc_score
            want = roc_auc_score(labels[lo:hi].cpu().numpy(), score[lo:hi].cpu().numpy())
            assert abs(out[r, 0].item() - want) <= 1e-12
    return out


def test_auc_segments_single_segment():
    g = torch.Generator(device=DEV).manual_seed(0)
    s = torch.rand(5000, device=DEV, generator=g)
    y = (torch.rand(5000, device=DEV, generator=g) < 0.3).float()
    _check_auc_segments(s, y, [5000])


def test_auc_segments_degenerate_segments():
    g = torch.Generator(device=DEV).manual_seed(1)
    sizes = [0, 1, 50, 40, 0, 30, 60, 1, 0]
    P = sum(sizes)
    s = torch.rand(P, device=DEV, generator=g)
    y = (torch.rand(P, device=DEV, generator=g) < 0.5).float()
    b = np.concatenate([[0], np.cumsum(sizes)])
    y[b[3]:b[4]] = 1.0                                     # one class only: positives
    y[b[5]:b[6]] = 0.0                                     # one class only: negatives
    s[b[6] + 7] = float("nan")                             # a NaN score
    out = _check_auc_segments(s, y, sizes)
    auc = out[:, 0].tolist()
    for r in (0, 1, 3, 4, 5, 6, 7, 8):
        assert math.isnan(auc[r]), r
    assert not math.isnan(auc[2])


def test_auc_segments_ties_across_boundaries():
    """Every segment holds the same few score values (ties inside and across segments), labels differ."""
    g = torch.Generator(device=DEV).manual_seed(2)
    sizes = [17, 33, 1, 64, 9, 128]
    P = sum(sizes)
    s = torch.randint(0, 4, (P,), device=DEV, generator=g).float() * 0.25
    s[:5] = -0.0                                            # -0.0 ties with +0.0
    y = (torch.rand(P, device=DEV, generator=g) < 0.5).float()
    _check_auc_segments(s, y, sizes)
    b = np.concatenate([[0], np.cumsum(sizes)])             # constant scores: the boundary is the only thing
    s2 = torch.full((P,), 0.5, device=DEV)                  # that keeps two segments' ties apart
    y2 = torch.zeros(P, device=DEV)
    for r in range(len(sizes)):
        y2[b[r]:b[r] + sizes[r] // 2] = 1.0
    out = _check_auc_segments(s2, y2, sizes)
    for r in range(len(sizes)):
        if sizes[r] > 1:
            assert out[r, 0].item() == 0.5


def test_auc_segments_many_tiny_segments():
    g = torch.Generator(device=DEV).manual_seed(3)
    sizes = torch.randint(0, 6, (1000,), generator=torch.Generator().manual_seed(3)).tolist()
    P = sum(sizes)
    s = torch.randint(0, 8, (P,), device=DEV, generator=g).float()
    y = (torch.rand(P, device=DEV, generator=g) < 0.5).float()
    _check_auc_segments(s, y, sizes, sklearn_check=False)


def test_auc_segments_large():
    g = torch.Generator(device=DEV).manual_seed(4)
    P, R = 10**7, 10
    s = torch.rand(P, device=DEV, generator=g)
    s = torch.round(s * 2**16) / 2**16                     # many ties
    y = (torch.rand(P, device=DEV, generator=g) < 0.2).float()
    sizes = [P // R] * R
    sizes[-1] += P - sum(sizes)
    _check_auc_segments(s, y, sizes)


def test_link_bce_segments():
    g = torch.Generator(device=DEV).manual_seed(5)
    sizes = [0, 1, 1000, 7, 0, 50000, 3]
    P = sum(sizes)
    prob = torch.rand(P, device=DEV, generator=g)
    prob[::97] = 0.0                                         # saturated scores: the -100 clamps
    prob[5::101] = 1.0
    y = (torch.rand(P, device=DEV, generator=g) < 0.5).float()
    w = torch.rand(P, device=DEV, generator=g) / 1000
    seg = _ptr(sizes)
    b = seg.tolist()
    for weights in (w, None):
        got = ops.link_bce_segments(prob, y, weights, seg).cpu()
        again = ops.link_bce_segments(prob, y, weights, seg).cpu()
        assert torch.equal(got, again)
        for r in range(len(sizes)):
            lo, hi = b[r], b[r + 1]
            if hi == lo:
                assert got[r].item() == 0.0
                continue
            ref, _ = ops.link_bce(prob[lo:hi], y[lo:hi], None if weights is None else weights[lo:hi], want_grad=False)
            ref = ref.item()
            assert abs(got[r].item() - ref) <= 2.0**-24 * abs(ref), (r, got[r].item(), ref)


# ---- one union step against R separate steps -------------------------------------------------------------
def _cora():
    g = load_golden("cora_K3_d32")
    ei = torch.stack([torch.as_tensor(g["src"]), torch.as_tensor(g["dst"])]).to(DEV)
    return ei, int(g["N"]), int(g["K"]), int(g["d"]), float(g["beta"]), float(g["T"])


def _rel(a, b):
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-30)


@pytest.mark.parametrize("directed", [False, True])
def test_union_step_equals_separate_steps(directed):
    ei, N, K, d, beta, T = _cora()
    seeds = [0, 1, 2]
    union = RunSet(ei, N, seeds, m=2, directed=directed)
    R = len(seeds)
    gz = torch.Generator(device=DEV).manual_seed(9)
    Z = (torch.randn(R * N, K, d, device=DEV, generator=gz) * 0.3).contiguous()
    kU, wU, sU = ops.edge_attn_fwd(union.graph, Z, T)
    ZU = Z.clone().requires_grad_(True)
    lossU, probU, HU = ops.link_bce_loss(ZU, union.graph, union.train, union.train_labels, union.train_weights, beta, T)
    lossU.backward()
    rp = union.graph.rowptr.tolist()
    tp = union.train_ptr.tolist()
    for r, seed in enumerate(seeds):
        one = RunSet(ei, N, [seed], m=2, directed=directed)
        Zr = Z[r * N:(r + 1) * N].contiguous()
        k1, w1, s1 = ops.edge_attn_fwd(one.graph, Zr, T)
        e0, e1 = rp[r * N], rp[(r + 1) * N]
        assert e1 - e0 == one.graph.nnz
        assert torch.equal(union.graph.col[e0:e1] - r * N, one.graph.col)
        assert torch.equal(kU[e0:e1], k1)
        assert torch.equal(wU[e0:e1].view(torch.int32), w1.view(torch.int32))
        assert _rel(sU[r * N:(r + 1) * N], s1) <= 1e-6
        Z1 = Zr.clone().requires_grad_(True)
        loss1, prob1, H1 = ops.link_bce_loss(Z1, one.graph, one.train, one.train_labels, one.train_weights, beta, T)
        loss1.backward()
        assert torch.equal(union.train_labels[tp[r]:tp[r + 1]], one.train_labels)
        assert _rel(HU[r * N:(r + 1) * N], H1) <= 1e-6
        assert _rel(probU[tp[r]:tp[r + 1]], prob1) <= 1e-6
        assert _rel(ZU.grad[r * N:(r + 1) * N], Z1.grad) <= 1e-5
        seg_loss = ops.link_bce_segments(probU, union.train_labels, union.train_weights, union.train_ptr)
        assert abs(seg_loss[r].item() - loss1.item()) <= 1e-6 * abs(loss1.item())


def test_runset_refuses_int32_overflow():
    ei, N, *_ = _cora()
    with pytest.raises(ValueError):
        RunSet(ei, 2**30, [0, 1], m=1)


# ---- the example's loop ----------------------------------------------------------------------------------
def _args(**kw):
    a = dict(nfactor=4, nhidden=64, nembed=16, beta=0.7, temperature=1, m=2, lr=0.01, epochs=20, seed=3,
             log_every=1000, standardize=True, run=3)
    a.update(kw)
    return argparse.Namespace(**a)


def test_run_batched_matches_single_runs():
    import train_link
    args = _args()
    x, edge_index, _ = train_link.synthetic(n=2000, seed=0)
    seeds = [args.seed + r for r in range(args.run)]
    model = train_link.batched_model(args, x.shape[1], seeds)
    for r, seed in enumerate(seeds):                      # run()'s model after torch.manual_seed(seed)
        torch.manual_seed(seed)
        ref = Disentangle(x.shape[1], args.nhidden, args.nembed, nfactor=args.nfactor, beta=args.beta,
                          t=args.temperature).state_dict()
        got = model.run_state_dict(r)
        assert all(torch.equal(got[k], ref[k]) for k in ref)
    out = train_link.run_batched(args, x, edge_index, torch.device(DEV), log=lambda *_: None)
    drift = 0.0
    for r, seed in enumerate(seeds):
        torch.manual_seed(seed)
        single = train_link.run(argparse.Namespace(**{**vars(args), "seed": seed}), x, edge_index, torch.device(DEV),
                                log=lambda *_: None)
        b = out["runs"][r]
        assert b["seed"] == seed
        (l0, a0), (l1, a1) = b["history"][0], single["history"][0]
        assert abs(l0 - l1) <= 1e-5 * abs(l1) and abs(a0 - a1) <= 1e-5, (r, b["history"][0], single["history"][0])
        losses = [l for l, _ in b["history"]]
        assert all(math.isfinite(l) for l in losses) and losses[-1] < losses[0]
        d = max(abs(b["best_val_auc"] - single["best_val_auc"]), abs(b["test_auc"] - single["test_auc"]))
        drift = max(drift, d)
        assert d <= 0.02, (r, b["best_val_auc"], single["best_val_auc"], b["test_auc"], single["test_auc"])
    print(f"run_batched vs run(): max |best val / test AUC difference| = {drift:.2e}")
    assert abs(out["test_auc_mean"] - np.mean([b["test_auc"] for b in out["runs"]])) < 1e-12


def test_run_batched_is_deterministic():
    import train_link
    args = _args(epochs=8, seed=0)
    x, edge_index, _ = train_link.synthetic(n=2000, seed=0)
    a = train_link.run_batched(args, x, edge_index, torch.device(DEV), log=lambda *_: None)
    b = train_link.run_batched(args, x, edge_index, torch.device(DEV), log=lambda *_: None)
    assert [r["history"] for r in a["runs"]] == [r["history"] for r in b["runs"]]
    assert [r["test_auc"] for r in a["runs"]] == [r["test_auc"] for r in b["runs"]]


def test_segment_wrappers_check_their_inputs():
    prob = torch.rand(10, device=DEV)
    lab = torch.zeros(10, device=DEV)
    seg = _ptr([4, 6])
    with pytest.raises(TypeError):
        ops.link_bce_segments(prob.double(), lab, None, seg)
    with pytest.raises(ValueError):
        ops.link_bce_segments(prob, lab[:9], None, seg)
    with pytest.raises(ValueError):
        ops.link_bce_segments(prob, lab, torch.ones(10), seg)          # weights on the host
    with pytest.raises(ValueError):
        ops.roc_auc_segments(prob, lab[:9], seg)
    with pytest.raises(ValueError):
        ops.roc_auc_segments(prob, lab, seg.int())
