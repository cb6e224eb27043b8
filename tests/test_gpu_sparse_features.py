"""The first layer from sparse features (features.SparseFeatures, ops.feature_projection, csrc/feat_proj.cu): the
kernels against float64, bitwise determinism and run independence inside a union, the modules against their dense
path, the captured epoch against the eager one, and training through examples/train_link.py --sparse-features."""
import argparse
import copy
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden
from disenlink_b200 import data, ops
from disenlink_b200.capture import CapturedEpoch
from disenlink_b200.features import SparseFeatures
from disenlink_b200.model import Disentangle
from disenlink_b200.runs import DisentangleRuns, RunSet

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "examples"))
from sparse_features_bench import zipf_bag_of_words  # noqa: E402

N_CORA, F_CORA = 2708, 1433
CORA_RAW = os.path.join(ROOT, "baseline", "_ref", "data", "cora", "raw")


def _bits(t):
    return t.detach().contiguous().view(torch.int32)


def _features(case, seed=0):
    """-> dense x [N, F] (CPU) of one input case."""
    g = torch.Generator().manual_seed(seed)
    if case == "zipf":
        return zipf_bag_of_words(N_CORA, F_CORA, 0.0127, seed=seed)
    if case == "n1":
        return zipf_bag_of_words(1, F_CORA, 0.05, seed=seed)
    if case == "zero_rows_cols":                     # every third row and column empty
        x = zipf_bag_of_words(N_CORA, F_CORA, 0.0127, seed=seed)
        x[::3] = 0
        x[:, ::3] = 0
        return x
    if case == "dense_column":                       # column 7 in every row: 11 chunks of the weight gradient
        x = zipf_bag_of_words(N_CORA, F_CORA, 0.0127, seed=seed)
        x[:, 7] = 1.0
        return x
    if case == "values":                             # non-binary, signed, some rows much longer
        x = zipf_bag_of_words(N_CORA, F_CORA, 0.0127, seed=seed) * torch.randn(N_CORA, F_CORA, generator=g)
        x[:40, :400] = torch.randn(40, 400, generator=g)
        return x
    if case == "cora":
        x, _, _ = data.read_planetoid(CORA_RAW, "cora")
        return x
    raise KeyError(case)


def _blocks(J):
    return {1: 1, 111: 3, 1536: 3, 25600: 100}[J]


def _run_layer(feats, Wt, b, G, relu, blocks):
    """-> (A [N, J], dWt, db) of the kernels, G given as the contiguous [blocks, N, nh] the second layer returns."""
    Wt = Wt.detach().clone().requires_grad_()
    b = b.detach().clone().requires_grad_()
    out = ops.feature_projection(feats, Wt, b, relu=relu, blocks=blocks)
    assert out.shape == (blocks, feats.N, Wt.shape[1] // blocks)
    out.backward(G)
    return out.detach().transpose(0, 1).reshape(feats.N, -1), Wt.grad, b.grad


def _inputs(N, F, J, blocks, seed=1):
    g = torch.Generator(device=DEV).manual_seed(seed)
    Wt = torch.randn(F, J, device=DEV, generator=g) / 8
    b = 0.1 * torch.randn(J, device=DEV, generator=g)
    G = torch.randn(blocks, N, J // blocks, device=DEV, generator=g)
    return Wt, b, G


U = 2.0 ** -24


@pytest.mark.parametrize("case", ["zipf", "n1", "zero_rows_cols", "dense_column", "values",
                                  pytest.param("cora", marks=pytest.mark.skipif(
                                      not os.path.exists(CORA_RAW), reason="baseline/_ref not staged"))])
@pytest.mark.parametrize("J", [1, 111, 1536, 25600])
@pytest.mark.parametrize("relu", [True, False])
def test_kernels_against_float64(case, J, relu):
    x = _features(case).to(DEV)
    feats = SparseFeatures.from_dense(x)
    N, F = x.shape
    blocks = _blocks(J)
    Wt, b, G = _inputs(N, F, J, blocks)
    x64, W64, b64 = x.double(), Wt.double(), b.double()
    pre = x64 @ W64 + b64                                                    # float64 pre-activation
    row_len = (x != 0).sum(1, keepdim=True).double()
    bound_a = (row_len + 1) * U * (x64.abs() @ W64.abs() + b64.abs())
    ambiguous = (pre.abs() <= bound_a) if relu else torch.zeros_like(pre, dtype=torch.bool)
    # the cotangent is zeroed where the ReLU mask is ambiguous, so neither dWt nor db depends on it
    Gm = G.transpose(0, 1).reshape(N, J).clone()
    Gm[ambiguous] = 0
    G = Gm.view(N, blocks, J // blocks).transpose(0, 1).contiguous()
    A, dWt, db = _run_layer(feats, Wt, b, G, relu, blocks)
    ref_a = pre.clamp(min=0) if relu else pre
    ok = (A.double() - ref_a).abs() <= bound_a
    assert bool((ok | ambiguous).all()), f"A: {int((~ok & ~ambiguous).sum())} elements outside the bound"
    Gp = Gm.double() * (pre > 0) if relu else Gm.double()
    col_len = (x != 0).sum(0).double().view(F, 1)
    bound_w = (col_len + 1) * U * (x64.abs().t() @ Gp.abs())
    assert bool(((dWt.double() - x64.t() @ Gp).abs() <= bound_w).all())
    bound_b = (N + 1) * U * Gp.abs().sum(0)
    assert bool(((db.double() - Gp.sum(0)).abs() <= bound_b).all())
    print(f"{case} J={J} relu={relu}: {int(ambiguous.sum())} ReLU-mask entries within the bound of zero excluded")


@pytest.mark.parametrize("relu", [True, False])
def test_two_calls_are_bitwise_equal(relu):
    x = _features("dense_column").to(DEV)
    feats = SparseFeatures.from_dense(x)
    Wt, b, G = _inputs(*x.shape, 1536, 3)
    first = _run_layer(feats, Wt, b, G, relu, 3)
    second = _run_layer(feats, Wt, b, G, relu, 3)
    for p, q in zip(first, second):
        assert torch.equal(_bits(p), _bits(q))


def test_union_blocks_equal_the_runs_alone():
    """A union of R = 3 runs (K = 3, nhid = 64: J = 576): block r of A, dWt and db is what run r's Wt gives alone."""
    x = _features("dense_column").to(DEV)
    feats = SparseFeatures.from_dense(x)
    N, F = x.shape
    R, K, nh = 3, 3, 64
    runs = [_inputs(N, F, K * nh, K, seed=10 + r) for r in range(R)]
    Wt = torch.cat([w for w, _, _ in runs], dim=1)
    b = torch.cat([bb for _, bb, _ in runs])
    G = torch.cat([g for _, _, g in runs], dim=0)                    # [R*K, N, nh]
    A, dWt, db = _run_layer(feats, Wt, b, G, True, R * K)
    J = K * nh
    for r, (w, bb, g) in enumerate(runs):
        a_r, dw_r, db_r = _run_layer(feats, w, bb, g, True, K)
        assert torch.equal(_bits(A[:, r * J:(r + 1) * J]), _bits(a_r))
        assert torch.equal(_bits(dWt[:, r * J:(r + 1) * J]), _bits(dw_r))
        assert torch.equal(_bits(db[r * J:(r + 1) * J]), _bits(db_r))


def _rel(a, b):
    return float((a - b).abs().max()) / max(float(b.abs().max()), 1e-30)


@pytest.mark.parametrize("kind", ["factor2", "nhid1", "runs3"])
def test_module_against_dense_x(kind):
    x = _features("zipf").to(DEV)
    feats = SparseFeatures.from_dense(x)
    torch.manual_seed(0)
    if kind == "runs3":
        model = DisentangleRuns(F_CORA, 64, 16, 4, 0.7, runs=3).to(DEV)
    else:
        model = Disentangle(F_CORA, 1 if kind == "nhid1" else 64, 16, nfactor=4, beta=0.7).to(DEV)
    keys = list(model.state_dict().keys())
    out = {}
    for name, xin in (("dense", x), ("sparse", feats)):
        model.zero_grad(set_to_none=True)
        Z = model.project(xin)
        C = torch.randn(Z.shape, device=DEV, generator=torch.Generator(device=DEV).manual_seed(3))
        Z.backward(C)
        out[name] = (Z.detach(), [p.grad.clone() for p in model.parameters()])
    assert _rel(out["sparse"][0], out["dense"][0]) <= 1e-5
    for gs, gd in zip(out["sparse"][1], out["dense"][1]):
        assert _rel(gs, gd) <= 1e-5
    assert list(model.state_dict().keys()) == keys
    if kind != "runs3":                                              # forward takes the handle too
        g = load_golden("cora_K3_d32")
        ei = torch.stack([torch.as_tensor(g["src"]), torch.as_tensor(g["dst"])]).to(DEV)
        H, scorer = model(feats, ei)
        assert H.shape == (N_CORA, 4 * 16) and torch.isfinite(H).all()


@pytest.mark.parametrize("R", [1, 3])
def test_replay_equals_eager(R):
    g = load_golden("cora_K3_d32")
    ei = torch.stack([torch.as_tensor(g["src"]), torch.as_tensor(g["dst"])]).to(DEV)
    beta, T = float(g["beta"]), float(g["T"])
    runs = RunSet(ei, N_CORA, list(range(R)), m=2)
    feats = SparseFeatures.from_dense(_features("zipf").to(DEV))
    torch.manual_seed(0)
    base = (Disentangle(F_CORA, 64, 32, nfactor=3, beta=0.7) if R == 1 else
            DisentangleRuns(F_CORA, 64, 32, 3, 0.7, runs=R)).to(DEV)
    ces = []
    for capture in (False, True):
        m = copy.deepcopy(base)
        opt = torch.optim.Adam(m.parameters(), lr=0.01, weight_decay=5e-4, capturable=True)
        ptrs = dict(train_ptr=runs.train_ptr, val_ptr=runs.val_ptr, test_ptr=runs.test_ptr) if R > 1 else {}
        ces.append(CapturedEpoch(m, opt, feats, runs.graph, runs.train, runs.train_labels, runs.train_weights,
                                 runs.val, runs.val_labels, runs.test, runs.test_labels, beta, T, chunk=5,
                                 capture=capture, **ptrs))
    eager, cap = ces
    rows_e, rows_c = eager.step(5), cap.step(5)
    assert np.array_equal(np.array(rows_e), np.array(rows_c), equal_nan=True)
    assert torch.equal(eager.records.view(torch.int64), cap.records.view(torch.int64))
    for pa, pb in zip(eager.model.parameters(), cap.model.parameters()):
        assert torch.equal(_bits(pa), _bits(pb))
        for k in eager.opt.state[pa]:
            assert torch.equal(_bits(eager.opt.state[pa][k].float()), _bits(cap.opt.state[pb][k].float())), k
    assert all(np.isfinite(r[0]) for r in rows_c)


def test_training_against_dense_x():
    """20 epochs of run() and run_batched(R = 3) with --sparse-features against dense x on the Cora graph and Zipf
    features: best validation and test AUC within 0.02."""
    import train_link
    g = load_golden("cora_K3_d32")
    ei = torch.stack([torch.as_tensor(g["src"]), torch.as_tensor(g["dst"])])
    x = _features("zipf")
    args = argparse.Namespace(nfactor=3, nhidden=64, nembed=16, beta=float(g["beta"]), temperature=1, m=2, lr=0.01,
                              epochs=20, seed=3, log_every=1000, standardize=False, run=1, capture=None)
    quiet = lambda *_: None                                                # noqa: E731
    drift = []
    for R in (1, 3):
        ref = []
        for sparse in (False, True):
            torch.manual_seed(args.seed)
            a = argparse.Namespace(**{**vars(args), "run": R, "sparse_features": sparse})
            out = (train_link.run if R == 1 else train_link.run_batched)(a, x, ei, torch.device(DEV), log=quiet)
            ref.append(out["runs"] if R > 1 else [out])
        for r, (d_, s_) in enumerate(zip(*ref)):
            assert len(s_["history"]) == len(d_["history"]) == 20
            d = (abs(d_["best_val_auc"] - s_["best_val_auc"]), abs(d_["test_auc"] - s_["test_auc"]))
            drift.append(d)
            assert max(d) <= 0.02, (R, r, d_["best_val_auc"], s_["best_val_auc"], d_["test_auc"], s_["test_auc"])
    print("sparse vs dense x (best val AUC, test AUC) differences: " +
          ", ".join(f"{a:.2e}/{b:.2e}" for a, b in drift))


def test_example_sparse_features_capture():
    cmd = [sys.executable, os.path.join(ROOT, "examples", "train_link.py"), "--dataset", "synthetic",
           "--sparse-features", "--capture", "10", "--epochs", "30", "--nhidden", "64"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    assert "test auc" in out.stdout
