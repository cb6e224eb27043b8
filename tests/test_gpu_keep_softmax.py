"""Backward pass 2 reading the softmax the symmetric attention stored (default) against recomputing it
(DL_F_NO_KEEPA).

With a symmetric pass-2 plan, the forward writes a[t, k] of every primary entry t into the plan's coefficient
buffer and phase A of pass 2 reads it back instead of rebuilding it from the dots, exponentials and softmax
sum.  Checked here, on the golden fixtures, a ~10^6-node power-law graph at (8, 16) and (5, 32) and the real
Pubmed graph, for both paths:
  * the forward outputs (kstar, w, s, H, prob, loss) of PartitionedLinkStep are bitwise equal;
  * the stored a is the forward's softmax: a[t, kstar] is the oracle's w bit for bit, kstar is its first
    maximum, and every factor is within a few ulps of a float64 softmax of the same dots (the oracle exposes
    w = a[kstar], not the other factors);
  * dZ is within 1e-5 of its max-abs (5e-5 of the row's max-abs on rows of degree >= 512) of the oracle and
    of the NO_KEEPA path.  The paths differ only in the backward using the forward's IEEE a instead of an
    8-lane butterfly sum with an approximate reciprocal.
"""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR, GRAPH_FIXTURES, load_golden

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL, HUB_TOL, HUB_DEG = 1e-5, 5e-5, 512


def t(x, dtype=None):
    return torch.as_tensor(np.ascontiguousarray(x), device=DEV, dtype=dtype)


def relerr(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)) if b.size else 0.0


def _fixture_case(name):
    g = load_golden(name)
    return (g["src"], g["dst"], int(g["N"]), g["Z"], float(g["beta"]), float(g["T"]))


def _power_law_case(N, E, K, d):
    sys.path.insert(0, ROOT)
    import bench
    src, dst = bench.gen_edges(N, E, 0, "cpu")
    rng = np.random.default_rng(K * 100 + d)
    Z = rng.standard_normal((N, K, d), dtype=np.float32) * np.float32(d ** -0.25)
    return src.numpy(), dst.numpy(), N, Z, 0.5, 1.0


def _pubmed_case(K, d):
    gd = dict(np.load(os.path.join(GOLDEN_DIR, "pubmed_graph.npz")))
    N = int(gd["N"])
    rng = np.random.default_rng(d)
    Z = rng.standard_normal((N, K, d), dtype=np.float32) * np.float32(d ** -0.25)
    return gd["src"].astype(np.int64), gd["dst"].astype(np.int64), N, Z, 0.6, 1.0


NONEMPTY_FIXTURES = [n for n in GRAPH_FIXTURES if np.load(os.path.join(GOLDEN_DIR, n + ".npz"))["src"].size]
CASES = {**{name: (lambda n=name: _fixture_case(n)) for name in NONEMPTY_FIXTURES},
         "powerlaw_1M_K8_d16": lambda: _power_law_case(1_000_000, 5_000_000, 8, 16),
         "powerlaw_1M_K5_d32": lambda: _power_law_case(1_000_000, 5_000_000, 5, 32),
         "pubmed_K8_d8": lambda: _pubmed_case(8, 8)}


@pytest.fixture(scope="module")
def dl():
    import disenlink_b200.ops as ops
    from disenlink_b200 import _lib
    from disenlink_b200.graph import Graph
    _lib.lib()
    return ops, Graph, _lib


@pytest.fixture
def sym_everywhere(dl, monkeypatch):
    """The symmetric paths on graphs of every size (by default only from 2^20 entries on)."""
    _, Graph, _ = dl
    monkeypatch.setattr(Graph, "SYM_MIN_NNZ", 0)


def _hub_rows_ok(dZ, ref, deg):
    hub = deg >= HUB_DEG
    n = deg.size
    err = np.abs(dZ.reshape(n, -1).astype(np.float64) - ref.reshape(n, -1)).max(1)
    scale = np.maximum(np.abs(ref.reshape(n, -1)).max(1), 1e-30)
    assert np.all(err[hub] <= HUB_TOL * scale[hub])


def _check_stored_a(a, kstar_u, w_u, Z, rows_u, cols_u, T):
    """a [nu, K] as stored by the forward, kstar / w of the same primary entries."""
    nu, K = a.shape
    ar = torch.arange(nu, device=DEV)
    assert torch.equal(a[ar, kstar_u].view(torch.int32), w_u.view(torch.int32))
    # first maximum (no NaN here: Z is finite)
    assert torch.equal(torch.argmax(a, dim=1), kstar_u)
    Zt = t(Z)
    step = 1 << 20
    for lo in range(0, nu, step):
        hi = min(nu, lo + step)
        q = (Zt[rows_u[lo:hi]].double() * Zt[cols_u[lo:hi]].double()).sum(-1) / T
        ref = torch.softmax(q, dim=1)
        assert float((a[lo:hi].double() - ref).abs().max()) <= 1e-5


def _run_step(ops, _lib, src, dst, N, Z, beta, T, keepa):
    from disenlink_b200.partition import PartitionedLinkStep
    K, d = int(Z.shape[1]), int(Z.shape[2])
    rng = np.random.default_rng(7)
    E = src.size
    assert E > 0
    P = min(1 << 18, max(6, E))
    pu = src[rng.integers(0, E, P)]
    pv = rng.integers(0, N, P)
    order = np.argsort(pu, kind="stable")
    lab = (rng.random(P) < 0.2).astype(np.float32)
    wts = np.full(P, 1.0 / P, dtype=np.float32)
    step = PartitionedLinkStep(t(src), t(dst), N, t(pu[order]), t(pv[order]), t(lab), t(wts), K, d, beta, T,
                               world=1, rank=0, device=DEV)
    if not keepa:
        step.graph.flags = step.graph.flags | _lib.DL_F_NO_KEEPA
    step.Z_own.copy_(t(Z))
    step.forward()
    plan = step.plan_bwd
    a = None
    if plan["mode"] == "sym":
        assert plan["a_valid"] == keepa
        nu = plan["upper"].nnz
        if keepa:
            a = plan["coef"][:nu * K].view(nu, K).clone()
    else:
        assert not plan["a_valid"]
    step.loss_and_grad_logit()
    step.backward()
    assert not plan["a_valid"]                     # pass 2 overwrote the softmax with coefficients
    n = step.n_own
    out = {"kstar": step.kstar[:step.graph.nnz].clone(), "w": step.w[:step.graph.nnz].clone(),
           "s": step.s[:n].clone(), "H": step.H[:n].clone(), "prob": step.prob[:P].clone(),
           "loss": step.loss.clone(), "dZ": step.dZ.clone()}
    return out, a, step


@pytest.mark.parametrize("case", list(CASES))
def test_step_forward_bitwise_and_stored_softmax(dl, oracle, sym_everywhere, case):
    ops, Graph, _lib = dl
    src, dst, N, Z, beta, T = CASES[case]()
    o1, a, step = _run_step(ops, _lib, src, dst, N, Z, beta, T, keepa=True)
    o0, _, _ = _run_step(ops, _lib, src, dst, N, Z, beta, T, keepa=False)
    for k in ("kstar", "w", "s", "H", "prob", "loss"):
        assert torch.equal(o1[k].reshape(-1).view(torch.uint8), o0[k].reshape(-1).view(torch.uint8)), k
    assert relerr(o1["dZ"].cpu().numpy(), o0["dZ"].cpu().numpy()) < TOL
    K, d = int(Z.shape[1]), int(Z.shape[2])
    sym = step.plan_bwd["mode"] == "sym"
    assert sym == bool(_lib.lib().dl_factor_bwd_edges_sym_supported(K, d))
    if sym:
        g = step.graph
        eidx = g.sym_view()[1].long()
        prim = eidx >= 0
        rows = torch.repeat_interleave(torch.arange(g.N, device=DEV), g.rowptr[1:] - g.rowptr[:-1])
        pos = eidx[prim]
        rows_u = torch.empty_like(pos)
        cols_u = torch.empty_like(pos)
        kstar_u = torch.empty_like(pos)
        w_u = torch.empty(pos.numel(), dtype=torch.float32, device=DEV)
        rows_u[pos], cols_u[pos] = rows[prim], g.col[prim].long()
        kstar_u[pos], w_u[pos] = o1["kstar"][prim].long(), o1["w"][prim]
        assert pos.numel() == a.shape[0]
        rowptr, col = oracle.csr_from_edges(src, dst, N)
        o_k, o_w, _ = oracle.edge_attn_fwd(rowptr, col, Z, T)
        assert np.array_equal(o1["kstar"].cpu().numpy(), o_k)
        assert np.array_equal(o1["w"].cpu().numpy().view(np.uint32), o_w.view(np.uint32))
        _check_stored_a(a, kstar_u, w_u, Z, rows_u, cols_u, T)


@pytest.mark.parametrize("case", list(CASES))
def test_factor_backward_vs_oracle(dl, oracle, sym_everywhere, case):
    ops, Graph, _lib = dl
    oracle.set_num_threads(os.cpu_count() or 1)
    src, dst, N, Z, beta, T = CASES[case]()
    K, d = int(Z.shape[1]), int(Z.shape[2])
    rng = np.random.default_rng(3)
    G = rng.standard_normal(Z.shape, dtype=np.float32)
    dZ0 = rng.standard_normal(Z.shape, dtype=np.float32)
    rowptr, col = oracle.csr_from_edges(src, dst, N)
    o_k, o_w, o_s = oracle.edge_attn_fwd(rowptr, col, Z, T)
    o_dZ = oracle.factor_bwd(rowptr, col, Z, G, o_k, o_w, o_s, beta, T, dZ_init=dZ0)
    deg = np.diff(rowptr)
    got = {}
    for keepa in (True, False):
        g = Graph.from_edges(t(src), t(dst), N)
        if not keepa:
            g.flags = g.flags | _lib.DL_F_NO_KEEPA
        plan = ops.bwd_plan(g, K, d)
        kstar, w, s = ops.edge_attn_fwd(g, t(Z), T, plan=plan)
        assert plan["a_valid"] == (keepa and plan["mode"] == "sym")
        dZ = t(dZ0).clone()
        r = torch.empty(N, K, dtype=torch.float32, device=DEV)
        ops.factor_bwd_gather(g, t(Z), t(G), kstar, w, s, beta, dZ, r, plan=plan)
        ops.factor_bwd_edges(g, t(Z), t(G), kstar, w, s, r, beta, T, dZ, plan=plan)
        assert not plan["a_valid"]
        got[keepa] = dZ.cpu().numpy()
        assert relerr(got[keepa], o_dZ) < TOL
        _hub_rows_ok(got[keepa], o_dZ, deg)
    assert relerr(got[True], got[False]) < TOL
    _hub_rows_ok(got[True], got[False].astype(np.float64), deg)
