"""The dense drop-in path against a float64 reference (pytest -m gpu for the GPU half).

When `adj` is a dense tensor, `Disentangle.forward` returns `link_pred` [N,N] from `k_allpairs_fwd` and its
gradient from `k_allpairs_bwd`; `Disentangle_layer.forward` returns `alpha0` from `k_dense_alpha0` and `att`
from `k_dense_att` (csrc/dense_compat.cu).  This file holds those four kernels to the per-element bounds the
sparse paths are held to in test_gpu_kernel_paths.py:

  * DenseRef64: the all-pairs decoder in float64 (one matmul per factor), its gradients from torch.autograd and
    the bounds A (every term in absolute value).  Pinned in the CPU suite to Ref64.decoder on all N^2 pairs and
    to dense_forward of model.py, so the bound is the sparse one restated, not a new one.
  * the checker's sensitivity: fp32 emulations of the kernels' summation orders pass, single faults (the
    transpose term of dS lost, the last d-chunk dropped, T not applied, the partial tile's last row unwritten,
    a factor's dZ from its neighbour's window) are rejected.
  * the four kernels over d across the chunk (64) and register-window (32) edges, K up to 32, N on and off the
    16-row tile, T in {1, 1.5, 2}; att bit-exact on hub rows, on a directed graph with clamped row sums, on an
    empty graph and on one node.
  * the module at the training script's shapes on the real edge columns of the golden fixtures, and the limits.
"""
from functools import lru_cache

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import load_golden
from test_directed import csr_of, directed_graph, routed_mask
from test_gpu_kernel_paths import Ref64, case_inputs, dense64, hard_graph, row_ratio, sum_ratio
from test_oracle_live_reference import _Leaf, adj_sym_of, dense_forward, dense_mask

DEV = "cuda:0"
SIG_ULPS = 4.0       # dl_sigmoid = 1 / (1 + dl_expf(-x)): the exp's few ulps, one add, one division

# Bars of the per-element checker in units of 2^-24 * A (sum_ratio) and, for the module's dL/dZ, of
# 2^-24 * max(|row|_inf, 1e-3 |dZ|_inf) (row_ratio).  Each is at most 4x the largest ratio observed over this
# file on an NVIDIA B200 (1000 W power limit); the observed value is in the comment.
C_DENSE = {
    "prob": 3.5,       # 0.893 (K = 1, d = 33, N = 1000, T = 2)
    "dZ": 16.0,        # 4.20  (K = 10, d = 64, N = 2708, dense dS)
    "dH": 15.0,        # 3.90  (K = 10, d = 64, N = 2708, dense dS)
    "alpha0": 50.0,    # 12.7  (K = 1, d = 256, N = 1000)
    "H": 9.5,          # 2.48  (Cora, K = 10, d = 64)
    "dZ_row": 52.0,    # 13.3  (chameleon, K = 5, d = 32)
}


def _f64(x, device=None):
    if isinstance(x, torch.Tensor):
        return x.detach().to(device=device, dtype=torch.float64)
    return torch.from_numpy(np.ascontiguousarray(x)).to(device=device, dtype=torch.float64)


def _np(x):
    return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


# ------------------------------------------------------------------------------------------
# float64 reference
# ------------------------------------------------------------------------------------------
class DenseRef64:
    """The all-pairs decoder of model.py:109-113 in float64: S[u,v] = sum_k exp(<Z_u,k, Z_v,k>/T) <H_u,k, H_v,k>,
    one [N,N] matmul per factor so that N ~ 5200 fits.  Z and H are the kernels' fp32 inputs, held exactly.

    Bounds (the construction of Ref64.decoder in matmul form; A_H = 0 unless given, H being an exact input):
      EA_k     = E_k (2 + 2 |Z_k||Z_k|^T / T)          the exp of a rounded dot, as _w_abs treats it
      HA_k     = |H_k||H_k|^T + A_H,k |H_k|^T + |H_k| A_H,k^T
      A_logit  = sum_k EA_k . HA_k
      D        = |dS| + |dS|^T                         covers the fp32 sum dSsym = dS + dS^T the kernel receives
      A_dH[:,k] = (D . EA_k) @ (|H_k| + A_H,k)
      A_dZ[:,k] = (D . EA_k . HA_k / T) @ |Z_k|
    The kernel returns prob = sigmoid(S), not S.  An error dS in the logit moves the probability by
    sigmoid'(S) dS = p (1 - p) dS to first order, and dl_sigmoid itself (exp, add, divide) adds a few ulps of p:
      A_prob   = p (1 - p) A_logit + SIG_ULPS p.
    alpha0[k] = E_k with A = E_k (2 + |Z_k||Z_k|^T / T): the dot's rounding carried through exp, plus the exp's."""

    def __init__(self, Z, H, T, A_H=None, device=None):
        self.Z, self.H = _f64(Z, device), _f64(H, device)
        self.A_H = None if A_H is None else _f64(A_H, device)
        self.T = float(T)
        self.N, self.K, self.d = self.Z.shape

    def _factor(self, k):
        z, h = self.Z[:, k], self.H[:, k]
        za, hd = z.abs(), h.abs()
        E = torch.exp(z @ z.t() / self.T)
        EA = E * (2.0 + 2.0 * (za @ za.t()) / self.T)
        HA = hd @ hd.t()
        if self.A_H is not None:
            ah = self.A_H[:, k]
            HA = HA + ah @ hd.t() + hd @ ah.t()
        return E, EA, HA

    def forward(self):
        logit = A = 0.0
        with torch.no_grad():
            for k in range(self.K):
                E, EA, HA = self._factor(k)
                h = self.H[:, k]
                logit = logit + E * (h @ h.t())
                A = A + EA * HA
            p = torch.sigmoid(logit)
        return dict(logit=logit, A_logit=A, prob=p, A_prob=p * (1.0 - p) * A + SIG_ULPS * p)

    def backward(self, dS):
        """dZ, dH (autograd of sum S . dS, factor by factor) and their A for a dense dS = dL/dlogit."""
        dS = _f64(dS, self.Z.device)
        D = dS.abs() + dS.abs().t()
        dZ, dH = torch.zeros_like(self.Z), torch.zeros_like(self.H)
        A_dZ, A_dH = torch.zeros_like(self.Z), torch.zeros_like(self.H)
        for k in range(self.K):
            z = self.Z[:, k].clone().requires_grad_(True)
            h = self.H[:, k].clone().requires_grad_(True)
            Sk = torch.exp(z @ z.t() / self.T) * (h @ h.t())
            dZ[:, k], dH[:, k] = torch.autograd.grad((Sk * dS).sum(), (z, h))
            with torch.no_grad():
                _, EA, HA = self._factor(k)
                W = D * EA
                hb = self.H[:, k].abs() + (0.0 if self.A_H is None else self.A_H[:, k])
                A_dH[:, k] = W @ hb
                A_dZ[:, k] = (W * HA / self.T) @ self.Z[:, k].abs()
        return dict(dZ=dZ, A_dZ=A_dZ, dH=dH, A_dH=A_dH)

    def alpha0(self, k):
        with torch.no_grad():
            z = self.Z[:, k]
            E = torch.exp(z @ z.t() / self.T)
            return E, E * (2.0 + (z.abs() @ z.abs().t()) / self.T)


RATIOS = {}


def check_ratio(tag, name, x, ref, A, bar=None):
    q = sum_ratio(_np(x), _np(ref), _np(A))
    RATIOS.setdefault(tag, {})[name] = q
    print(f"RATIO {tag} {name}={q:.3g}")
    bar = C_DENSE[name] if bar is None else bar
    assert np.isfinite(q) and q <= bar, f"{tag} {name}: error {q:.3g} x 2^-24 x A (bar {bar})"


def rejects(x, ref, A, name):
    return sum_ratio(_np(x), _np(ref), _np(A)) > C_DENSE[name]


# ------------------------------------------------------------------------------------------
# fp32 emulations of the kernels' summation orders (numpy, for the checker's sensitivity)
# ------------------------------------------------------------------------------------------
def _fma32(a, b, c):
    """fp32 fma: the product is exact in float64 and the sum is rounded once more (a double rounding through
    float64 differs from one rounding only on exact ties)."""
    return (a.astype(np.float64) * b.astype(np.float64) + c).astype(np.float32)


def emu_allpairs_fwd(Z, H, T, d_used=None):
    """k_allpairs_fwd: per factor two sequential fma chains over d, exp(q / T) * gh, factors summed in order."""
    N, K, d = Z.shape
    T32 = np.float32(T)
    S = None
    for k in range(K):
        q = np.zeros((N, N), np.float32)
        gh = np.zeros((N, N), np.float32)
        for x in range(d if d_used is None else d_used):
            q = _fma32(Z[:, None, k, x], Z[None, :, k, x], q)
            gh = _fma32(H[:, None, k, x], H[None, :, k, x], gh)
        tv = np.exp(q / T32) * gh
        S = tv if S is None else S + tv
    return np.float32(1) / (np.float32(1) + np.exp(-S))


def emu_allpairs_bwd(Z, H, dSsym, T):
    """k_allpairs_bwd: lane partials over the 32-wide windows, a butterfly across the lanes, then per live o
    (dSsym != 0) in order dH += ch H_o and dZ += cz Z_o with ch = dSsym exp(q / T), cz = ch gh / T."""
    N, K, d = Z.shape
    R = (d + 31) // 32
    pad = ((0, 0), (0, 0), (0, 32 * R - d))
    Zp = np.pad(Z, pad).reshape(N, K, R, 32)
    Hp = np.pad(H, pad).reshape(N, K, R, 32)
    dZ = np.zeros((N, K, R, 32), np.float32)
    dH = np.zeros((N, K, R, 32), np.float32)
    T32 = np.float32(T)
    for k in range(K):
        pq = np.zeros((N, N, 32), np.float32)
        ph = np.zeros((N, N, 32), np.float32)
        for t_ in range(R):
            pq = _fma32(Zp[:, None, k, t_], Zp[None, :, k, t_], pq)
            ph = _fma32(Hp[:, None, k, t_], Hp[None, :, k, t_], ph)
        for off in (16, 8, 4, 2, 1):
            lanes = np.arange(32) ^ off
            pq = pq + pq[:, :, lanes]
            ph = ph + ph[:, :, lanes]
        ch = dSsym * np.exp(pq[:, :, 0] / T32)
        cz = (ch * ph[:, :, 0]) / T32
        for o in range(N):
            live = dSsym[:, o] != 0
            dH[live, k] = _fma32(ch[live, o, None, None], Hp[o, k][None], dH[live, k])
            dZ[live, k] = _fma32(cz[live, o, None, None], Zp[o, k][None], dZ[live, k])
    return dZ.reshape(N, K, 32 * R)[:, :, :d], dH.reshape(N, K, 32 * R)[:, :, :d]


def kernel_inputs(n, K, d, seed):
    """Z and H scaled as case_inputs scales Z (q = O(1)); H is a second draw of the same law."""
    m = max(n, 50)
    Z = case_inputs(m, K, d, 0, seed)[0][:n]
    H = case_inputs(m, K, d, 0, seed + 1)[0][:n]
    return np.ascontiguousarray(Z), np.ascontiguousarray(H)


# ------------------------------------------------------------------------------------------
# CPU suite: DenseRef64 pinned to Ref64 and to dense_forward; the checker's sensitivity
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,K,d,T,with_AH", [(33, 3, 5, 1.5, False), (33, 3, 5, 1.5, True), (64, 2, 40, 2.0, True),
                                            (17, 1, 8, 1.0, False)])
def test_dense_ref64_is_ref64_decoder_on_all_pairs(n, K, d, T, with_AH):
    """On all N^2 pairs, DenseRef64's logit, dZ and dH and their A equal Ref64.decoder's to 1e-12 (with Ref64's H
    and, where given, its A_H; without A_H both drop the same terms)."""
    rng = np.random.default_rng(n * 100 + K * 10 + d)
    src, dst = rng.integers(0, n, 3 * n), rng.integers(0, n, 3 * n)
    rowptr, col = csr_of(np.concatenate([src, dst]), np.concatenate([dst, src]), n)
    Z = kernel_inputs(n, K, d, n + K + d)[0]
    kstar = rng.integers(0, K, col.size).astype(np.uint8)
    ref = Ref64(rowptr, col, Z, kstar, 0.6, T, chunk=29)
    if not with_AH:
        ref.A_H = torch.zeros_like(ref.A_H)
    dS = (rng.standard_normal((n, n)) * (rng.random((n, n)) < 0.4) / 16).astype(np.float32)
    u, v = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    sp = ref.decoder(u.reshape(-1), v.reshape(-1), dS.reshape(-1))
    dr = DenseRef64(Z, ref.H, T, A_H=ref.A_H if with_AH else None)
    fw, bw = dr.forward(), dr.backward(dS)
    pairs = {"logit": fw["logit"].reshape(-1), "A_logit": fw["A_logit"].reshape(-1), "dZp": bw["dZ"],
             "A_dZp": bw["A_dZ"], "dHp": bw["dH"], "A_dHp": bw["A_dH"]}
    for key, x in pairs.items():
        x, y = _np(x), sp[key]
        assert np.allclose(x, y, rtol=1e-12, atol=1e-12 * np.abs(y).max()), key
    assert torch.allclose(fw["prob"], torch.sigmoid(fw["logit"]))


@pytest.mark.parametrize("name", ["tiny_deadfactor_T2", "tiny_generic"])
def test_dense_ref64_is_the_restated_model(name):
    """link_pred and alpha0 of dense_forward (model.py restated, float64) from DenseRef64 with its H."""
    g = load_golden(name)
    n, K, T, beta = int(g["N"]), int(g["K"]), float(g["T"]), float(g["beta"])
    zs = [torch.from_numpy(g["Z"][:, k, :].astype(np.float64)) for k in range(K)]
    alpha0, _, H, link_pred = dense_forward(zs, adj_sym_of(g["src"], g["dst"], n).double(), beta, T)
    dr = DenseRef64(g["Z"], H.view(n, K, -1), T)
    assert torch.allclose(dr.forward()["prob"], link_pred, rtol=1e-12, atol=0)
    for k in range(K):
        assert torch.allclose(dr.alpha0(k)[0], alpha0[k], rtol=1e-12, atol=0)


@lru_cache(maxsize=None)
def _emu_case():
    """N = 33 (N mod 16 = 1: the last row is alone in its tile), d = 65 (a partial second chunk and a third
    register window), T = 2, a dS with 60 % exact zeros (the pairs the backward skips)."""
    n, K, d, T = 33, 3, 65, 2.0
    Z, H = kernel_inputs(n, K, d, 5)
    rng = np.random.default_rng(5)
    dS = (rng.standard_normal((n, n)) * (rng.random((n, n)) < 0.4) / 16).astype(np.float32)
    dSsym = dS + dS.T
    dr = DenseRef64(Z, H, T)
    return Z, H, T, dS, dSsym, dr.forward(), dr.backward(dS)


def test_checker_accepts_emulation_and_rejects_faults():
    Z, H, T, dS, dSsym, fw, bw = _emu_case()
    prob = emu_allpairs_fwd(Z, H, T)
    dZ, dH = emu_allpairs_bwd(Z, H, dSsym, T)
    check_ratio("fp32 emulation", "prob", prob, fw["prob"], fw["A_prob"])
    check_ratio("fp32 emulation", "dZ", dZ, bw["dZ"], bw["A_dZ"])
    check_ratio("fp32 emulation", "dH", dH, bw["dH"], bw["A_dH"])
    # dS where dSsym belongs: the transpose term is lost
    dZ_b, dH_b = emu_allpairs_bwd(Z, H, dS, T)
    assert rejects(dZ_b, bw["dZ"], bw["A_dZ"], "dZ") and rejects(dH_b, bw["dH"], bw["A_dH"], "dH")
    # the last (partial) d-chunk dropped: 64 of the 65 elements summed
    assert rejects(emu_allpairs_fwd(Z, H, T, d_used=64), fw["prob"], fw["A_prob"], "prob")
    # T not applied in the score
    assert rejects(emu_allpairs_fwd(Z, H, 1.0), fw["prob"], fw["A_prob"], "prob")
    # the row at the partial tile edge left at zero
    p_bad = prob.copy()
    p_bad[-1] = 0
    assert rejects(p_bad, fw["prob"], fw["A_prob"], "prob")
    # dZ of factor k >= 1 taken from factor k - 1's window
    for k in range(1, Z.shape[1]):
        dZ_bad = dZ.copy()
        dZ_bad[:, k] = dZ[:, k - 1]
        assert rejects(dZ_bad, bw["dZ"], bw["A_dZ"], "dZ")


# ------------------------------------------------------------------------------------------
# GPU: the four kernels against DenseRef64
# ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def L():
    from disenlink_b200 import _lib
    return _lib.lib()


def _t(x):
    return torch.as_tensor(np.ascontiguousarray(x), device=DEV)


def _stream():
    from disenlink_b200._lib import stream_of
    return stream_of(torch.device(DEV))


def _nan(*shape):
    return torch.full(shape, float("nan"), dtype=torch.float32, device=DEV)


def raw_fwd(L, Z, H, T):
    N, K, d = Z.shape
    prob = _nan(N, N)
    assert L.dl_allpairs_score_fwd(Z.data_ptr(), H.data_ptr(), N, K, d, float(T), prob.data_ptr(), _stream()) == 0
    return prob


def raw_bwd(L, Z, H, dSsym, T):
    N, K, d = Z.shape
    dZ, dH = _nan(N, K, d), _nan(N, K, d)
    assert L.dl_allpairs_score_bwd(Z.data_ptr(), H.data_ptr(), dSsym.data_ptr(), N, K, d, float(T), dZ.data_ptr(),
                                   dH.data_ptr(), _stream()) == 0
    return dZ, dH


def script_loss(link_pred, pos, neg, m):
    """main_disentangled.py:195: mean BCE over the positives + mean BCE over the negatives / m."""
    lp, ln = link_pred[pos].unsqueeze(0), link_pred[neg].unsqueeze(0)
    return F.binary_cross_entropy(lp, torch.ones_like(lp)) + F.binary_cross_entropy(ln, torch.zeros_like(ln)) / m


# (K, d, N, T): every d across the 64-chunk and 32-window edges, the script's (3,32), (5,32), (10,64), (5,64),
# K * d up to 32 x 256, N on and off the 16-row tile, the grid-stride wrap of alpha0 at N >= 1000
KERNEL_CASES = [
    (1, 1, 1, 1.0), (3, 7, 15, 1.5), (5, 31, 16, 2.0), (3, 32, 17, 1.0), (5, 32, 1000, 1.5), (3, 32, 2708, 1.0),
    (10, 64, 2708, 1.0), (5, 64, 2708, 2.0), (1, 33, 1000, 2.0), (3, 63, 17, 1.5), (10, 64, 1000, 1.5),
    (3, 65, 1000, 1.0), (2, 128, 1000, 2.0), (1, 200, 17, 1.5), (1, 256, 1000, 1.0), (32, 256, 17, 2.0),
    (32, 8, 1000, 1.5), (5, 32, 15, 1.0), (2, 256, 16, 1.5),
]


@pytest.mark.gpu
@pytest.mark.parametrize("K,d,N,T", KERNEL_CASES)
def test_allpairs_and_alpha0_kernels(L, K, d, N, T):
    from disenlink_b200 import ops
    tag = f"K={K} d={d} N={N} T={T}"
    Zn, Hn = kernel_inputs(N, K, d, 1000 * K + d + N)
    Z, H = _t(Zn), _t(Hn)
    dr = DenseRef64(Zn, Hn, T, device=DEV)
    fw = dr.forward()

    # forward: every element written, within the bound, bitwise equal run to run and to the autograd wrapper
    prob = raw_fwd(L, Z, H, T)
    check_ratio(tag, "prob", prob, fw["prob"], fw["A_prob"])
    assert torch.equal(prob, raw_fwd(L, Z, H, T))
    Zg, Hg = Z.clone().requires_grad_(True), H.clone().requires_grad_(True)
    link_pred = ops.allpairs_score(Zg, Hg, T)
    assert torch.equal(link_pred, prob)

    # backward with a dense random dS
    rng = np.random.default_rng(N + K + d)
    dS = _t((rng.standard_normal((N, N)) / 64).astype(np.float32))
    dSsym = (dS + dS.t()).contiguous()
    dZ, dH = raw_bwd(L, Z, H, dSsym, T)
    bw = dr.backward(dS)
    check_ratio(tag + " dense dS", "dZ", dZ, bw["dZ"], bw["A_dZ"])
    check_ratio(tag + " dense dS", "dH", dH, bw["dH"], bw["A_dH"])
    dZ2, dH2 = raw_bwd(L, Z, H, dSsym, T)
    assert torch.equal(dZ, dZ2) and torch.equal(dH, dH2)

    # backward with the script's gradient: BCE over boolean masks, dSsym mostly exact zeros
    P = max(1, N * N // 20)
    pos = dense_mask(rng.integers(0, N, P), rng.integers(0, N, P), N).to(DEV) == 1
    neg = dense_mask(rng.integers(0, N, P), rng.integers(0, N, P), N).to(DEV) == 1
    seen = {}

    def keep(g):
        seen["gP"] = g.detach().clone()
    link_pred.register_hook(keep)
    script_loss(link_pred, pos, neg, 5).backward()
    dS_used = seen["gP"] * (1.0 - prob) * prob                         # what _AllPairsScore.backward forms
    dSsym_used = (dS_used + dS_used.t()).contiguous()
    if N > 16:
        assert (dSsym_used == 0).float().mean().item() > 0.5
    bwm = dr.backward(dS_used)
    check_ratio(tag + " script dS", "dZ", Zg.grad, bwm["dZ"], bwm["A_dZ"])
    check_ratio(tag + " script dS", "dH", Hg.grad, bwm["dH"], bwm["A_dH"])
    dZ3, dH3 = raw_bwd(L, Z, H, dSsym_used, T)
    assert torch.equal(dZ3, Zg.grad) and torch.equal(dH3, Hg.grad)

    # alpha0 [K,N,N], every element written
    a0 = _nan(K, N, N)
    assert L.dl_dense_alpha0(Z.data_ptr(), N, K, d, float(T), a0.data_ptr(), _stream()) == 0
    for k in range(K):
        E, A = dr.alpha0(k)
        check_ratio(tag, "alpha0", a0[k], E, A)


def check_att(att, rowptr, col, kstar, w, s):
    """att [K,N,N] == fp32(w / s[col, kstar]) at (kstar, row, col) of every entry (a single IEEE division: bit for
    bit) and exactly 0 everywhere else."""
    rowptr, col, kstar, w, s = (_np(x) for x in (rowptr, col, kstar, w, s))
    nnz = int(rowptr[-1])
    rows = np.repeat(np.arange(rowptr.size - 1), np.diff(rowptr))
    cols, ks = col[:nnz].astype(np.int64), kstar[:nnz].astype(np.int64)
    want = w[:nnz] / s[cols, ks]
    assert want.dtype == np.float32
    got = att[_t(ks), _t(rows), _t(cols)].cpu().numpy()
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert int(torch.count_nonzero(att)) == int(np.count_nonzero(want))


def _att_case(ops, Graph, src, dst, n, K, d, T, directed=False):
    Z = _t(kernel_inputs(n, K, d, n + K)[0])
    g = Graph.from_edges(_t(src), _t(dst), n, directed=directed)
    kstar, w, s = ops.edge_attn_fwd(g, Z, T)
    att = ops.dense_att(g, kstar, w, s, K)
    check_att(att, g.rowptr, g.col, kstar, w, s)
    return g, kstar, s


@pytest.mark.gpu
def test_dense_att_hub_rows_and_grid_wrap():
    """hard_graph: hub rows of 511 .. 2049 entries (the lane loop); N = 40000 > the 37888 warps of the capped
    grid (the grid-stride loop), K = 2 so that the [K,N,N] offsets pass 2^31."""
    from disenlink_b200 import ops
    from disenlink_b200.graph import Graph
    for n, m, K, d in ((6000, 20000, 5, 32), (40000, 120000, 2, 16)):
        src, dst = hard_graph(n, m, 11)
        g, _, _ = _att_case(ops, Graph, src, dst, n, K, d, 1.5)
        assert int(np.diff(_np(g.rowptr)).max()) >= 2049


@pytest.mark.gpu
def test_dense_att_directed_graph_with_clamped_row_sums():
    """A graph marked directed: a column j with no out-entry routed to k has s[j,k] clamped to 1, and att divides
    by it."""
    from disenlink_b200 import ops
    from disenlink_b200.graph import Graph
    n, K = 6000, 4
    src, dst = directed_graph(n, 20000, 4)
    g, kstar, s = _att_case(ops, Graph, src, dst, n, K, 16, 2.0, directed=True)
    rowptr, col = csr_of(src, dst, n)
    assert np.array_equal(_np(g.rowptr), rowptr) and np.array_equal(_np(g.col)[:g.nnz], col)
    kstar = _np(kstar)[:g.nnz]
    k64, c64 = kstar.astype(np.int64), col.astype(np.int64)
    clamped = ~routed_mask(rowptr, kstar, K)[c64, k64]
    assert clamped.any(), "no entry whose column has no out-entry routed to its factor"
    assert np.all(_np(s)[c64[clamped], k64[clamped]] == 1.0)


@pytest.mark.gpu
def test_dense_att_empty_graph_and_one_node():
    from disenlink_b200 import ops
    from disenlink_b200.graph import Graph
    e = np.zeros(0, np.int64)
    g, _, _ = _att_case(ops, Graph, e, e, 20, 3, 8, 1.0)
    assert g.nnz == 0
    g, _, s = _att_case(ops, Graph, np.zeros(1, np.int64), np.zeros(1, np.int64), 1, 3, 8, 1.0)
    assert g.nnz == 1


# ------------------------------------------------------------------------------------------
# GPU: the module at the script's shapes
# ------------------------------------------------------------------------------------------
# (fixture, K, nhid, d, beta, T): main_disentangled.py's defaults on Cora (K=3, nhid=512, d=32), the tuned Cora,
# chameleon and squirrel settings of hyperparameters_setting, T = 2 on squirrel
MODULE_CASES = [("cora_K3_d32", 3, 512, 32, 0.9, 1), ("cora_K3_d32", 10, 256, 64, 0.6, 1),
                ("chameleon_K5_d32", 5, 512, 32, 0.7, 1), ("squirrel_K8_d16", 5, 512, 64, 0.5, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,K,nhid,d,beta,T", MODULE_CASES)
def test_module_dense_path_at_script_shapes(oracle, name, K, nhid, d, beta, T):
    from disenlink_b200.graph import Graph
    from disenlink_b200.model import Disentangle
    tag = f"{name} K={K} nhid={nhid} d={d} T={T}"
    g = load_golden(name)
    n, m_neg = int(g["N"]), float(g["m"])
    src, dst = g["src"], g["dst"]
    nfeat = 96
    torch.manual_seed(K * 100 + d)
    m = Disentangle(nfeat, nhid, d, K, beta, t=T).to(DEV)
    x = _t(np.random.default_rng(K + d).standard_normal((n, nfeat)).astype(np.float32))
    adj = adj_sym_of(src, dst, n).to(DEV)
    pos = dense_mask(g["loss_pos_u"], g["loss_pos_v"], n).to(DEV) == 1
    neg = dense_mask(g["loss_neg_u"], g["loss_neg_v"], n).to(DEV) == 1

    # routing: bit-exact against the oracle on the fp32 Z of the projection
    Z = m.project(x).detach()
    Hs, kstar, w, s, graph = m.disentangle_layer1.sparse_forward(Z, adj)
    rowptr, col = oracle.csr_from_edges(src, dst, n)
    assert np.array_equal(_np(graph.rowptr), rowptr) and np.array_equal(_np(graph.col), col)
    o_k, o_w, _ = oracle.edge_attn_fwd(rowptr, col, _np(Z), float(T))
    nnz = graph.nnz
    kstar, w = kstar[:nnz], w[:nnz]
    assert np.array_equal(_np(kstar), o_k)
    assert np.array_equal(_np(w).view(np.uint32), o_w.view(np.uint32))

    # the script's step
    H, link_pred = m(x, adj)
    loss = script_loss(link_pred, pos, neg, m_neg)
    loss.backward()
    grads = {k: p.grad.detach().clone() for k, p in m.named_parameters()}
    assert torch.equal(H.view(n, K, d), Hs)
    # dL/dZ with Z a leaf (the factor MLPs replaced by _Leaf, as the live-reference test does)
    leaf = _Leaf(Z).to(DEV)
    object.__setattr__(m, "project", leaf)
    seen = {}

    def keep(gP):
        seen["gP"] = gP.detach().clone()
    try:
        H2, lp2 = m(x, adj)
        lp2.register_hook(keep)
        script_loss(lp2, pos, neg, m_neg).backward()
    finally:
        del m.__dict__["project"]
    assert torch.equal(lp2, link_pred) and torch.equal(H2, H)
    dZ = leaf.z.grad
    # dL/dlogit as the step forms it (_AllPairsScore.backward).  torch's fp32 BCE passes no gradient through a
    # probability that rounds to 1 or 0 -- model.py's fp32 link_pred does the same, and at these shapes some
    # masked pairs have logits of several hundred -- so the float64 reference takes this dS, not its own loss's.
    dS_step = seen["gP"] * (1.0 - lp2.detach()) * lp2.detach()

    # float64: H and its A from Ref64, dL/dZ from dense64 carrying dS_step, both routed by the GPU's kstar
    ref = Ref64(rowptr, col, _np(Z), o_k, beta, T)
    check_ratio(tag, "H", H.view(n, K, d), ref.H, ref.A_H)
    fw = DenseRef64(Z, ref.H, T, A_H=ref.A_H, device=DEV).forward()
    check_ratio(tag, "prob", link_pred, fw["prob"], fw["A_prob"])
    Zd = Z.double().requires_grad_(True)
    kd = torch.zeros(n, n, dtype=torch.float64, device=DEV)
    rows = torch.repeat_interleave(torch.arange(n, device=DEV), torch.diff(graph.rowptr))
    kd[rows, graph.col.long()] = kstar.double() + 1
    H64, logits64 = dense64(Zd, adj.double(), kd, beta, float(T))
    assert torch.allclose(H64.detach().cpu(), ref.H.detach(), rtol=1e-12, atol=1e-12)
    assert torch.allclose(logits64.detach(), fw["logit"], rtol=1e-12, atol=1e-12)
    (dZ64,) = torch.autograd.grad(logits64, Zd, grad_outputs=dS_step.double())
    del kd, H64, logits64
    q = row_ratio(_np(dZ), _np(dZ64))
    RATIOS.setdefault(tag, {})["dZ_row"] = q
    print(f"RATIO {tag} dZ_row={q:.3g}")
    assert q <= C_DENSE["dZ_row"], f"{tag} dZ: {q:.3g} (bar {C_DENSE['dZ_row']})"
    # every parameter gradient: the float64 projection's vector-Jacobian product with dL/dZ, through the ReLU
    # pattern of the fp32 forward (a hidden unit within rounding of 0 may take the other branch in float64, and
    # that moves a first-layer gradient by a whole term)
    P64 = {k: p.detach().double().requires_grad_(True) for k, p in m.named_parameters()}
    with torch.no_grad():
        W1 = torch.cat([f.mlp1.weight for f in m.factors], 0)
        b1 = torch.cat([f.mlp1.bias for f in m.factors], 0)
        live = (torch.addmm(b1, x, W1.t()) > 0).view(n, K, nhid)       # Disentangle.project's first layer
    x64 = x.double()
    Z64 = torch.stack([(((x64 @ P64[f"factor_{k}.mlp1.weight"].t() + P64[f"factor_{k}.mlp1.bias"]) * live[:, k])
                        @ P64[f"factor_{k}.mlp2.weight"].t() + P64[f"factor_{k}.mlp2.bias"]) for k in range(K)], 1)
    g64 = torch.autograd.grad(Z64, list(P64.values()), grad_outputs=dZ64)
    for k, gr in zip(P64, g64):
        err = (grads[k].double() - gr).abs().max().item() / max(gr.abs().max().item(), 1e-30)
        assert err < 5e-5, f"{tag} grad {k}: max-abs rel err {err:.2e}"

    # Disentangle_layer's triplet at this size
    h_list, alpha0, att = m.disentangle_layer1([Z[:, k] for k in range(K)], adj)
    assert torch.equal(torch.stack(h_list, 1), Hs)
    dr = DenseRef64(Z, Hs, T, device=DEV)
    for k in range(K):
        E, A = dr.alpha0(k)
        check_ratio(tag, "alpha0", alpha0[k], E, A)
    check_att(torch.stack(att), graph.rowptr, graph.col, kstar, w, s)
    del alpha0, att

    # the Graph / LinkScorer path scores the same masked pairs within the same bound
    _, scorer = m(x, Graph.from_edges(_t(src), _t(dst), n))
    for mask in (pos, neg):
        check_ratio(tag + " scorer", "prob", scorer[mask], fw["prob"][mask], fw["A_prob"][mask])


# ------------------------------------------------------------------------------------------
# GPU: limits and errors
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_empty_inputs_return_empty_tensors():
    from disenlink_b200 import ops
    Z = torch.zeros(0, 3, 8, device=DEV, requires_grad=True)
    H = torch.zeros(0, 3, 8, device=DEV, requires_grad=True)
    prob = ops.allpairs_score(Z, H, 1.0)
    assert prob.shape == (0, 0)
    prob.sum().backward()
    assert Z.grad.shape == (0, 3, 8) and H.grad.shape == (0, 3, 8)
    assert ops.dense_alpha0(Z, 2.0).shape == (3, 0, 0)


@pytest.mark.gpu
def test_entry_points_refuse_bad_arguments(L):
    from disenlink_b200 import _lib, ops
    from disenlink_b200._lib import DlError
    EINVAL = -1
    N, K, d = 17, 3, 8
    Z = torch.ones(N, K, d, device=DEV)
    buf = torch.zeros(4 * N * N * K, device=DEV)
    st = _stream()
    p, b = Z.data_ptr(), buf.data_ptr()

    def fwd(N_, K_, d_, T_):
        return L.dl_allpairs_score_fwd(p, p, N_, K_, d_, T_, b, st)

    def bwd(N_, K_, d_, T_):
        return L.dl_allpairs_score_bwd(p, p, b, N_, K_, d_, T_, b, b, st)

    def a0(N_, K_, d_, T_):
        return L.dl_dense_alpha0(p, N_, K_, d_, T_, b, st)

    for f in (fwd, bwd, a0):
        assert f(0, K, d, 1.0) == 0
        for T_ in (0.0, float("nan")):
            assert f(N, K, d, T_) == EINVAL
        for K_, d_ in ((0, d), (_lib.DL_MAX_K + 1, d), (K, 0), (K, _lib.DL_MAX_D + 1)):
            assert f(N, K_, d_, 1.0) == EINVAL
        assert f(-1, K, d, 1.0) == EINVAL
    # more than 65535 tiles of 16 per side: refused before any launch or read
    assert fwd(16 * 65535 + 1, K, d, 1.0) == _lib.DL_EUNSUPPORTED
    torch.cuda.synchronize()
    assert torch.count_nonzero(buf).item() == 0
    for T_ in (0.0, float("nan")):
        with pytest.raises(DlError):
            ops.allpairs_score(Z, Z, T_)
        with pytest.raises(DlError):
            ops.dense_alpha0(Z, T_)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["Disentangle", "Disentangle_layer"])
def test_dense_limit_raises_before_allocating(which):
    """Over dense_limit the forward raises before the [N,N] / [K,N,N] output is allocated."""
    from disenlink_b200.model import Disentangle, Disentangle_layer
    K, d = 2, 8
    n = 16385 if which == "Disentangle" else 8193
    adj = torch.zeros(n, n, device=DEV)
    i = torch.arange(n - 1, device=DEV)
    adj[i, i + 1] = 1
    adj[i + 1, i] = 1
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    if which == "Disentangle":
        m = Disentangle(4, 1, d, K, 0.5).to(DEV)
        x = torch.randn(n, 4, device=DEV)
        with pytest.raises(RuntimeError, match="dense_limit"):
            m(x, adj)
    else:
        layer = Disentangle_layer(K, 0.5)
        Z = torch.randn(n, K, d, device=DEV)
        with pytest.raises(RuntimeError, match="dense_limit"):
            layer([Z[:, k] for k in range(K)], adj)
    assert torch.cuda.max_memory_allocated() - base < n * n * 4
