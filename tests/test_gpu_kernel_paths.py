"""Every kernel path against a float64 reference (pytest -m gpu for the GPU half).

Each hot-path entry point picks one of several implementations on the host side (factor-per-lane, streaming,
row-per-warp with hub segments + fixup kernels, runtime-generic), depending on (K, d), dl_graph.flags and whether
the graph carries its COO row array (erow).  DESIGN.md section 4.4 promises identical results up to the stated
tolerances under every flag; this file holds every path to that promise:

  * Ref64: the sparse hot path restated on the CSR entries in float64 with torch.autograd (routing kstar taken
    from the oracle: bit-exact routing is the contract).  Pinned in the CPU suite to the dense restatement of
    model.py (tests/test_oracle_live_reference.py) and to the oracle.
  * a per-element checker: |gpu - ref64| <= C * 2^-24 * A, A = the same sum with every term in absolute value
    (the rounding error a correctly ordered fp32 evaluation can reach), so a wrong term in a small row is not
    hidden by the tensor's largest value.  Its sensitivity to a missing entry, a wrong normaliser and a scaled
    isolated row is tested in the CPU suite.
  * a graph generator that asserts it produced the cases the kernels special-case: hub rows around the
    DL_SEG = 512 segment length, rows starting / ending exactly on a streaming range boundary, rows spanning
    three or more ranges, empty rows at a boundary, an active last node.
  * the path matrix (flag sets x shapes), a kernel-name check per flag set under torch.profiler, the
    erow = NULL entry points, a graph at the largest range length (nnz >= 2^24), and single ranks of the
    node-partitioned step (rectangular rank-local graphs with halo columns) on one GPU.
"""
import re
from functools import lru_cache

import numpy as np
import pytest
import torch
from torch.utils.checkpoint import checkpoint

from conftest import load_golden
from test_gpu_parity import ORA_TOL, dl, random_graph, relerr, run_all, t  # noqa: F401  (dl is a fixture)
from test_oracle_live_reference import adj_sym_of

EPS = 2.0 ** -24
TINY = 1e-37
DL_SEG = 512
HUB_DEGREES = (511, 512, 513, 1024, 1025, 2049)
BETA, TEMP = 0.3, 1.5            # T != 1 and beta away from 0.5: both enter every kernel's arithmetic

# Bars of the per-element checker, in units of 2^-24 * A (see sum_ratio) and, for the factor backward's dZ, of
# 2^-24 * max(|row|_inf, 1e-3 |dZ|_inf) (see row_ratio).  Each is at most 4x the largest ratio observed over every
# path, shape, graph size and partitioned rank of this file on an NVIDIA B200 (1000 W power limit); the observed
# value is in the comment.  The paths agree with each other far more closely than these bars.
C_BAR = {
    "s": 5.6,          # 1.40  (K = 32, d = 8)
    "H": 10.0,         # 2.57  (K = 10, d = 32)
    "logit": 0.3,      # 0.077 (A bounds the exp factor loosely)
    "dZp": 2.8,        # 0.717
    "dHp": 3.2,        # 0.802
    "r": 1.7,          # 0.445
    "dZ_row": 92.0,    # 23.3  (partitioned rank, decoder + factor gradient)
}


# ------------------------------------------------------------------------------------------
# streaming range length (dl_common.cuh: dl_range_shift; a range is 32 << shift entries)
# ------------------------------------------------------------------------------------------
def dl_range_shift(nnz):
    n_chunks = (int(nnz) + 31) // 32
    sh = 6
    while sh > 0 and (n_chunks >> sh) < 8192:
        sh -= 1
    return sh


def range_len(nnz):
    return 32 << dl_range_shift(nnz)


# ------------------------------------------------------------------------------------------
# graph generator
# ------------------------------------------------------------------------------------------
def hard_graph(n, m_rand, seed, hubs=HUB_DEGREES):
    """Symmetric edge list (src, dst) over n nodes with hub rows of exactly the degrees `hubs`, a row that starts
    (and its predecessor, which ends) exactly on a streaming range boundary, two empty rows sitting on another
    boundary, and an active last node.  Stars make the hubs (their centres touch nothing else); self-loops move
    the entry offsets one at a time without breaking symmetry."""
    rng = np.random.default_rng(seed)
    i0, ia = n // 3, (2 * n) // 3          # row i0 starts on a boundary; rows ia, ia+1 are empty, on another one
    special = np.array([i0 - 1, i0, ia - 1, ia, ia + 1, ia + 2, n - 1])
    hub_ids = rng.choice(np.setdiff1d(np.arange(1, n - 1), special), len(hubs), replace=False)
    plain = np.setdiff1d(np.arange(n), np.concatenate([hub_ids, [ia, ia + 1]]))
    a, b = rng.choice(plain, m_rand), rng.choice(plain, m_rand)
    a, b = a[a != b], b[a != b]
    sa = [a, np.repeat(hub_ids, hubs)]
    sb = [b, np.concatenate([rng.choice(plain[plain != h], m, replace=False) for h, m in zip(hub_ids, hubs)])]
    must = np.array([i0 - 1, i0, ia - 1, ia + 2, n - 1])
    sa.append(must)
    sb.append(np.where(must == plain[0], plain[1], plain[0]))
    a, b = np.concatenate(sa), np.concatenate(sb)
    key = np.unique(np.minimum(a, b) * n + np.maximum(a, b))
    lo, hi = key // n, key % n
    deg = np.bincount(lo, minlength=n) + np.bincount(hi, minlength=n)
    RL = range_len(deg.sum())
    loops = []
    for target, first in ((i0, 1), (ia, i0)):
        off = int(deg[:target].sum())
        delta = (-off) % RL
        cand = np.setdiff1d(plain[(plain >= first) & (plain < target - 1)], np.array(loops + [i0 - 1], np.int64))
        pick = rng.choice(cand, delta, replace=False)
        deg[pick] += 1
        loops += pick.tolist()
    assert range_len(deg.sum()) == RL
    loops = np.array(loops, np.int64)
    return np.concatenate([lo, loops]).astype(np.int64), np.concatenate([hi, loops]).astype(np.int64)


def graph_cases(rowptr, hubs=HUB_DEGREES):
    """Asserts the hard cases are present in the CSR; -> dict of example rows for each."""
    rowptr = np.asarray(rowptr, np.int64)
    deg = np.diff(rowptr)
    nnz = int(rowptr[-1])
    RL = range_len(nnz)
    rows = np.arange(deg.size)
    live = deg > 0
    for m in hubs:
        assert (deg == m).any(), f"no hub row of degree {m}"
    start = rows[live & (rowptr[:-1] % RL == 0) & (rowptr[:-1] > 0)]
    end = rows[live & (rowptr[1:] % RL == 0) & (rowptr[1:] < nnz)]
    span3 = rows[live & ((rowptr[1:] - 1) // RL - rowptr[:-1] // RL >= 2)]
    empty = rows[~live & (rowptr[:-1] % RL == 0) & (rowptr[:-1] > 0) & (rowptr[:-1] < nnz)]
    assert start.size, "no row starts on a range boundary"
    assert end.size, "no row ends on a range boundary"
    assert span3.size, "no row spans 3 ranges"
    assert empty.size, "no empty row at a range boundary"
    assert deg[-1] > 0, "last node has no entries"
    cross = rows[live & ((rowptr[1:] - 1) // RL > rowptr[:-1] // RL) & (deg < DL_SEG)]
    assert cross.size, "no non-hub row crosses a range boundary"
    return dict(RL=RL, shift=dl_range_shift(nnz), start=start, end=end, span3=span3, empty=empty,
                cross=cross, hubs=rows[deg >= DL_SEG], isolated=rows[~live])


# nnz ~ 5e4 (range shift 0), ~ 6e5 (shift 1), ~ 1.7e7 (shift 6: nnz >= 2^24)
SIZES = {"shift0": (6000, 20000, 1, HUB_DEGREES),
         "shift1": (60000, 296000, 2, HUB_DEGREES),
         "shift6": (2_000_000, 8_500_000, 3, HUB_DEGREES + (4200,))}
SIZE_SHIFT = {"shift0": 0, "shift1": 1, "shift6": 6}


@lru_cache(maxsize=None)
def hard_case(size):
    """-> (src, dst, n, rowptr, col, cases) of one generated graph (oracle CSR)."""
    from oracle import oracle as O
    n, m, seed, hubs = SIZES[size]
    src, dst = hard_graph(n, m, seed, hubs)
    rowptr, col = O.csr_from_edges(src, dst, n)
    cases = graph_cases(rowptr, hubs)
    assert cases["shift"] == SIZE_SHIFT[size]
    return src, dst, n, rowptr, col, cases


# ------------------------------------------------------------------------------------------
# float64 reference
# ------------------------------------------------------------------------------------------
def _spans(n, chunk):
    return [(a, min(a + chunk, n)) for a in range(0, n, chunk)]


def _w_chunk(Z, r, c, k, T):
    """softmax weight of the routed factor per entry (model.py:56-60 on the entries)."""
    q = (Z[r] * Z[c]).sum(-1) / T
    return torch.softmax(q, 1).gather(1, k[:, None])[:, 0]


def _agg_chunk(Z, s, w, r, c, k):
    """sum_e w / s[col, k] * Z[col, k] into row (r, k) (model.py:75 on the entries)."""
    K = Z.shape[1]
    return torch.zeros(Z.shape[0] * K, Z.shape[2], dtype=Z.dtype).index_add(0, r * K + k, (w / s[c, k])[:, None] * Z[c, k])


def _w_abs(w, Za, r, c, T):
    """A of w: the routed softmax weight carries the dot products' rounding (<= 2^-24 x sum |z_i z_j| each) through
    exp and the normalisation, twice."""
    qa = (Za[r] * Za[c]).sum(-1) / T
    return w * (2.0 + 2.0 * qa.amax(1))


class Ref64:
    """The hot path of one layer in float64 on the CSR entries; gradients from torch.autograd.

    Values: w, s, H (with graph to Z); A_s, A_H: the same sums with every term in absolute value (the A of each
    factor stands in for that factor, so error carried in from w and s is part of the bound)."""

    def __init__(self, rowptr, col, Z, kstar, beta, T, chunk=1 << 15):
        N, K, d = Z.shape
        self.N, self.K, self.d, self.beta, self.T = N, K, d, float(beta), float(T)
        self.rows = torch.from_numpy(np.repeat(np.arange(N, dtype=np.int64), np.diff(rowptr)))
        self.cols = torch.from_numpy(np.asarray(col, np.int64))
        self.ks = torch.from_numpy(np.asarray(kstar, np.int64))
        self.spans = _spans(self.cols.numel(), chunk)
        self.Z = torch.from_numpy(np.ascontiguousarray(Z)).double().requires_grad_(True)
        Z64, T = self.Z, self.T
        Za = Z64.detach().abs()
        ws, was = [], []
        for a, b in self.spans:
            r, c, k = self.rows[a:b], self.cols[a:b], self.ks[a:b]
            ws.append(checkpoint(_w_chunk, Z64, r, c, k, T, use_reentrant=False))
            with torch.no_grad():
                was.append(_w_abs(ws[-1].detach(), Za, r, c, T))
        self.w = torch.cat(ws) if ws else Z64.new_zeros(0)
        wa = torch.cat(was) if was else Z64.new_zeros(0)
        idx = self.rows * K + self.ks
        s = Z64.new_zeros(N * K).index_add(0, idx, self.w).view(N, K)
        self.s = torch.where(s == 0, torch.ones_like(s), s)
        agg = Z64.new_zeros(N * K, d)
        for a, b in self.spans:
            agg = agg + checkpoint(_agg_chunk, Z64, self.s, self.w[a:b], self.rows[a:b], self.cols[a:b], self.ks[a:b],
                                   use_reentrant=False)
        self.H = self.beta * Z64 + (1.0 - self.beta) * agg.view(N, K, d)
        with torch.no_grad():
            w, sd = self.w.detach(), self.s.detach()
            self.A_s = Z64.new_zeros(N * K).index_add(0, idx, wa).view(N, K)
            self.wa = wa
            sc, asc = sd[self.cols, self.ks], self.A_s[self.cols, self.ks]
            coefA = (wa + w * asc / sc + w) / sc
            AH = Z64.new_zeros(N * K, d)
            for a, b in self.spans:
                AH.index_add_(0, idx[a:b], coefA[a:b, None] * Za[self.cols[a:b], self.ks[a:b]])
            self.A_H = self.beta * Za + (1.0 - self.beta) * AH.view(N, K, d)

    def logits(self, u, v, H):
        Z = self.Z
        e = torch.exp((Z[u] * Z[v]).sum(-1) / self.T)
        return (e * (H[u] * H[v]).sum(-1)).sum(1)

    def decoder(self, u, v, dS):
        """-> dict(logit, dZp, dHp and their A) for the pair list (u, v) and dL/dlogit = dS (H held fixed)."""
        u, v = torch.from_numpy(np.asarray(u, np.int64)), torch.from_numpy(np.asarray(v, np.int64))
        dS = torch.from_numpy(np.asarray(dS, np.float64))
        Hl = self.H.detach().requires_grad_(True)
        logit = self.logits(u, v, Hl)
        dZp, dHp = torch.autograd.grad((logit * dS).sum(), (self.Z, Hl))
        with torch.no_grad():
            Za, Hd, AH, T = self.Z.detach().abs(), Hl.detach().abs(), self.A_H, self.T
            e = torch.exp((self.Z[u] * self.Z[v]).sum(-1) / T)
            ea = e * (2.0 + 2.0 * (Za[u] * Za[v]).sum(-1) / T)
            ha = (AH[u] * Hd[v] + Hd[u] * AH[v] + Hd[u] * Hd[v]).sum(-1)
            g = dS.abs()[:, None]
            A_dH = torch.zeros_like(Hd).index_add(0, u, (g * ea)[:, :, None] * (AH[v] + Hd[v]))
            A_dH.index_add_(0, v, (g * ea)[:, :, None] * (AH[u] + Hd[u]))
            cz = (g * ea * ha / T)[:, :, None]
            A_dZ = torch.zeros_like(Za).index_add(0, u, cz * Za[v]).index_add(0, v, cz * Za[u])
            A_logit = (ea * ha).sum(1)
        return dict(logit=logit.detach().numpy(), A_logit=A_logit.numpy(), dZp=dZp.numpy(), A_dZp=A_dZ.numpy(),
                    dHp=dHp.numpy(), A_dHp=A_dH.numpy())

    def factor_bwd(self, G):
        """-> dict(dZ = autograd of <H, G> w.r.t. Z, r, A_r) for G = dL/dH."""
        G64 = torch.from_numpy(np.ascontiguousarray(G)).double()
        (dZ,) = torch.autograd.grad(self.H, self.Z, grad_outputs=G64, retain_graph=True)
        with torch.no_grad():
            N, K = self.N, self.K
            Z, Za, Ga = self.Z.detach(), self.Z.detach().abs(), G64.abs()
            w, s, As = self.w.detach(), self.s.detach(), self.A_s
            idx = self.rows * K + self.ks
            racc = torch.zeros(N * K, dtype=torch.float64)
            aacc = torch.zeros(N * K, dtype=torch.float64)
            si, asi = s[self.rows, self.ks], As[self.rows, self.ks]
            for a, b in self.spans:
                r, c, k = self.rows[a:b], self.cols[a:b], self.ks[a:b]
                racc.index_add_(0, idx[a:b], w[a:b] * (Z[r, k] * G64[c, k]).sum(-1))
                aacc.index_add_(0, idx[a:b], (self.wa[a:b] + 2 * w[a:b] * asi[a:b] / si[a:b] + w[a:b]) *
                                (Za[r, k] * Ga[c, k]).sum(-1))
            omb = 1.0 - self.beta
            rr = omb * racc.view(N, K) / s ** 2
            A_r = omb * aacc.view(N, K) / s ** 2
        return dict(dZ=dZ.numpy(), r=rr.numpy(), A_r=A_r.numpy())

    def forward_dict(self):
        return dict(s=self.s.detach().numpy(), A_s=self.A_s.numpy(), H=self.H.detach().numpy(),
                    A_H=self.A_H.numpy())


def ref64_rows(rowptr, col, Z, kstar, beta, T, G, rows_sel, chunk=1 << 16):
    """s, H, r (and their A) of the rows `rows_sel` only, for graphs too large for Ref64 on the host: the row
    sums of the rows and of their neighbours come from the entries of those rows alone."""
    rowptr = np.asarray(rowptr, np.int64)
    col = np.asarray(col, np.int64)
    rows_sel = np.unique(rows_sel)

    def entries(rows):
        cnt = rowptr[rows + 1] - rowptr[rows]
        start = np.repeat(rowptr[rows] - np.cumsum(cnt) + cnt, cnt)
        return np.repeat(rows, cnt), start + np.arange(cnt.sum())

    r0, e0 = entries(rows_sel)
    need = np.unique(np.concatenate([rows_sel, col[e0]]))
    r1, e1 = entries(need)
    N, K, d = Z.shape
    loc = np.full(N, -1, np.int64)
    loc[need] = np.arange(need.size)
    Zn = torch.from_numpy(Z[need]).double()
    s = torch.zeros(need.size * K, dtype=torch.float64)
    As = torch.zeros_like(s)
    ws, was = [], []
    cl = torch.from_numpy(loc[col[e1]])
    rl = torch.from_numpy(loc[r1])
    k1 = torch.from_numpy(kstar[e1].astype(np.int64))
    Zna = Zn.abs()
    for a, b in _spans(e1.size, chunk):
        # the neighbours' rows reach two hops out: their Z is gathered per chunk
        zr = torch.from_numpy(Z[r1[a:b]]).double()
        zc = torch.from_numpy(Z[col[e1[a:b]]]).double()
        ar = torch.arange(b - a)
        w = _w_chunk(torch.cat([zr, zc]), ar, ar + (b - a), k1[a:b], T)
        ws.append(w)
        was.append(_w_abs(w, torch.cat([zr, zc]).abs(), ar, ar + (b - a), T))
    w, wa = torch.cat(ws), torch.cat(was)
    s.index_add_(0, rl * K + k1, w)
    As.index_add_(0, rl * K + k1, wa)
    s, As = s.view(-1, K), As.view(-1, K)
    s = torch.where(s == 0, torch.ones_like(s), s)
    # entries of the selected rows inside the e1 list
    pos = np.searchsorted(e1, e0)
    assert np.array_equal(e1[pos], e0)
    pos = torch.from_numpy(pos)
    w0, wa0 = w[pos], wa[pos]
    rs = torch.from_numpy(np.searchsorted(rows_sel, r0))
    c0, k0 = cl[pos], k1[pos]
    sc, asc = s[c0, k0], As[c0, k0]
    idx = rs * K + k0
    M = rows_sel.size
    agg = torch.zeros(M * K, d, dtype=torch.float64).index_add(0, idx, (w0 / sc)[:, None] * Zn[c0, k0])
    coefA = (wa0 + w0 * asc / sc + w0) / sc
    aggA = torch.zeros(M * K, d, dtype=torch.float64).index_add(0, idx, coefA[:, None] * Zna[c0, k0])
    zs = Zn[torch.from_numpy(loc[rows_sel])]
    H = beta * zs + (1 - beta) * agg.view(M, K, d)
    A_H = beta * zs.abs() + (1 - beta) * aggA.view(M, K, d)
    ri = torch.from_numpy(loc[r0])
    si, asi = s[ri, k0], As[ri, k0]
    Gc = torch.from_numpy(G[col[e0]]).double()
    ar = torch.arange(e0.size)
    x = (Zn[ri, k0] * Gc[ar, k0]).sum(-1)
    xa = (Zna[ri, k0] * Gc[ar, k0].abs()).sum(-1)
    racc = torch.zeros(M * K, dtype=torch.float64).index_add(0, idx, w0 * x)
    aacc = torch.zeros(M * K, dtype=torch.float64).index_add(0, idx, (wa0 + 2 * w0 * asi / si + w0) * xa)
    ss = s[torch.from_numpy(loc[rows_sel])]
    return rows_sel, dict(s=ss.numpy(), A_s=As[torch.from_numpy(loc[rows_sel])].numpy(), H=H.numpy(),
                          A_H=A_H.numpy(), r=((1 - beta) * racc.view(M, K) / ss ** 2).numpy(),
                          A_r=((1 - beta) * aacc.view(M, K) / ss ** 2).numpy())


# ------------------------------------------------------------------------------------------
# the checker
# ------------------------------------------------------------------------------------------
def sum_ratio(x, ref, A):
    """max |x - ref| / (2^-24 A): the error in units of what one rounding per term can reach."""
    x = np.asarray(x, np.float64)
    if x.size == 0:
        return 0.0
    return float((np.abs(x - ref) / (EPS * np.asarray(A) + TINY)).max())


def row_ratio(x, ref):
    """max over rows of max|x_row - ref_row| / (2^-24 max(|ref_row|_inf, 1e-3 |ref|_inf))."""
    x = np.asarray(x, np.float64).reshape(len(x), -1)
    ref = np.asarray(ref, np.float64).reshape(len(ref), -1)
    if x.size == 0:
        return 0.0
    den = np.maximum(np.abs(ref).max(1), 1e-3 * np.abs(ref).max())
    return float((np.abs(x - ref).max(1) / (EPS * den + TINY)).max())


RATIOS = {}


def check_outputs(tag, out, ref, names=("s", "H", "logit", "dZp", "dHp", "r", "dZ")):
    """out: fp32 results; ref: Ref64 values and their A.  Records and asserts every ratio."""
    got = {}
    for k in names:
        if k not in out:
            continue
        if k == "dZ":
            q = row_ratio(out[k], ref[k])
            got["dZ_row"] = q
            assert relerr(out[k], ref[k]) < 5 * ORA_TOL, f"{tag} dZ: max-abs rel err {relerr(out[k], ref[k]):.2e}"
        else:
            got[k] = sum_ratio(out[k], ref[k], ref["A_" + k])
    RATIOS[tag] = got
    print(f"RATIO {tag} " + " ".join(f"{k}={v:.3g}" for k, v in got.items()))
    for k, q in got.items():
        assert np.isfinite(q) and q <= C_BAR[k], f"{tag} {k}: error {q:.3g} x 2^-24 x A (bar {C_BAR[k]})"


def reject(out, ref, name):
    """True when the checker flags `out[name]`."""
    if name == "dZ":
        return row_ratio(out[name], ref[name]) > C_BAR["dZ_row"]
    return sum_ratio(out[name], ref[name], ref["A_" + name]) > C_BAR[name]


# ------------------------------------------------------------------------------------------
# inputs of one (graph, shape) case
# ------------------------------------------------------------------------------------------
def case_inputs(n, K, d, hub_node, seed):
    rng = np.random.default_rng(seed)
    Z = (rng.standard_normal((n, K, d)) * (0.8 / np.sqrt(np.sqrt(d)))).astype(np.float32)
    G = rng.standard_normal((n, K, d)).astype(np.float32)
    pu = np.concatenate([np.repeat(rng.integers(0, n, 300), 6), np.full(700, hub_node), np.arange(0, n, n // 50)])
    pv = np.concatenate([rng.integers(0, n, 2500), np.arange(0, n, n // 50)])        # incl. u == v pairs
    dS = (rng.standard_normal(pu.size) / 64).astype(np.float32)
    return Z, G, pu.astype(np.int64), pv.astype(np.int64), dS


@lru_cache(maxsize=None)
def shape_case(size, K, d):
    """Oracle routing and the float64 reference of one (graph, shape): shared by every flag set."""
    from oracle import oracle as O
    src, dst, n, rowptr, col, cases = hard_case(size)
    Z, G, pu, pv, dS = case_inputs(n, K, d, int(cases["hubs"][0]), K * 1000 + d)
    o_k, o_w, o_s = O.edge_attn_fwd(rowptr, col, Z, TEMP)
    ref = Ref64(rowptr, col, Z, o_k, BETA, TEMP)
    res = ref.forward_dict()
    res.update(ref.decoder(pu, pv, dS))
    res.update(ref.factor_bwd(G))
    del ref
    return dict(Z=Z, G=G, pu=pu, pv=pv, dS=dS, o_k=o_k, o_w=o_w, ref=res)


def gpu_run(ops, Graph, src, dst, n, c, erow_null=False):
    """One step of the hot path on the GPU under the flags in DL_FLAGS: both aggregation variants (pre-scaled
    slices and the per-entry normaliser copy sj, which pass 2 then reads)."""
    g = Graph.from_edges(t(src), t(dst), n)
    g.sym_min_nnz = 0
    if erow_null:
        g.struct.erow = None
    Zt = t(c["Z"])
    kstar, w, s = ops.edge_attn_fwd(g, Zt, TEMP)
    H = ops.factor_spmm_fwd(g, Zt, kstar, w, s, BETA, zs=torch.empty_like(Zt))
    sj = torch.full((max(g.nnz, 1),), float("nan"), dtype=torch.float32, device=Zt.device)
    H_sj = ops.factor_spmm_fwd(g, Zt, kstar, w, s, BETA, sj=sj)
    batch = ops.PairBatch(t(c["pu"]), t(c["pv"]), n)
    logit, _ = ops.pair_score_fwd(Zt, H, batch, TEMP)
    dZp, dHp = ops.pair_score_bwd(Zt, H, batch, t(c["dS"]), TEMP)
    dZ, r = ops.factor_bwd(g, Zt, t(c["G"]), kstar, w, s, BETA, TEMP, sj=sj[:g.nnz])
    cpu = lambda x: x.cpu().numpy()
    return dict(kstar=cpu(kstar), w=cpu(w), s=cpu(s), H=cpu(H), H_sj=cpu(H_sj), logit=cpu(logit), dZp=cpu(dZp),
                dHp=cpu(dHp), dZ=cpu(dZ), r=cpu(r), sj=cpu(sj[:g.nnz]), col=cpu(g.col), flags=g.flags)


def check_case(tag, out, c):
    assert np.array_equal(out["kstar"], c["o_k"]), f"{tag}: {(out['kstar'] != c['o_k']).sum()} routing mismatches"
    assert np.array_equal(out["w"].view(np.uint32), c["o_w"].view(np.uint32)), f"{tag}: w not bit-identical"
    ref = c["ref"]
    check_outputs(tag, out, ref)
    check_outputs(tag + " H_sj", dict(H=out["H_sj"]), ref, names=("H",))
    s = out["s"]
    assert np.array_equal(out["sj"], s[out["col"].astype(np.int64), out["kstar"].astype(np.int64)])


# ------------------------------------------------------------------------------------------
# CPU suite: generator, reference pins, checker sensitivity
# ------------------------------------------------------------------------------------------
def test_generator_produces_the_hard_cases():
    for size in ("shift0", "shift1"):
        src, dst, n, rowptr, col, cases = hard_case(size)
        deg = np.diff(rowptr)
        assert cases["RL"] == 32 << SIZE_SHIFT[size]
        assert (deg[cases["empty"]] == 0).all() and deg[-1] > 0
        # symmetric, with self-loops
        rows = np.repeat(np.arange(n), deg)
        key = rows * n + col
        assert np.array_equal(np.sort(col.astype(np.int64) * n + rows), key)
        assert (rows == col).any()


def test_range_shift_matches_the_library():
    """dl_range_shift above against the library's scratch sizing, which uses it (3 records per range)."""
    import ctypes
    from disenlink_b200 import _lib
    try:
        L = _lib.lib()
    except RuntimeError:
        pytest.skip("library not built")
    for nnz in (1, 31, 32, 2 ** 19 - 1, 2 ** 19, 2 ** 20, 2 ** 24 - 1, 2 ** 24, 3 * 2 ** 25):
        g = _lib.DlGraph(1, nnz, None, None, None, 0, 0, None, None, None, 0, 0)
        RE = range_len(nnz)
        assert L.dl_hub_scratch_floats(ctypes.byref(g), 1) == (nnz + RE - 1) // RE * 3
    # the shift steps at whole 32-entry chunks: 2^14 chunks -> 1, 2^19 chunks -> 6
    assert [dl_range_shift(x) for x in (2 ** 19 - 32, 2 ** 19 - 31, 2 ** 24 - 32, 2 ** 24 - 31)] == [0, 1, 5, 6]


def dense64(Z, adj, kstar_dense, beta, T):
    """dense_layer / dense_forward of test_oracle_live_reference.py in float64 with the routing given
    (p_adj = kstar + 1 on the entries): -> (H [N,K,d], logits [N,N])."""
    K = Z.shape[1]
    zs = [Z[:, k, :] for k in range(K)]
    alpha0 = torch.stack([torch.exp(torch.mm(z, z.t()) / T) for z in zs])
    alpha = alpha0 / torch.sum(alpha0, dim=0)
    p_adj = kstar_dense * adj
    h_list = []
    for k, z in enumerate(zs):
        a1 = (p_adj == k + 1).double() * alpha[k]
        s = torch.sum(a1, dim=1)
        s = torch.where(s == 0, torch.ones_like(s), s)
        a1 = a1 / s
        h_list.append(beta * z + (1 - beta) * torch.mm(a1, z))
    logits = sum(torch.mm(h, h.t()) * a for h, a in zip(h_list, alpha0))
    return torch.stack(h_list, 1), logits


PIN_FIXTURES = ["tiny_generic", "tiny_deadfactor_T2", "tiny_ties", "tiny_K1", "tiny_empty", "cora_K3_d32",
                "chameleon_K5_d32"]


@pytest.mark.parametrize("name", PIN_FIXTURES)
def test_ref64_matches_dense_restatement(oracle, name):
    """Ref64 (sparse, chunked, autograd) against the dense restatement of model.py in float64, same routing:
    a BCE over the fixture's pairs and its dL/dZ through decoder, aggregation and attention within 1e-9."""
    gd = load_golden(name)
    n, beta, T = int(gd["N"]), float(gd["beta"]), float(gd["T"])
    Z = gd["Z"].astype(np.float32)
    rowptr, col = oracle.csr_from_edges(gd["src"], gd["dst"], n)
    ks, _, _ = oracle.edge_attn_fwd(rowptr, col, Z, T)
    pu, pv = gd["pu"], gd["pv"]
    y = torch.from_numpy((np.random.default_rng(0).random(pu.size) < 0.5).astype(np.float64))
    bce = torch.nn.functional.binary_cross_entropy_with_logits

    ref = Ref64(rowptr, col, Z, ks, beta, T, chunk=97)      # small chunks: the chunk seams are exercised
    loss_s = bce(ref.logits(torch.from_numpy(pu), torch.from_numpy(pv), ref.H), y)
    (g_s,) = torch.autograd.grad(loss_s, ref.Z)

    Zd = torch.from_numpy(Z).double().requires_grad_(True)
    adj = adj_sym_of(gd["src"], gd["dst"], n).double()
    kd = torch.zeros(n, n, dtype=torch.float64)
    kd[torch.from_numpy(oracle.rows_of(rowptr)), torch.from_numpy(col.astype(np.int64))] = torch.from_numpy(ks.astype(np.float64)) + 1
    Hd, logits = dense64(Zd, adj, kd, beta, T)
    loss_d = bce(logits[torch.from_numpy(pu), torch.from_numpy(pv)], y)
    (g_d,) = torch.autograd.grad(loss_d, Zd)
    assert abs(loss_s.item() - loss_d.item()) <= 1e-9 * abs(loss_d.item())
    assert relerr(ref.H.detach().numpy(), Hd.detach().numpy()) < 1e-9
    assert relerr(g_s.numpy(), g_d.numpy()) < 1e-9


@lru_cache(maxsize=None)
def _hub_random_case():
    from oracle import oracle as O
    rng = np.random.default_rng(77)
    n, K, d = 3000, 5, 16
    src, dst = random_graph(rng, n - 30, 20000, hubs=((7, 2049), (11, 600), (13, 512)))   # the last 30: isolated
    rowptr, col = O.csr_from_edges(src, dst, n)
    Z = (rng.standard_normal((n, K, d)) * 0.4).astype(np.float32)
    G = rng.standard_normal((n, K, d)).astype(np.float32)
    pu = np.concatenate([rng.integers(0, n, 2000), np.full(600, 7)])
    pv = rng.integers(0, n, pu.size)
    dS = (rng.standard_normal(pu.size) / 32).astype(np.float32)
    o_k, o_w, o_s = O.edge_attn_fwd(rowptr, col, Z, TEMP)
    o_H = O.factor_spmm_fwd(rowptr, col, Z, o_k, o_w, o_s, BETA)
    o_logit, _ = O.pair_score_fwd(pu, pv, Z, o_H, TEMP)
    o_dZp, o_dHp = O.pair_score_bwd(pu, pv, Z, o_H, dS, TEMP)
    o_dZ, o_r = O.factor_bwd(rowptr, col, Z, G, o_k, o_w, o_s, BETA, TEMP, return_r=True)
    ref = Ref64(rowptr, col, Z, o_k, BETA, TEMP)
    res = ref.forward_dict()
    res.update(ref.decoder(pu, pv, dS))
    res.update(ref.factor_bwd(G))
    orc = dict(s=o_s, H=o_H, logit=o_logit, dZp=o_dZp, dHp=o_dHp, r=o_r, dZ=o_dZ)
    return rowptr, col, Z, o_k, o_w, res, orc


def test_ref64_matches_oracle_on_hub_graph():
    """The oracle's fp32 outputs against Ref64 with the oracle's routing: within 1e-6 of the tensor's max-abs;
    the factor backward's dZ within 5e-6 (the factor of 5 every gradient bar of the suite has: pass 2 subtracts
    r[i] + r[j] from c_ij / s[j] + c_ji / s[i], terms of similar size)."""
    rowptr, col, Z, o_k, o_w, ref, orc = _hub_random_case()
    assert np.diff(rowptr).max() >= 4 * DL_SEG
    for k in ("s", "H", "logit", "dZp", "dHp", "r"):
        assert relerr(orc[k], ref[k]) < 1e-6, k
    assert relerr(orc["dZ"], ref["dZ"]) < 5e-6


def test_ref64_rows_matches_ref64():
    """The sampled-row reference used at nnz >= 2^24 against the whole-graph one."""
    rowptr, col, Z, o_k, o_w, ref, orc = _hub_random_case()
    G = np.random.default_rng(77 + 1).standard_normal(Z.shape).astype(np.float32)
    full = Ref64(rowptr, col, Z, o_k, BETA, TEMP)
    rb = full.factor_bwd(G)
    deg = np.diff(rowptr)
    sel = np.concatenate([np.nonzero(deg >= DL_SEG)[0], np.nonzero(deg == 0)[0][:3], np.arange(0, Z.shape[0], 37)])
    rows, sub = ref64_rows(rowptr, col, Z, o_k, BETA, TEMP, G, sel)
    fd = full.forward_dict()
    for k in ("s", "A_s", "H", "A_H"):
        assert np.allclose(sub[k], fd[k][rows], rtol=1e-12, atol=0), k
    for k in ("r", "A_r"):
        assert np.allclose(sub[k], rb[k][rows], rtol=1e-12, atol=1e-300), k


def test_checker_accepts_oracle_and_rejects_faults():
    rowptr, col, Z, o_k, o_w, ref, orc = _hub_random_case()
    check_outputs("oracle hub graph", orc, ref)
    deg = np.diff(rowptr)
    rows = np.repeat(np.arange(deg.size), deg)
    s64 = ref["s"]
    w64 = o_w.astype(np.float64)

    def term(e):
        i, j, k = rows[e], int(col[e]), int(o_k[e])
        return i, k, (1 - BETA) * w64[e] / s64[j, k] * Z[j, k].astype(np.float64)

    def faulted(fn):
        H = ref["H"].copy()
        fn(H)
        return dict(H=H)

    # one entry's contribution removed from a hub row
    hub = int(np.argmax(deg))
    e = rowptr[hub] + deg[hub] // 2
    i, k, tm = term(e)
    assert reject(faulted(lambda H: H.__setitem__((i, k), H[i, k] - tm)), ref, "H")
    # one entry removed from a row that crosses a streaming range boundary (last entry before the boundary)
    RL = range_len(rowptr[-1])
    cross = np.nonzero((deg > 1) & (deg < DL_SEG) & ((rowptr[1:] - 1) // RL > rowptr[:-1] // RL))[0]
    x = int(cross[0])
    e = (rowptr[x] // RL + 1) * RL - 1
    i, k, tm = term(e)
    assert reject(faulted(lambda H: H.__setitem__((i, k), H[i, k] - tm)), ref, "H")
    # s[row] used where s[col] belongs (an entry whose two row sums differ)
    j_ = col.astype(np.int64)
    diff = np.nonzero(np.abs(s64[rows, o_k] - s64[j_, o_k]) > 1e-3 * s64[j_, o_k])[0]
    e = int(diff[0])
    i, j, k = rows[e], j_[e], int(o_k[e])
    wrong = (1 - BETA) * w64[e] * Z[j, k].astype(np.float64) * (1 / s64[i, k] - 1 / s64[j, k])
    assert reject(faulted(lambda H: H.__setitem__((i, k), H[i, k] + wrong)), ref, "H")
    # one isolated row's H scaled by (1 + 1e-4)
    iso = int(np.nonzero(deg == 0)[0][0])
    assert reject(faulted(lambda H: H.__setitem__(iso, H[iso] * (1 + 1e-4))), ref, "H")
    # the same fault (one entry of a hub row lost) on s and r
    e = rowptr[hub] + 3
    k = int(o_k[e])
    s_bad = ref["s"].copy()
    s_bad[hub, k] -= w64[e]
    assert reject(dict(s=s_bad), ref, "s")
    # r of a low-degree row off by 1/256 of its value
    low = np.nonzero((deg > 0) & (deg <= 4))[0]
    i = int(low[np.argmax(np.abs(ref["r"][low]).max(1))])
    r_bad = ref["r"].copy()
    r_bad[i] *= 1 + 2.0 ** -8
    assert reject(dict(r=r_bad), ref, "r")


# ------------------------------------------------------------------------------------------
# GPU: the path matrix
# ------------------------------------------------------------------------------------------
# NO_SJ / NO_SR switch off inputs of the two-sided pass 2 only (the symmetric pass 2 packs (s, r) itself and
# needs no per-entry normaliser), so that set runs two-sided
FLAG_SETS = ["", "NO_SYM", "NO_FL_ATTN", "NO_FL", "NO_XDOT", "NO_SJ,NO_SR,NO_SYM", "NO_PRESCALE", "NO_STREAM",
             "EROW_NULL"]
FL_SHAPES = [(8, 16), (8, 8), (8, 32), (5, 16), (5, 32), (3, 32), (4, 32)]
PATH_SHAPES = FL_SHAPES + [(10, 32), (7, 20), (32, 8), (2, 256), (1, 255)]
SHIFT1_SHAPES = [(8, 16), (8, 32), (3, 32), (10, 32), (7, 20)]


def _set_flags(monkeypatch, flags):
    monkeypatch.setenv("DL_FLAGS", "NO_SYM" if flags == "EROW_NULL" else flags)


def run_path_case(dl, monkeypatch, size, K, d, flags):
    ops, Graph = dl
    from disenlink_b200._lib import DlError
    src, dst, n, rowptr, col, cases = hard_case(size)
    c = shape_case(size, K, d)
    _set_flags(monkeypatch, flags)
    tag = f"{size} K={K} d={d} flags={flags or 'default'}"
    out = gpu_run(ops, Graph, src, dst, n, c, erow_null=(flags == "EROW_NULL"))
    check_case(tag, out, c)
    if flags == "EROW_NULL":
        # without the COO row array the row-per-warp kernels run: the NO_STREAM path, bit for bit
        monkeypatch.setenv("DL_FLAGS", "NO_STREAM")
        ns = gpu_run(ops, Graph, src, dst, n, c)
        for k in ("kstar", "w", "s", "H", "H_sj", "logit", "dZ", "r", "sj"):
            assert np.array_equal(out[k].view(np.uint8), ns[k].view(np.uint8)), k
        # the symmetric attention needs the row array: refused on the host before any launch
        monkeypatch.setenv("DL_FLAGS", "")
        g = Graph.from_edges(t(src), t(dst), n)
        g.sym_min_nnz = 0
        g.struct.erow = None
        with pytest.raises(DlError):
            ops.edge_attn_fwd(g, t(c["Z"]), TEMP)


@pytest.mark.gpu
@pytest.mark.parametrize("flags", FLAG_SETS)
@pytest.mark.parametrize("K,d", PATH_SHAPES)
def test_path_matrix_shift0(dl, oracle, monkeypatch, K, d, flags):
    run_path_case(dl, monkeypatch, "shift0", K, d, flags)


@pytest.mark.gpu
@pytest.mark.parametrize("flags", FLAG_SETS)
@pytest.mark.parametrize("K,d", SHIFT1_SHAPES)
def test_path_matrix_shift1(dl, oracle, monkeypatch, K, d, flags):
    run_path_case(dl, monkeypatch, "shift1", K, d, flags)


# kernel names (from the .cu files) that must / must not run for (K, d) = (8, 16) under each flag set
_GRAPH_ROW_PER_WARP = [r"k_edge_attn_fwd<", r"k_attn_hub_fixup", r"k_factor_gather<", r"k_spmm_hub_fixup",
                       r"k_factor_bwd_gather_hub<", r"k_factor_bwd_edges<", r"k_bwd_edges_hub_fixup"]
KERNELS = {
    "": ([r"k_attn_fl<", r"k_sym_expand", r"k_scale_rows", r"k_gather_stream<", r"k_bwd_edges_fl<8,\s*16,\s*2>",
          r"k_bwd_sym_lower", r"k_pair_bwd_stream"],
         [r"k_attn_hub_fixup", r"k_edge_attn_fwd<", r"k_factor_gather<", r"k_attn_stream", r"k_bwd_edges_stream"]),
    "NO_SYM": ([r"k_attn_fl<", r"k_bwd_edges_fl<8,\s*16,\s*1>", r"k_pack_sr"], [r"k_sym_expand", r"k_bwd_sym_lower"]),
    "NO_FL_ATTN": ([r"k_attn_stream<", r"k_row_sums|k_gather_chain", r"k_bwd_edges_fl<"], [r"k_attn_fl<", r"k_sym_expand"]),
    "NO_FL": ([r"k_attn_stream<", r"k_bwd_edges_stream<"], [r"k_attn_fl<", r"k_bwd_edges_fl<", r"k_sym_expand"]),
    "NO_XDOT": ([r"k_bwd_edges_fl<8,\s*16,\s*0>"], [r"k_bwd_edges_fl<8,\s*16,\s*[12]>", r"k_bwd_sym_lower"]),
    "NO_SJ,NO_SR,NO_SYM": ([r"k_bwd_edges_fl<8,\s*16,\s*1>"], [r"k_pack_sr", r"k_sym_expand"]),
    "NO_PRESCALE": ([r"k_gather_stream<"], [r"k_scale_rows"]),
    "NO_STREAM": (_GRAPH_ROW_PER_WARP + [r"k_pair_score_bwd<", r"k_pair_bwd_hub_fixup"],
                  [r"k_attn_fl<", r"stream", r"k_scale_rows", r"k_sym_expand", r"k_bwd_edges_fl<"]),
    "EROW_NULL": (_GRAPH_ROW_PER_WARP + [r"k_pair_bwd_stream"],
                  [r"k_attn_fl<", r"k_attn_stream", r"k_gather_stream", r"k_bwd_edges_stream", r"k_scale_rows",
                   r"k_bwd_edges_fl<", r"k_sym_expand"]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("flags", FLAG_SETS)
def test_flag_set_changes_the_path(dl, oracle, monkeypatch, flags):
    from torch.profiler import ProfilerActivity, profile
    ops, Graph = dl
    src, dst, n, rowptr, col, cases = hard_case("shift0")
    c = shape_case("shift0", 8, 16)
    _set_flags(monkeypatch, flags)
    gpu_run(ops, Graph, src, dst, n, c, erow_null=(flags == "EROW_NULL"))      # warm: module loads
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        gpu_run(ops, Graph, src, dst, n, c, erow_null=(flags == "EROW_NULL"))
        torch.cuda.synchronize()
    names = sorted({e.key for e in prof.key_averages() if re.search(r"\bk_\w+", e.key)})
    print(f"KERNELS {flags or 'default'}: " + " | ".join(re.search(r"k_\w+(<[^>]*>)?", x).group(0) for x in names))
    want, absent = KERNELS[flags]
    for pat in want:
        assert any(re.search(pat, x) for x in names), f"{flags}: no kernel matching {pat!r} ran"
    for pat in absent:
        hit = [x for x in names if re.search(pat, x)]
        assert not hit, f"{flags}: {pat!r} ran: {hit[:2]}"


# ------------------------------------------------------------------------------------------
# GPU: largest range length (nnz >= 2^24)
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("flags", ["", "NO_STREAM"])
def test_range_shift6_graph(dl, oracle, monkeypatch, flags):
    import os
    ops, Graph = dl
    oracle.set_num_threads(os.cpu_count() or 1)
    monkeypatch.setenv("DL_FLAGS", flags)
    src, dst, n, rowptr, col, cases = hard_case("shift6")
    K, d = 8, 16
    rng = np.random.default_rng(6)
    Z = (rng.standard_normal((n, K, d), dtype=np.float32) * np.float32(0.8 / np.sqrt(np.sqrt(d))))
    G = rng.standard_normal((n, K, d), dtype=np.float32)
    pu = np.concatenate([rng.integers(0, n, 400000), np.full(3000, int(cases["hubs"][0]))])
    pv = rng.integers(0, n, pu.size)
    res, g = run_all(ops, Graph, oracle, src, dst, n, Z, BETA, TEMP, pu, pv, Gin=G)
    assert g.nnz >= 2 ** 24
    pg, po = res.pop("prob")
    lg, lo = res["logit"]
    assert np.abs(pg - po).max() <= 0.25 * np.abs(lg.astype(np.float64) - lo).max() + 2e-7
    res["prob"] = (po, po)
    from test_gpu_parity import assert_matches_oracle
    assert_matches_oracle(res, tol=1e-5)
    # float64 on sampled rows: boundary rows, hub rows and 10k random ones
    sel = np.concatenate([cases[k][:64] for k in ("start", "end", "span3", "empty", "cross")] +
                         [cases["hubs"], rng.integers(0, n, 10000), [n - 1]])
    rows_sel, ref = ref64_rows(rowptr, col, Z, res["kstar"][1], BETA, TEMP, G, sel)
    out = {k: res[k][0][rows_sel] for k in ("s", "H", "r")}
    check_outputs(f"shift6 K={K} d={d} flags={flags or 'default'} (sampled rows)", out, ref, names=("s", "H", "r"))


# ------------------------------------------------------------------------------------------
# GPU: one rank of the node-partitioned step
# ------------------------------------------------------------------------------------------
SENTINEL = -7.25e30


@pytest.mark.gpu
@pytest.mark.parametrize("flags", ["", "NO_STREAM"])
@pytest.mark.parametrize("agg", ["zs", "sj"])
@pytest.mark.parametrize("world,rank", [(2, 0), (2, 1), (8, 0), (8, 4), (8, 7)])
def test_partitioned_rank_on_one_gpu(dl, oracle, monkeypatch, world, rank, agg, flags):
    from disenlink_b200.partition import CudaBackend, NodePartition, pair_shard
    ops, Graph = dl
    monkeypatch.setenv("DL_FLAGS", flags)
    K, d = 8, 16
    src, dst, n, rowptr, col, cases = hard_case("shift0")
    c = shape_case("shift0", K, d)
    dev = torch.device("cuda:0")
    f32 = dict(dtype=torch.float32, device=dev)

    # checked single-GPU full-graph run: its halo rows are what the pushes would deliver
    full = gpu_run(ops, Graph, src, dst, n, c)
    check_case(f"partition full-graph flags={flags or 'default'}", full, c)
    dHp_full = full["dHp"]
    ref = Ref64(rowptr, col, c["Z"], c["o_k"], BETA, TEMP)
    rb = ref.factor_bwd(dHp_full)                    # factor backward of the step: G = the decoder's dH
    ref_dZ = c["ref"]["dZp"] + rb["dZ"]
    del ref

    src_t, dst_t = t(src), t(dst)
    part = NodePartition.nnz_balanced(src_t, dst_t, n, world, rank)
    lo, hi = part.lo, part.hi
    assert hi > lo
    be = CudaBackend()
    u, v = t(c["pu"]), t(c["pv"])
    P = int(u.numel())
    p_per, p_lo, p_hi = pair_shard(P, world, rank)
    rowptr_l, col_g = be.build_csr(src_t, dst_t, part)
    inc_ptr, inc_other_g, inc_pair = be.build_incidence(u, v, part)
    su, sv = u[p_lo:p_hi].to(torch.int64), v[p_lo:p_hi].to(torch.int64)

    def remote(x):
        x = x.to(torch.int64)
        return x[(x < lo) | (x >= hi)]
    # PartitionedLinkStep.__init__ / HaloPlan.to_local without the process group
    halo_pair = torch.unique(torch.cat([remote(su), remote(sv), remote(inc_other_g)]))
    halo = torch.unique(torch.cat([remote(col_g), halo_pair]))
    n_own, n_halo = hi - lo, int(halo.numel())
    n_tot = n_own + n_halo
    assert n_halo > 0

    def to_local(ids):
        own = (ids >= lo) & (ids < hi)
        pos = torch.searchsorted(halo, ids).clamp_(max=n_halo - 1)
        return torch.where(own, ids - lo, pos + n_own)
    g = be.make_graph(rowptr_l, to_local(col_g.to(torch.int64)).to(torch.int32), n_own, n_tot)
    shard = be.make_pairs(to_local(su), to_local(sv), n_tot)
    inc = be.make_graph(inc_ptr, to_local(inc_other_g.to(torch.int64)).to(torch.int32), n_own, n_tot)
    gid = torch.cat([torch.arange(lo, hi, device=dev), halo])          # global id of every local row
    # the rank's CSR is the owned block of the full one, columns mapped to local ids
    assert np.array_equal(rowptr_l.cpu().numpy(), rowptr[lo:hi + 1] - rowptr[lo])
    assert np.array_equal(col_g.cpu().numpy(), col[rowptr[lo]:rowptr[hi]])

    def full_rows(a):
        return torch.as_tensor(a, device=dev)[gid]
    Z = full_rows(c["Z"]).contiguous()
    nnz = g.nnz
    kstar = torch.empty(max(nnz, 1), dtype=torch.uint8, device=dev)
    w = torch.empty(max(nnz, 1), **f32)
    s = torch.full((n_tot, K), SENTINEL, **f32)
    H = torch.full((n_tot, K, d), SENTINEL, **f32)
    dZ = torch.full((n_tot, K, d), SENTINEL, **f32)
    dH = torch.full((n_tot, K, d), SENTINEL, **f32)
    r = torch.full((n_tot, K), SENTINEL, **f32)
    untouched = lambda x: bool((x[n_own:] == SENTINEL).all())
    e0, e1 = rowptr[lo], rowptr[hi]

    # forward
    be.edge_attn_fwd(g, Z, TEMP, kstar, w, s)
    assert untouched(s)
    assert np.array_equal(kstar[:nnz].cpu().numpy(), c["o_k"][e0:e1])
    assert np.array_equal(w[:nnz].cpu().numpy().view(np.uint32), c["o_w"][e0:e1].view(np.uint32))
    s[n_own:] = full_rows(full["s"])[n_own:]                     # the push of s after the attention
    sj = torch.full((max(nnz, 1),), float("nan"), **f32) if agg == "sj" else None
    zs = torch.empty(n_tot, K, d, **f32) if agg == "zs" else None
    be.factor_spmm_fwd(g, Z, kstar, w, s, BETA, H, sj, zs)
    assert untouched(H)
    if sj is not None:
        assert torch.equal(sj[:nnz], s[g.col.long(), kstar[:nnz].long()])
    H[n_own:] = full_rows(full["H"])[n_own:]
    logit, _ = ops.pair_score_fwd(Z, H, shard, TEMP)
    # backward: decoder, pass 1, pass 2 (PartitionedLinkStep.backward)
    dS = t(c["dS"])
    be.pair_score_bwd(inc, inc_pair, Z, H, dS, TEMP, dZ, dH)
    assert untouched(dZ) and untouched(dH)
    dZp_own, dHp_own = dZ[:n_own].cpu().numpy(), dH[:n_own].cpu().numpy()
    dH[n_own:] = full_rows(dHp_full)[n_own:]
    plan = be.bwd_plan(g, K, d)
    be.factor_bwd_gather(g, Z, dH, kstar, w, s, BETA, dZ, r, plan=plan)
    assert untouched(dZ) and untouched(r)
    r_full = ops.factor_bwd(Graph.from_edges(src_t, dst_t, n), t(c["Z"]), t(dHp_full), t(c["o_k"]),
                            t(c["o_w"]), t(full["s"]), BETA, TEMP)[1]
    check_outputs("partition full-graph r (G = decoder dH)", dict(r=r_full.cpu().numpy()), rb, names=("r",))
    r[n_own:] = r_full[gid][n_own:]
    be.factor_bwd_edges(g, Z, dH, kstar, w, s, r, BETA, TEMP, dZ, sj, plan=plan)
    assert untouched(dZ)

    # owned rows against the float64 reference of the full graph
    own = slice(lo, hi)
    cref = c["ref"]
    p = slice(p_lo, p_hi)
    out = dict(s=s[:n_own].cpu().numpy(), H=H[:n_own].cpu().numpy(), logit=logit.cpu().numpy(),
               dZp=dZp_own, dHp=dHp_own, r=r[:n_own].cpu().numpy(), dZ=dZ[:n_own].cpu().numpy())
    rf = dict(s=cref["s"][own], A_s=cref["A_s"][own], H=cref["H"][own], A_H=cref["A_H"][own],
              logit=cref["logit"][p], A_logit=cref["A_logit"][p], dZp=cref["dZp"][own], A_dZp=cref["A_dZp"][own],
              dHp=cref["dHp"][own], A_dHp=cref["A_dHp"][own], r=rb["r"][own], A_r=rb["A_r"][own], dZ=ref_dZ[own])
    check_outputs(f"partition world={world} rank={rank} agg={agg} flags={flags or 'default'}", out, rf)
    # and against the checked full-graph run (same kernels on a different index space)
    assert relerr(out["H"], full["H"][own]) < ORA_TOL
