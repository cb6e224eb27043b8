"""CPU suite of the directed backward (graphs marked directed, any 0/1 pattern).

The float64 reference is Ref64 of test_gpu_kernel_paths.py (the hot path restated on the CSR entries, dZ from
torch.autograd, valid for any pattern) with its r replaced by the directed one: r[j,k] sums over the IN-entries
of j and is 0 where row j has no entry routed to k (the reference's clamped s = 1 passes no gradient).  Pinned
here to the dense restatement of model.py (dense_forward of test_oracle_live_reference.py, itself pinned to the
golden outputs) on random asymmetric graphs, and to a closed-form numpy statement of the gradient.
"""
from functools import lru_cache

import numpy as np
import pytest
import torch

from test_gpu_kernel_paths import BETA, DL_SEG, HUB_DEGREES, TEMP, Ref64, check_outputs, range_len, reject
from test_oracle_live_reference import dense_forward


# ------------------------------------------------------------------------------------------
# directed graphs with the hard cases
# ------------------------------------------------------------------------------------------
def csr_of(src, dst, n):
    """De-duplicated directed CSR, columns ascending in a row (Graph.from_edges(..., directed=True))."""
    key = np.unique(np.asarray(src, np.int64) * n + np.asarray(dst, np.int64))
    rows, col = key // n, key % n
    rowptr = np.zeros(n + 1, np.int64)
    rowptr[1:] = np.cumsum(np.bincount(rows, minlength=n))
    return rowptr, col.astype(np.int32)


def transpose_of(rowptr, col):
    """(trowptr, tcol, tperm) in numpy: the in-entries of every node in CSR order."""
    n = rowptr.size - 1
    tperm = np.argsort(col, kind="stable").astype(np.int32)
    rows = np.repeat(np.arange(n), np.diff(rowptr)).astype(np.int32)
    trowptr = np.zeros(n + 1, np.int64)
    trowptr[1:] = np.cumsum(np.bincount(col, minlength=n))
    return trowptr, rows[tperm], tperm


def directed_graph(n, m_rand, seed, hubs=HUB_DEGREES):
    """Directed edge list over n nodes: one-way and reciprocal edges mixed, self-loops, sinks (in-edges, no
    out-edges), sources (out-edges, no in-edges), out-hubs and in-hubs of exactly the degrees `hubs`, isolated
    nodes and an active last node."""
    rng = np.random.default_rng(seed)
    nodes = rng.permutation(np.arange(1, n - 1))
    nh = len(hubs)
    out_hubs, in_hubs = nodes[:nh], nodes[nh:2 * nh]
    sinks, sources, isolated = nodes[2 * nh:2 * nh + 20], nodes[2 * nh + 20:2 * nh + 40], nodes[2 * nh + 40:2 * nh + 45]
    special = np.concatenate([out_hubs, in_hubs, sinks, sources, isolated])
    plain = np.setdiff1d(np.arange(n), special)
    a, b = rng.choice(plain, m_rand), rng.choice(plain, m_rand)
    recip = rng.random(m_rand) < 0.3                     # 30 % of the random edges in both directions
    sa = [a, b[recip], np.repeat(out_hubs, hubs), rng.choice(plain, 3 * sinks.size), np.repeat(sources, 3)]
    sb = [b, a[recip], np.concatenate([rng.choice(plain, m, replace=False) for m in hubs]),
          np.repeat(sinks, 3), rng.choice(plain, 3 * sources.size)]
    sa.append(np.concatenate([rng.choice(plain, m, replace=False) for m in hubs]))
    sb.append(np.repeat(in_hubs, hubs))
    loops = rng.choice(plain, 40, replace=False)
    sa += [loops, [n - 1]]
    sb += [loops, [0]]
    return np.concatenate(sa).astype(np.int64), np.concatenate(sb).astype(np.int64)


def directed_cases(rowptr, col, hubs=HUB_DEGREES):
    """Asserts the structural hard cases are present; -> dict of example nodes."""
    n = rowptr.size - 1
    outdeg = np.diff(rowptr)
    indeg = np.bincount(col, minlength=n)
    rows = np.repeat(np.arange(n), outdeg)
    key = rows * n + col
    rev = np.isin(col.astype(np.int64) * n + rows, key)
    nnz = int(rowptr[-1])
    RL = range_len(nnz)
    cross = np.nonzero((outdeg > 0) & ((rowptr[1:] - 1) // RL > rowptr[:-1] // RL) & (outdeg < DL_SEG))[0]
    for m in hubs:
        assert (outdeg == m).any(), f"no out-hub of degree {m}"
        assert (indeg == m).any(), f"no in-hub of degree {m}"
    sinks = np.nonzero((outdeg == 0) & (indeg > 0))[0]
    sources = np.nonzero((outdeg > 0) & (indeg == 0))[0]
    assert sinks.size and sources.size, "no sinks / sources"
    assert (rows == col).any(), "no self-loops"
    assert (rev & (rows != col)).any() and (~rev).any(), "reciprocal and one-way edges are not both present"
    assert cross.size, "no row crosses a streaming range boundary"
    assert outdeg[-1] > 0, "last node has no entries"
    assert ((outdeg == 0) & (indeg == 0)).any(), "no isolated node"
    return dict(sinks=sinks, sources=sources, cross=cross, in_hubs=np.nonzero(indeg >= DL_SEG)[0],
                out_hubs=np.nonzero(outdeg >= DL_SEG)[0])


def routed_mask(rowptr, kstar, K):
    """has[i,k] = row i has an entry routed to k."""
    n = rowptr.size - 1
    rows = np.repeat(np.arange(n), np.diff(rowptr))
    has = np.zeros((n, K), bool)
    has[rows, kstar.astype(np.int64)] = True
    return has


def in_only_pairs(rowptr, col, kstar, K):
    """(node, factor) pairs with a routed in-entry and no routed out-entry: the clamp rule's cases."""
    has = routed_mask(rowptr, kstar, K)
    tin = np.zeros_like(has)
    tin[col.astype(np.int64), kstar.astype(np.int64)] = True
    return np.argwhere(tin & ~has)


# ------------------------------------------------------------------------------------------
# float64 references
# ------------------------------------------------------------------------------------------
class RefDir64(Ref64):
    """Ref64 on a directed pattern: w, s, H and dZ (autograd) hold for any pattern; r and its A are the
    directed ones (in-entries of j, divided by s[j]^2, 0 where row j has no entry routed to k)."""

    def factor_bwd(self, G):
        G64 = torch.from_numpy(np.ascontiguousarray(G)).double()
        (dZ,) = torch.autograd.grad(self.H, self.Z, grad_outputs=G64, retain_graph=True)
        with torch.no_grad():
            N, K = self.N, self.K
            Z, Za, Ga = self.Z.detach(), self.Z.detach().abs(), G64.abs()
            w, s, As = self.w.detach(), self.s.detach(), self.A_s
            jdx = self.cols * K + self.ks
            racc = torch.zeros(N * K, dtype=torch.float64)
            aacc = torch.zeros(N * K, dtype=torch.float64)
            sj, asj = s[self.cols, self.ks], As[self.cols, self.ks]
            for a, b in self.spans:
                r, c, k = self.rows[a:b], self.cols[a:b], self.ks[a:b]
                racc.index_add_(0, jdx[a:b], w[a:b] * (Z[c, k] * G64[r, k]).sum(-1))
                aacc.index_add_(0, jdx[a:b], (self.wa[a:b] + 2 * w[a:b] * asj[a:b] / sj[a:b] + w[a:b]) *
                                (Za[c, k] * Ga[r, k]).sum(-1))
            has = torch.zeros(N * K, dtype=torch.bool)
            has[self.rows * K + self.ks] = True
            has = has.view(N, K)
            omb = 1.0 - self.beta
            rr = torch.where(has, omb * racc.view(N, K) / s ** 2, torch.zeros_like(s))
            A_r = torch.where(has, omb * aacc.view(N, K) / s ** 2, torch.zeros_like(s))
        return dict(dZ=dZ.numpy(), r=rr.numpy(), A_r=A_r.numpy())


def closed_form(rowptr, col, Z, kstar, G, beta, T):
    """The directed backward in numpy float64, entry by entry (DESIGN.md section 1): -> (dZ, r)."""
    Z = Z.astype(np.float64)
    G = G.astype(np.float64)
    N, K, d = Z.shape
    rows = np.repeat(np.arange(N), np.diff(rowptr))
    cols = col.astype(np.int64)
    ks = kstar.astype(np.int64)
    q = (Z[rows] * Z[cols]).sum(-1) / T
    a = np.exp(q - q.max(1, keepdims=True))
    a /= a.sum(1, keepdims=True)
    w = a[np.arange(ks.size), ks]
    s = np.zeros((N, K))
    np.add.at(s, (rows, ks), w)
    has = s != 0
    s[~has] = 1.0
    omb = 1.0 - beta
    Tin = np.zeros((N, K, d))
    np.add.at(Tin, (cols, ks), (omb * w / s[cols, ks])[:, None] * G[rows, ks])
    r = np.where(has, (Z * Tin).sum(-1) / s, 0.0)
    dZ = beta * G + Tin
    c = omb * (G[rows, ks] * Z[cols, ks]).sum(-1)
    dw = c / s[cols, ks] - r[rows, ks]
    onehot = np.eye(K)[ks]
    coef = (dw * w / T)[:, None] * (onehot - a)
    np.add.at(dZ, rows, coef[:, :, None] * Z[cols])
    np.add.at(dZ, cols, coef[:, :, None] * Z[rows])
    return dZ, r


def relerr(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)) if b.size else 0.0


def route64(rowptr, col, Z, T):
    """Routing of the entries in float64 (model.py:56-61, first maximum)."""
    Z = Z.astype(np.float64)
    rows = np.repeat(np.arange(rowptr.size - 1), np.diff(rowptr))
    q = (Z[rows] * Z[col.astype(np.int64)]).sum(-1) / T
    return np.argmax(q, 1).astype(np.uint8)


def small_directed(seed, n, m, K, d):
    rng = np.random.default_rng(seed)
    src, dst = rng.integers(0, n, m), rng.integers(0, n, m)
    keep = rng.random(m) < 0.8
    src = np.concatenate([src, dst[~keep][:5], np.arange(0, n, 7)])     # a few reciprocal edges, self-loops
    dst = np.concatenate([dst, src[:m][~keep][:5], np.arange(0, n, 7)])
    rowptr, col = csr_of(src, dst, n)
    Z = (rng.standard_normal((n, K, d)) * 0.7).astype(np.float32)
    G = rng.standard_normal((n, K, d)).astype(np.float32)
    return rowptr, col, Z, G


# ------------------------------------------------------------------------------------------
# tests
# ------------------------------------------------------------------------------------------
def test_generator_produces_the_directed_cases():
    src, dst = directed_graph(6000, 20000, 3)
    rowptr, col = csr_of(src, dst, 6000)
    directed_cases(rowptr, col)


def test_numpy_transpose_is_the_in_entry_list():
    rowptr, col, _, _ = small_directed(5, 40, 150, 2, 4)
    trowptr, tcol, tperm = transpose_of(rowptr, col)
    rows = np.repeat(np.arange(40), np.diff(rowptr))
    for j in range(40):
        p = np.arange(trowptr[j], trowptr[j + 1])
        assert np.all(col[tperm[p]] == j) and np.array_equal(tcol[p], rows[tperm[p]])
        assert np.all(np.diff(tperm[p]) > 0)
    assert np.array_equal(np.sort(tperm), np.arange(col.size))


@pytest.mark.parametrize("seed,K,d", [(0, 3, 4), (1, 1, 5), (2, 4, 8), (3, 2, 3), (4, 5, 2)])
def test_refdir64_matches_dense_restatement(seed, K, d):
    """Loss, H and dL/dZ of RefDir64 (sparse, chunked, autograd) against dense_forward of model.py in float64 on a
    random asymmetric adjacency, within 1e-9; the routing is model.py's own (float64 argmax)."""
    n = 30 + 7 * seed
    rowptr, col, Z, G = small_directed(seed, n, 4 * n, K, d)
    adj = np.zeros((n, n))
    rows = np.repeat(np.arange(n), np.diff(rowptr))
    adj[rows, col] = 1
    assert not np.array_equal(adj, adj.T)
    ks = route64(rowptr, col, Z, 1.3)
    rng = np.random.default_rng(seed)
    pu, pv = rng.integers(0, n, 200), rng.integers(0, n, 200)
    y = torch.from_numpy((rng.random(200) < 0.5).astype(np.float64))
    bce = torch.nn.functional.binary_cross_entropy

    ref = RefDir64(rowptr, col, Z, ks, 0.35, 1.3, chunk=37)
    loss_s = bce(torch.sigmoid(ref.logits(torch.from_numpy(pu), torch.from_numpy(pv), ref.H)), y)
    (g_s,) = torch.autograd.grad(loss_s, ref.Z)

    Zd = torch.from_numpy(Z).double().requires_grad_(True)
    _, _, Hd, link_pred = dense_forward([Zd[:, k, :] for k in range(K)], torch.from_numpy(adj), 0.35, 1.3)
    loss_d = bce(link_pred[torch.from_numpy(pu), torch.from_numpy(pv)], y)
    (g_d,) = torch.autograd.grad(loss_d, Zd)
    assert abs(loss_s.item() - loss_d.item()) <= 1e-9 * abs(loss_d.item())
    assert relerr(ref.H.detach().numpy().reshape(n, -1), Hd.detach().numpy()) < 1e-9
    assert relerr(g_s.numpy(), g_d.numpy()) < 1e-9


@pytest.mark.parametrize("seed,K,d", [(0, 3, 4), (1, 1, 5), (2, 4, 8), (6, 6, 3)])
def test_closed_form_matches_autograd(seed, K, d):
    """The formulas the kernels implement (DESIGN.md section 1), clamp rule included, against RefDir64:
    dZ within 1e-9, r within 1e-12 and exactly 0 on the clamped (node, factor) pairs."""
    n = 40 + 5 * seed
    rowptr, col, Z, G = small_directed(seed, n, 3 * n, K, d)
    ks = route64(rowptr, col, Z, 0.8)
    clamp = in_only_pairs(rowptr, col, ks, K)
    assert clamp.size, "no (node, factor) with routed in-entries and no routed out-entry"
    if K == 1:
        outdeg = np.diff(rowptr)
        assert np.any((outdeg == 0) & (np.bincount(col, minlength=n) > 0))        # sinks: s clamped at K = 1
    ref = RefDir64(rowptr, col, Z, ks, 0.4, 0.8).factor_bwd(G)
    dZ, r = closed_form(rowptr, col, Z, ks, G, 0.4, 0.8)
    assert relerr(dZ, ref["dZ"]) < 1e-9
    assert np.allclose(r, ref["r"], rtol=1e-12, atol=1e-300)
    assert np.all(ref["r"][clamp[:, 0], clamp[:, 1]] == 0.0)
    assert not routed_mask(rowptr, ks, K)[clamp[:, 0], clamp[:, 1]].any()


def test_refdir64_equals_ref64_on_a_symmetric_pattern():
    """On a symmetric pattern the directed r is the symmetric one (the mirror turns column sums into row sums)."""
    rng = np.random.default_rng(9)
    n, K, d = 60, 3, 4
    a, b = rng.integers(0, n, 200), rng.integers(0, n, 200)
    rowptr, col = csr_of(np.concatenate([a, b]), np.concatenate([b, a]), n)
    Z = (rng.standard_normal((n, K, d)) * 0.7).astype(np.float32)
    G = rng.standard_normal((n, K, d)).astype(np.float32)
    ks = route64(rowptr, col, Z, 1.0)
    x = RefDir64(rowptr, col, Z, ks, 0.5, 1.0).factor_bwd(G)
    y = Ref64(rowptr, col, Z, ks, 0.5, 1.0).factor_bwd(G)
    assert np.allclose(x["r"], y["r"], rtol=1e-12, atol=1e-300)
    assert np.array_equal(x["dZ"], y["dZ"])


@lru_cache(maxsize=None)
def _fault_case():
    rng = np.random.default_rng(21)
    n, K, d = 3000, 4, 8
    src, dst = directed_graph(n, 12000, 21, hubs=(600, 1025))
    rowptr, col = csr_of(src, dst, n)
    Z = (rng.standard_normal((n, K, d)) * 0.5).astype(np.float32)
    G = rng.standard_normal((n, K, d)).astype(np.float32)
    ks = route64(rowptr, col, Z, TEMP)
    ref = RefDir64(rowptr, col, Z, ks, BETA, TEMP)
    res = ref.forward_dict()
    res.update(ref.factor_bwd(G))
    return rowptr, col, Z, G, ks, res


def test_checker_rejects_r_without_the_clamp_rule():
    """The per-element checker accepts the closed form rounded to fp32 and rejects r computed without the clamp
    rule (<Z[j,k], T_[j,k]> / s[j,k] on a (node, factor) that has no routed out-entry) and a lost in-entry."""
    rowptr, col, Z, G, ks, ref = _fault_case()
    K = Z.shape[1]
    dZ, r = closed_form(rowptr, col, Z, ks, G, BETA, TEMP)
    check_outputs("closed form fp32", dict(r=r.astype(np.float32), dZ=dZ.astype(np.float32)), ref, names=("r", "dZ"))
    clamp = in_only_pairs(rowptr, col, ks, K)
    assert clamp.size
    # the same sum without the rule
    N, d = Z.shape[0], Z.shape[2]
    Z64, G64 = Z.astype(np.float64), G.astype(np.float64)
    rows = np.repeat(np.arange(N), np.diff(rowptr))
    cols, k64 = col.astype(np.int64), ks.astype(np.int64)
    s = ref["s"]
    w = np.exp((Z64[rows] * Z64[cols]).sum(-1) / TEMP)
    w = w[np.arange(k64.size), k64] / w.sum(1)
    Tin = np.zeros((N, K, d))
    np.add.at(Tin, (cols, k64), ((1 - BETA) * w / s[cols, k64])[:, None] * G64[rows, k64])
    r_noclamp = ((Z64 * Tin).sum(-1) / s).astype(np.float32)
    assert np.allclose(r_noclamp[~np.isin(np.arange(N), clamp[:, 0])], r[~np.isin(np.arange(N), clamp[:, 0])],
                       rtol=1e-5, atol=1e-6)
    assert reject(dict(r=r_noclamp), ref, "r")
    # one in-entry of an in-hub lost from T_ (dZ and r of that node)
    indeg = np.bincount(cols, minlength=N)
    hub = int(np.argmax(indeg))
    e = int(np.nonzero(cols == hub)[0][indeg[hub] // 2])
    k = int(k64[e])
    lost = (1 - BETA) * w[e] / s[hub, k] * G64[rows[e], k]
    dZ_bad = dZ.copy()
    dZ_bad[hub, k] -= lost
    assert reject(dict(dZ=dZ_bad), ref, "dZ")
