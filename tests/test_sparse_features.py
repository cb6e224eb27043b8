"""CPU-side checks of the SparseFeatures handle (disenlink_b200/features.py): its CSR and CSC against scipy's, the
heavy-column chunk plan of the weight gradient, the refusal of CPU tensors by the kernels' entry point, and
examples/train_link.py's --sparse-features flag."""
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from conftest import ROOT
from disenlink_b200 import features
from disenlink_b200.features import SparseFeatures


def _coo(N, F, nnz, seed, dup=0, zeros=0, empty_rows=(), empty_cols=()):
    """Random COO entries with duplicates (to be summed) and explicit zeros (to be dropped)."""
    rng = np.random.default_rng(seed)
    r = rng.integers(0, N, nnz)
    c = rng.integers(0, F, nnz)
    # multiples of 1/8: duplicate sums are exact in any order (and some cancel to an explicit zero)
    v = (rng.integers(1, 9, nnz) * rng.choice([-1, 1], nnz) / 8).astype(np.float32)
    if dup:
        r, c, v = np.concatenate([r, r[:dup]]), np.concatenate([c, c[:dup]]), np.concatenate([v, -v[:dup // 2], v[dup // 2:dup]])
    if zeros:
        r = np.concatenate([r, rng.integers(0, N, zeros)])
        c = np.concatenate([c, rng.integers(0, F, zeros)])
        v = np.concatenate([v, np.zeros(zeros, np.float32)])
    keep = ~np.isin(r, list(empty_rows)) & ~np.isin(c, list(empty_cols))
    return r[keep], c[keep], v[keep]


CASES = {
    "plain": dict(N=50, F=40, nnz=300, seed=0),
    "dup_and_zeros": dict(N=60, F=30, nnz=400, seed=1, dup=80, zeros=50),
    "empty_rows_cols": dict(N=70, F=90, nnz=500, seed=2, dup=10, zeros=10, empty_rows=(0, 5, 69), empty_cols=(0, 1, 89)),
    "one_row": dict(N=1, F=20, nnz=12, seed=3, dup=3),
    "empty": dict(N=8, F=6, nnz=0, seed=4),
}


def _scipy(N, F, r, c, v):
    m = sp.coo_matrix((v, (r, c)), shape=(N, F)).tocsr()
    m.sum_duplicates()
    m.eliminate_zeros()
    m.sort_indices()
    return m, m.tocsc()


def _check_against_scipy(h: SparseFeatures, N, F, r, c, v):
    csr, csc = _scipy(N, F, r, c, v)
    csc.sort_indices()
    assert (h.N, h.F, h.nnz) == (N, F, csr.nnz) and h.shape == (N, F)
    assert np.array_equal(h.rowptr.numpy(), csr.indptr) and np.array_equal(h.col.numpy(), csr.indices)
    assert np.array_equal(h.val.numpy(), csr.data)
    assert np.array_equal(h.colptr.numpy(), csc.indptr) and np.array_equal(h.row.numpy(), csc.indices)
    assert np.array_equal(h.cval.numpy(), csc.data)
    assert h.col.dtype == h.row.dtype == torch.int32 and h.rowptr.dtype == h.colptr.dtype == torch.int64
    assert h.val.dtype == h.cval.dtype == torch.float32
    assert torch.equal(h.to_dense(), torch.as_tensor(csr.toarray()))


@pytest.mark.parametrize("case", list(CASES))
def test_from_sparse_equals_scipy(case):
    kw = CASES[case]
    N, F = kw["N"], kw["F"]
    r, c, v = _coo(**kw)
    x = torch.sparse_coo_tensor(torch.as_tensor(np.stack([r, c])), torch.as_tensor(v), (N, F))  # uncoalesced
    _check_against_scipy(SparseFeatures.from_sparse(x), N, F, r, c, v)
    _check_against_scipy(SparseFeatures.from_sparse(x.coalesce().to_sparse_csr()), N, F, r, c, v)


@pytest.mark.parametrize("case", list(CASES))
def test_from_dense_equals_scipy(case):
    kw = CASES[case]
    N, F = kw["N"], kw["F"]
    r, c, v = _coo(**kw)
    dense, _ = _scipy(N, F, r, c, v)
    x = torch.as_tensor(dense.toarray())
    _check_against_scipy(SparseFeatures.from_dense(x), N, F, r, c, v)


def _check_plan(h: SparseFeatures):
    """Heavy chunks first (slot = item index), then one item per other column; together every CSC entry once."""
    colptr = h.colptr.tolist()
    lens = [colptr[f + 1] - colptr[f] for f in range(h.F)]
    heavy = [f for f in range(h.F) if lens[f] > features.FEAT_CHUNK]
    assert h.heavy_col.tolist() == heavy and h.n_heavy == len(heavy)
    cols, lo, hi = h.item_col.tolist(), h.item_lo.tolist(), h.item_hi.tolist()
    assert len(cols) == len(lo) == len(hi) == h.n_items == h.F + h.n_slots - h.n_heavy
    hp = h.heavy_ptr.tolist()
    assert hp[0] == 0 and hp[-1] == h.n_slots
    for k, f in enumerate(heavy):                       # the chunks of heavy column f: contiguous, in order
        items = list(range(hp[k], hp[k + 1]))
        assert all(cols[t] == f for t in items)
        assert lo[items[0]] == colptr[f] and hi[items[-1]] == colptr[f + 1]
        assert all(hi[t] == lo[t + 1] for t in items[:-1])
        assert all(0 < hi[t] - lo[t] <= features.FEAT_CHUNK for t in items)
        assert all(hi[t] - lo[t] == features.FEAT_CHUNK for t in items[:-1])
    light = [f for f in range(h.F) if f not in set(heavy)]
    assert cols[h.n_slots:] == light
    assert all(lo[h.n_slots + i] == colptr[f] and hi[h.n_slots + i] == colptr[f + 1] for i, f in enumerate(light))
    covered = np.zeros(h.nnz, np.int64)
    for a, b in zip(lo, hi):
        covered[a:b] += 1
    assert np.all(covered == 1)


@pytest.mark.parametrize("case", list(CASES))
def test_chunk_plan_covers_every_entry_once(case):
    kw = CASES[case]
    r, c, v = _coo(**kw)
    x = torch.sparse_coo_tensor(torch.as_tensor(np.stack([r, c])), torch.as_tensor(v), (kw["N"], kw["F"]))
    _check_plan(SparseFeatures.from_sparse(x))


def test_chunk_plan_of_heavy_columns():
    """Columns of FEAT_CHUNK - 1 .. 3 FEAT_CHUNK + 1 entries, one in every row, next to light and empty ones."""
    C = features.FEAT_CHUNK
    N = 3 * C + 1
    x = torch.zeros(N, 8)
    for f, n in enumerate([N, 0, C, C + 1, 2 * C, 5, 2 * C + 7, C - 1]):
        x[torch.randperm(N, generator=torch.Generator().manual_seed(f))[:n], f] = f + 1.0
    h = SparseFeatures.from_dense(x)
    _check_plan(h)
    assert h.heavy_col.tolist() == [0, 3, 4, 6]
    assert h.heavy_ptr.tolist() == [0, 4, 6, 8, 11]


def test_bad_inputs_are_refused():
    with pytest.raises(ValueError):
        SparseFeatures.from_dense(torch.zeros(3, 4).to_sparse())
    with pytest.raises(ValueError):
        SparseFeatures.from_sparse(torch.zeros(3, 4))
    with pytest.raises(ValueError):
        SparseFeatures(torch.tensor([0, 3]), torch.tensor([0, 1]), torch.tensor([1.0, 2.0]), 3, 4)


def test_projection_refuses_cpu_tensors():
    from disenlink_b200 import ops
    h = SparseFeatures.from_dense(torch.eye(4))
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.feature_projection(h, torch.zeros(4, 8), torch.zeros(8), relu=True)


def test_train_link_parses_sparse_features():
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    import train_link
    assert train_link.parse_args(["--sparse-features"]).sparse_features is True
    assert train_link.parse_args([]).sparse_features is False
    a = train_link.parse_args(["--sparse-features", "--run", "3", "--capture", "10"])
    assert (a.sparse_features, a.run, a.capture) == (True, 3, 10)
