"""Sparse input features as a handle built once per dataset, for the first layer of the factor MLPs.

The Planetoid sets (Cora, Citeseer, Pubmed) are fed to the model as raw bag-of-words rows
(main_disentangled.py:117-123): Cora's x is 1.3 % dense.  ``SparseFeatures`` holds such an x as CSR (rows, for
the forward), as CSC (columns, for the weight gradient) and the chunk plan of the CSC columns, so that
``Disentangle.project`` / ``DisentangleRuns.project`` compute the first layer over the nonzeros only
(ops.feature_projection, csrc/feat_proj.cu) -- in eager steps, in the runs union and in captured epochs.

    feats = SparseFeatures.from_dense(x)          # or .from_sparse(x) for a torch COO / CSR tensor
    Z = model.project(feats)

Duplicate COO entries are summed and explicit zeros dropped.  The index structures are built with torch integer
ops on the tensor's own device (CPU tensors too); the kernels run on CUDA only.
"""
from __future__ import annotations

import torch

# CSC entries per chunk of a heavy column (word frequencies are Zipf-like: a few columns hold a large share of
# the rows).  Fixed, independent of the width J of the layer, so that a run's block of a union's weight gradient
# is summed exactly as that run's gradient alone.
FEAT_CHUNK = 256


class SparseFeatures:
    """x [N, F] as CSR, CSC and the weight gradient's chunk plan (see include/disenlink_b200.h, dl_feat_proj_bwd).

      rowptr int64 [N+1], col int32 [nnz], val float32 [nnz]        CSR, columns ascending inside a row
      colptr int64 [F+1], row int32 [nnz], cval float32 [nnz]       CSC, rows ascending inside a column
      item_col int32, item_lo / item_hi int64 [n_items]             CSC entries [lo, hi) of column item_col:
                                                                    the chunks of the heavy columns first
                                                                    (n_slots items), then one item per other column
      heavy_col int32 [n_heavy], heavy_ptr int64 [n_heavy+1]        the heavy columns and their item ranges
    """

    def __init__(self, rows: torch.Tensor, cols: torch.Tensor, vals: torch.Tensor, n_rows: int, n_cols: int):
        """Entries (rows, cols, vals) without duplicates; explicit zeros are dropped here."""
        N, F = int(n_rows), int(n_cols)
        if N < 0 or F < 0:
            raise ValueError(f"bad feature shape [{N}, {F}]")
        if N >= 2**31 or F >= 2**31:
            raise ValueError("N and F must stay below 2^31 (int32 indices)")
        keep = vals != 0
        r, c, v = rows[keep].to(torch.int64), cols[keep].to(torch.int64), vals[keep].to(torch.float32)
        if r.numel() and (int(r.min()) < 0 or int(r.max()) >= N or int(c.min()) < 0 or int(c.max()) >= F):
            raise ValueError(f"feature entry outside [{N}, {F}]")
        dev = v.device
        self.N, self.F, self.nnz = N, F, int(v.numel())
        o = torch.argsort(r * F + c)
        self.rowptr = _ptr(r, N, dev)
        self.col, self.val = c[o].to(torch.int32).contiguous(), v[o].contiguous()
        o = torch.argsort(c * N + r)
        self.colptr = _ptr(c, F, dev)
        self.row, self.cval = r[o].to(torch.int32).contiguous(), v[o].contiguous()
        self._plan(dev)

    def _plan(self, dev) -> None:
        lo, hi = self.colptr[:-1], self.colptr[1:]
        n_chunks = torch.clamp((hi - lo + FEAT_CHUNK - 1) // FEAT_CHUNK, min=1)
        heavy = n_chunks > 1
        hcol = torch.nonzero(heavy).flatten()
        hn = n_chunks[hcol]
        self.heavy_ptr = torch.zeros(hcol.numel() + 1, dtype=torch.int64, device=dev)
        self.heavy_ptr[1:] = torch.cumsum(hn, 0)
        self.n_heavy, self.n_slots = int(hcol.numel()), int(hn.sum())
        icol = torch.repeat_interleave(hcol, hn)
        chunk = torch.arange(self.n_slots, dtype=torch.int64, device=dev) - torch.repeat_interleave(self.heavy_ptr[:-1], hn)
        ilo = lo[icol] + chunk * FEAT_CHUNK
        ihi = torch.minimum(ilo + FEAT_CHUNK, hi[icol])
        lcol = torch.nonzero(~heavy).flatten()
        self.heavy_col = hcol.to(torch.int32)
        self.item_col = torch.cat([icol, lcol]).to(torch.int32)
        self.item_lo = torch.cat([ilo, lo[lcol]]).contiguous()
        self.item_hi = torch.cat([ihi, hi[lcol]]).contiguous()
        self.n_items = int(self.item_col.numel())

    @classmethod
    def from_sparse(cls, x: torch.Tensor) -> "SparseFeatures":
        """From a torch sparse COO or CSR tensor [N, F] (``read_planetoid(..., sparse_x=True)`` gives COO)."""
        if x.dim() != 2 or x.layout not in (torch.sparse_coo, torch.sparse_csr):
            raise ValueError("from_sparse takes a 2-D sparse COO or CSR tensor; use from_dense for a strided one")
        coo = (x.to_sparse_coo() if x.layout != torch.sparse_coo else x).coalesce()    # duplicates summed
        idx = coo.indices()
        return cls(idx[0], idx[1], coo.values(), x.shape[0], x.shape[1])

    @classmethod
    def from_dense(cls, x: torch.Tensor) -> "SparseFeatures":
        """From a strided [N, F] tensor (after the dataset's own preprocessing)."""
        if x.dim() != 2 or x.layout != torch.strided:
            raise ValueError("from_dense takes a 2-D strided tensor")
        r, c = torch.nonzero(x, as_tuple=True)
        return cls(r, c, x[r, c], x.shape[0], x.shape[1])

    @property
    def device(self) -> torch.device:
        return self.val.device

    @property
    def is_cuda(self) -> bool:
        return self.val.is_cuda

    @property
    def shape(self):
        return (self.N, self.F)

    def to_dense(self) -> torch.Tensor:
        """x [N, F] as a strided float32 tensor (tests, benchmarks)."""
        out = torch.zeros(self.N, self.F, dtype=torch.float32, device=self.device)
        rows = torch.repeat_interleave(torch.arange(self.N, device=self.device), self.rowptr[1:] - self.rowptr[:-1])
        out[rows, self.col.long()] = self.val
        return out


def _ptr(keys: torch.Tensor, n: int, dev) -> torch.Tensor:
    out = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    out[1:] = torch.cumsum(torch.bincount(keys, minlength=n), 0)
    return out
