"""Device-resident graph handle: CSR of adj_sym plus the degree-bucketed work items.

Replaces the dense [N,N] adjacency the reference builds once per run
(main_disentangled.py:137-142) and multiplies into the routing matrix every epoch (model.py:62).
The adjacency is constant across epochs, so the handle is built once and cached by the module.
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib
from ._lib import DlGraph, check, lib, ptr, require_cuda, stream_of


def _ws(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=device)


class Graph:
    """CSR (rowptr int64 [N+1], col int32 [nnz]) + degree buckets + hub work items, on one GPU.

    Rows are the destination nodes; ``col`` is ascending inside a row, so the entry order equals
    ``adj_sym.nonzero()``.  ``perm`` lists rows by degree class (bit length of the degree)
    descending; rows with degree >= 512 are "hub rows" and are cut into 512-edge segments so no
    warp owns more than one segment.

    ``directed`` marks a pattern that is used as given, not as an undirected graph: its backward runs
    over the pattern and its transpose (transpose_view) and accepts any 0/1 adjacency, symmetric or not.
    An unmarked graph needs a symmetric pattern for the backward (DL_EASYM otherwise).
    """

    # below this many entries the attention runs two-sided: the graph fits L2 and the extra launches
    # of the symmetric path cost more than the row gathers it saves
    SYM_MIN_NNZ = 1 << 20

    def __init__(self, rowptr: torch.Tensor, col: torch.Tensor, n_nodes: int, row_base: int = 0,
                 n_global: int = None, directed: bool = False):
        require_cuda(rowptr, "rowptr")
        assert rowptr.dtype == torch.int64 and col.dtype == torch.int32
        self.device = rowptr.device
        self.N = int(n_nodes)                 # rows held here
        self.row_base = int(row_base)         # global id of local row 0 (node-partitioned runs)
        self.n_global = int(n_global) if n_global is not None else self.N
        self.rowptr = rowptr.contiguous()
        self.col = col.contiguous()
        self.nnz = int(col.numel())
        self._rev = None
        self._sym = None                      # (upper Graph, eidx) | False (pattern not symmetric / unavailable)
        self._sym_lower = None
        self._transpose = None                # (transposed Graph, tperm int32 [nnz])
        self.directed = bool(directed)
        self.sym_min_nnz = self.SYM_MIN_NNZ
        self._flags = _lib.default_flags()
        self._build_items()

    # ------------------------------------------------------------------ constructors
    @classmethod
    def from_edges(cls, src: torch.Tensor, dst: torch.Tensor, n_nodes: int, symmetrize: bool = None,
                   directed: bool = False) -> "Graph":
        """Symmetrise + de-duplicate directed edge columns (self-loops kept).
        ``symmetrize=False`` keeps the directed columns as they are (de-duplicated) -- the edge set
        structured negative sampling tests membership against.  ``directed=True`` marks the graph
        directed (see the class doc) and keeps the columns as given unless ``symmetrize=True``.

        [ref: main_disentangled.py:137-142]"""
        require_cuda(src, "src")
        dev = src.device
        src = src.to(torch.int64).contiguous()
        dst = dst.to(torch.int64).contiguous()
        E = int(src.numel())
        N = int(n_nodes)
        if symmetrize is None:
            symmetrize = not directed
        L = lib()
        with torch.cuda.device(dev):
            rowptr = torch.empty(N + 1, dtype=torch.int64, device=dev)
            col = torch.empty(max(2 * E, 1), dtype=torch.int32, device=dev)
            meta = torch.zeros(2, dtype=torch.int64, device=dev)  # [nnz, status(int32 in low word)]
            ws_bytes = L.dl_csr_build_workspace_bytes(E, N)
            ws = _ws(ws_bytes, dev)
            if symmetrize:
                check(L.dl_csr_build(ptr(src), ptr(dst), E, N, ptr(rowptr), ptr(col), ptr(meta),
                                     meta[1:].data_ptr(), ptr(ws), ws_bytes, stream_of(dev)),
                      "dl_csr_build")
            else:
                check(L.dl_csr_build_rect(ptr(src), ptr(dst), E, N, N, 0, ptr(rowptr), ptr(col), ptr(meta),
                                          meta[1:].data_ptr(), ptr(ws), ws_bytes, stream_of(dev)),
                      "dl_csr_build_rect")
            nnz, status = (int(x) for x in meta.cpu())
            status = ctypes.c_int32(status & 0xFFFFFFFF).value
            if status != 0:
                raise _lib.DlError(status, "dl_csr_build")
            del ws
            col = col[:nnz].clone() if nnz < col.numel() else col
        return cls(rowptr, col, N, directed=directed)

    @classmethod
    def from_edge_index(cls, edge_index: torch.Tensor, n_nodes: int, directed: bool = False) -> "Graph":
        """Symmetrised, or with ``directed=True`` the columns as given (de-duplicated), marked directed."""
        return cls.from_edges(edge_index[0], edge_index[1], n_nodes, directed=directed)

    @classmethod
    def from_dense(cls, adj: torch.Tensor, directed: bool = False) -> "Graph":
        """From the dense adjacency the reference passes to ``Disentangle.forward`` (used as is,
        any non-zero entry is an edge).  [ref: model.py:62]"""
        require_cuda(adj, "adj")
        if adj.dim() != 2 or adj.shape[0] != adj.shape[1]:
            raise ValueError("adj must be a square [N,N] matrix")
        dev = adj.device
        a = adj.to(torch.float32).contiguous()
        N = int(a.shape[0])
        L = lib()
        with torch.cuda.device(dev):
            rowptr = torch.empty(N + 1, dtype=torch.int64, device=dev)
            ws = _ws((N + 1) * 8 + (1 << 20), dev)
            check(L.dl_csr_from_dense(ptr(a), N, ptr(rowptr), None, ptr(ws), ws.numel(),
                                      stream_of(dev)), "dl_csr_from_dense(count)")
            nnz = int(rowptr[-1].item())
            col = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
            check(L.dl_csr_from_dense(ptr(a), N, ptr(rowptr), ptr(col), None, 0, stream_of(dev)),
                  "dl_csr_from_dense(fill)")
        return cls(rowptr, col[:nnz], N, directed=directed)

    @classmethod
    def from_csr(cls, rowptr: torch.Tensor, col: torch.Tensor, directed: bool = False) -> "Graph":
        return cls(rowptr.to(torch.int64), col.to(torch.int32), int(rowptr.numel()) - 1, directed=directed)

    # ------------------------------------------------------------------ integer kernels
    def _build_items(self) -> None:
        L = lib()
        dev, N = self.device, self.N
        with torch.cuda.device(dev):
            self.perm = torch.empty(max(N, 1), dtype=torch.int32, device=dev)
            self.bucket_off = torch.zeros(_lib.DL_N_BUCKETS + 1, dtype=torch.int64, device=dev)
            ws_bytes = L.dl_degree_buckets_workspace_bytes(N)
            ws = _ws(ws_bytes, dev)
            check(L.dl_degree_buckets(ptr(self.rowptr), N, ptr(self.perm), ptr(self.bucket_off),
                                      ptr(ws), ws_bytes, stream_of(dev)), "dl_degree_buckets")
            self.bucket_off_host = self.bucket_off.cpu()
            self.n_hub = int(self.bucket_off_host[_lib.DL_HUB_BUCKET_END])
            self.hub_seg_ptr = torch.zeros(self.n_hub + 1, dtype=torch.int64, device=dev)
            self.n_hub_items = 0
            self.item_hub = torch.empty(1, dtype=torch.int32, device=dev)
            if self.n_hub > 0:
                check(L.dl_hub_items(ptr(self.rowptr), ptr(self.perm), self.n_hub,
                                     ptr(self.hub_seg_ptr), None, 0, stream_of(dev)),
                      "dl_hub_items(scan)")
                self.n_hub_items = int(self.hub_seg_ptr[-1].item())
                self.item_hub = torch.empty(max(self.n_hub_items, 1), dtype=torch.int32, device=dev)
                check(L.dl_hub_items(ptr(self.rowptr), ptr(self.perm), self.n_hub,
                                     ptr(self.hub_seg_ptr), ptr(self.item_hub), self.n_hub_items,
                                     stream_of(dev)), "dl_hub_items(fill)")
            # COO row array for the streaming kernels (4 bytes per entry)
            self.erow = torch.empty(max(self.nnz, 1), dtype=torch.int32, device=dev)
            check(L.dl_entry_rows(ptr(self.rowptr), N, self.nnz, ptr(self.erow), stream_of(dev)),
                  "dl_entry_rows")
        self.struct = DlGraph(self.N, self.nnz, ptr(self.rowptr), ptr(self.col), ptr(self.perm),
                              self.n_hub, self.n_hub_items, ptr(self.hub_seg_ptr),
                              ptr(self.item_hub), ptr(self.erow), self.row_base, self._flags)
        self._hub_ws = None

    @property
    def ref(self):
        return ctypes.byref(self.struct)

    @property
    def flags(self) -> int:
        """dl_graph.flags: kernel-path switches (_lib.DL_F_*), 0 = the fast paths.  The primary / secondary
        views of sym_view() are graphs of their own and keep the flags they were built with (DL_FLAGS at
        construction); a handle, its scratch buffers and its views serve one stream at a time."""
        return self._flags

    @flags.setter
    def flags(self, value: int) -> None:
        self._flags = int(value)
        self.struct.flags = self._flags

    def hub_scratch(self, width: int):
        """fp32 scratch for hub-row partials of `width` floats per segment (None if no hubs)."""
        need = int(lib().dl_hub_scratch_floats(self.ref, int(width)))
        # the symmetric kernels run on the primary / secondary views with this scratch; a view has fewer entries
        # but may be cut into shorter ranges (dl_range_shift), i.e. into more of them
        if self._sym:
            need = max(need, int(lib().dl_hub_scratch_floats(self._sym[0].ref, int(width))))
        if self._sym_lower:
            need = max(need, int(lib().dl_hub_scratch_floats(self._sym_lower[0].ref, int(width))))
        if need == 0:
            return None
        if self._hub_ws is None or self._hub_ws.numel() < need:
            self._hub_ws = torch.empty(need, dtype=torch.float32, device=self.device)
        return self._hub_ws

    def rev_index(self) -> torch.Tensor:
        """rev[e] = position of the mirrored entry; raises if the pattern is not symmetric."""
        if self._rev is None:
            dev = self.device
            with torch.cuda.device(dev):
                rev = torch.empty(max(self.nnz, 1), dtype=torch.int64, device=dev)
                status = torch.zeros(1, dtype=torch.int32, device=dev)
                check(lib().dl_rev_index(ptr(self.rowptr), ptr(self.col), self.N, self.nnz, ptr(rev),
                                         ptr(status), stream_of(dev)), "dl_rev_index")
                code = int(status.item())
            if code != 0:
                raise _lib.DlError(code, "dl_rev_index")
            self._rev = rev[:self.nnz]
        return self._rev

    def assert_symmetric(self) -> None:
        """Raises DlError(DL_EASYM) unless every entry (i,j) has its mirror (j,i); checked once."""
        if self._sym is None and self._rev is None:
            if self.row_base == 0 and self.n_global == self.N and self.nnz < 2**31 - 1:
                self.sym_view()
            else:
                self.rev_index()
        if self._sym is False and self._rev is None:
            self.rev_index()                   # raises with the library's message

    def sym_view(self):
        """-> (primary-view Graph, eidx int32 [nnz]) for the symmetric attention (dl_edge_attn_fwd_sym), or
        None when the pattern is not symmetric, the graph is row-partitioned or has >= 2^31 entries.  Of the
        two entries of an undirected edge the primary one is the entry whose row has the larger degree (ties:
        smaller id); eidx[e] = its position in the primary view, or ~(its mirror's position) for a secondary
        entry.  Integer work on the device, done once and cached."""
        if self._sym is None:
            self._sym = False
            if self.row_base == 0 and self.n_global == self.N and 0 < self.nnz < 2**31 - 1:
                L, dev, N = lib(), self.device, self.N
                with torch.cuda.device(dev):
                    ws_bytes = L.dl_sym_index_workspace_bytes(N, self.nnz)
                    ws = _ws(ws_bytes, dev)
                    uptr = torch.empty(N + 1, dtype=torch.int64, device=dev)
                    status = torch.zeros(1, dtype=torch.int32, device=dev)
                    check(L.dl_sym_index(ptr(self.rowptr), ptr(self.col), ptr(self.erow), N, self.nnz, ptr(uptr),
                                         None, None, None, None, None, ptr(ws), ws_bytes, stream_of(dev)),
                          "dl_sym_index(count)")
                    nnz_u = int(uptr[-1].item())
                    nnz_l = self.nnz - nnz_u
                    ucol = torch.empty(max(nnz_u, 1), dtype=torch.int32, device=dev)
                    eidx = torch.empty(self.nnz, dtype=torch.int32, device=dev)
                    lcol = torch.empty(max(nnz_l, 1), dtype=torch.int32, device=dev)
                    lmirror = torch.empty(max(nnz_l, 1), dtype=torch.int32, device=dev)
                    check(L.dl_sym_index(ptr(self.rowptr), ptr(self.col), ptr(self.erow), N, self.nnz, ptr(uptr),
                                         ptr(ucol), ptr(eidx), ptr(lcol), ptr(lmirror), ptr(status), ptr(ws), ws_bytes,
                                         stream_of(dev)), "dl_sym_index(fill)")
                    ok = int(status.item()) == 0
                    del ws
                if ok:
                    upper = Graph(uptr, ucol[:nnz_u], N)
                    upper._sym = False
                    lower = Graph(self.rowptr - uptr, lcol[:nnz_l], N)        # strictly-lower entries, same row order
                    lower._sym = False
                    self._sym = (upper, eidx)
                    self._sym_lower = (lower, lmirror[:nnz_l])
        return self._sym or None

    def sym_lower_view(self):
        """-> (strictly-lower-triangle Graph, lmirror int32 [nnz_l] = upper-view position of every lower entry's
        mirror) for the symmetric backward pass 2, or None (see sym_view)."""
        return self._sym_lower if self.sym_view() is not None else None

    def transpose_view(self):
        """-> (transposed Graph, tperm int32 [nnz]): row j of the transposed graph lists the in-entries of
        node j (their source rows, in CSR order) and tperm[p] is the CSR index of in-entry p.  A graph of its
        own, so in-hubs get degree buckets and hub work items; the directed backward gathers over it.  Needs
        row_base == 0 (one GPU) and nnz < 2^31 - 1.  Integer work on the device, done once and cached."""
        if self._transpose is None:
            if self.row_base != 0 or self.n_global != self.N or self.nnz >= 2**31 - 1:
                raise ValueError("the transposed view needs a whole graph on one GPU (row_base 0, nnz < 2^31 - 1)")
            L, dev, N = lib(), self.device, self.N
            with torch.cuda.device(dev):
                trowptr = torch.empty(N + 1, dtype=torch.int64, device=dev)
                tcol = torch.empty(max(self.nnz, 1), dtype=torch.int32, device=dev)
                tperm = torch.empty(max(self.nnz, 1), dtype=torch.int32, device=dev)
                ws_bytes = L.dl_transpose_index_workspace_bytes(N, self.nnz)
                ws = _ws(ws_bytes, dev)
                check(L.dl_transpose_index(ptr(self.col), ptr(self.erow), N, self.nnz, ptr(trowptr), ptr(tcol),
                                           ptr(tperm), ptr(ws), ws_bytes, stream_of(dev)), "dl_transpose_index")
                del ws
            tg = Graph(trowptr, tcol[:self.nnz], N)
            tg._sym = False
            tg.flags = self._flags
            self._transpose = (tg, tperm[:self.nnz])
        return self._transpose

    def rows(self) -> torch.Tensor:
        """Row id of every entry (torch op; for tests and dense views)."""
        deg = self.rowptr[1:] - self.rowptr[:-1]
        return torch.repeat_interleave(torch.arange(self.N, device=self.device), deg)

    def degrees(self) -> torch.Tensor:
        return self.rowptr[1:] - self.rowptr[:-1]
