"""Drop-in for the reference's ``model.py`` (sjz5202/DisenLink), backed by sm_100a CUDA kernels.

Same class names, constructor signatures, ``forward`` signatures and ``state_dict`` keys as the
reference, so ``from model import Disentangle`` in main_disentangled.py:14 can point here (see
INTEGRATION.md) and a reference checkpoint loads unchanged:

    Disentangle(nfeat, nhid, nebed, nfactor, beta, t=1)                     [ref: model.py:91-104]
    Disentangle.forward(x, adj) -> (H [N, K*nebed], link_pred)              [ref: model.py:105-114]
    Disentangle_layer(nfactor, beta, t).forward(Z_list, adj)
        -> (h_list, alpha0 [K,N,N], att list)                               [ref: model.py:49-77]
    Factor / Factor2 / Dec / Dec2 / Disentangle_out_layer                   [ref: model.py:7-48,79-89]

What differs is only HOW the math runs: the reference materialises K dense [N,N] similarity,
softmax and attention matrices per call; here the same quantities are evaluated per CSR entry of
adj (which is what ``p_adj = p * adj`` at model.py:62 keeps) and per scored pair, by the kernels
in csrc/.  ``adj`` may be

  * the dense [N,N] 0/1 tensor the reference script passes (drop-in mode: ``link_pred`` is then the
    dense [N,N] tensor the script indexes with boolean masks, for N up to ``dense_limit``), or
  * a ``Graph`` handle / an ``edge_index`` [2,E] tensor (scalable mode: ``link_pred`` is a
    ``LinkScorer`` that scores explicit pair batches lazily).

There is no CPU implementation: inputs must live on a CUDA device.
"""
from __future__ import annotations

import weakref
from typing import List, Optional, Union

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops
from ._lib import require_cuda
from .features import SparseFeatures
from .graph import Graph


class Factor(nn.Module):
    """[ref: model.py:7-15]"""

    def __init__(self, nfeat, nhid):
        super().__init__()
        self.nfeat = nfeat
        self.nhid = nhid
        self.mlp = nn.Linear(nfeat, nhid)

    def forward(self, x):
        return self.mlp(x)


class Factor2(nn.Module):
    """Per-factor 2-layer MLP; the only tensor-core / library GEMM on the path.
    [ref: model.py:16-27]"""

    def __init__(self, nfeat, nmid, nhid):
        super().__init__()
        self.nfeat = nfeat
        self.nhid = nhid
        self.nmid = nmid
        self.mlp1 = nn.Linear(nfeat, nmid)
        self.mlp2 = nn.Linear(nmid, nhid)

    def forward(self, x):
        return self.mlp2(F.relu(self.mlp1(x)))


class Dec2(nn.Module):
    """Unused by the reference's forward; kept importable.  [ref: model.py:28-39]"""

    def __init__(self, nembed, nhid, nfeat):
        super().__init__()
        self.nfeat = nfeat
        self.nhid = nhid
        self.nembed = nembed
        self.mlp1 = nn.Linear(nembed, nhid)
        self.mlp2 = nn.Linear(nhid, nfeat)

    def forward(self, x):
        return self.mlp2(F.relu(self.mlp1(x)))


class Dec(nn.Module):
    """Unused by the reference's forward; kept importable.  [ref: model.py:40-48]"""

    def __init__(self, nhid, nfeat):
        super().__init__()
        self.nfeat = nfeat
        self.nhid = nhid
        self.mlp = nn.Linear(nhid, nfeat)

    def forward(self, x):
        return self.mlp(x)


AdjLike = Union[torch.Tensor, Graph]


# ---- the factor projection on tensor cores: 3xTF32 -------------------------------------------------
# The projection X W is the one tensor-core contraction of the path.  Plain TF32 (10-bit mantissa) breaks the
# 1e-5 parity target, plain fp32 SGEMM leaves the tensor cores idle.  3xTF32 splits both operands into a
# TF32-exact high part and an fp32 remainder and spends three TF32 tensor-core GEMMs,
#     a b ~= a_hi b_hi + (a_hi b_lo + a_lo b_hi)        (a_lo b_lo ~ 2^-22 |a||b| is dropped),
# which keeps fp32-class accuracy (the products are exact, accumulation is fp32).  Library GEMMs (cuBLAS).
def _tf32_split(a: torch.Tensor):
    # round to nearest at 10 mantissa bits (what the tensor core keeps), remainder exact in fp32
    hi = ((a.contiguous().view(torch.int32) + 4096) & -8192).view(torch.float32)
    return hi, a - hi


class _Mm3xTF32(torch.autograd.Function):
    @staticmethod
    def _mm(a, b):
        ah, al = _tf32_split(a)
        bh, bl = _tf32_split(b)
        old = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        try:
            return torch.matmul(ah, bh) + (torch.matmul(ah, bl) + torch.matmul(al, bh))
        finally:
            torch.backends.cuda.matmul.allow_tf32 = old

    @staticmethod
    def forward(ctx, a, b):
        ctx.save_for_backward(a, b)
        return _Mm3xTF32._mm(a, b)

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        g = g.contiguous()
        return _Mm3xTF32._mm(g, b.transpose(-1, -2)), _Mm3xTF32._mm(a.transpose(-1, -2), g)


def mm_3xtf32(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """a @ b (2-D or batched) as three TF32 tensor-core GEMMs with fp32-class accuracy; differentiable."""
    return _Mm3xTF32.apply(a, b)


class _GraphCache:
    """adj is constant across the epochs of a run (main_disentangled.py:141 vs :192), so the CSR
    and its work items are built once per distinct adjacency tensor."""

    def __init__(self):
        self._ref = None                       # weakref to the tensor the cached graph was built from
        self._version = None
        self._graph: Optional[Graph] = None

    def get(self, adj: AdjLike, n_nodes: int, directed: bool = False) -> Graph:
        """A Graph is used as it is (marked or not); a tensor is turned into a graph marked ``directed``."""
        if isinstance(adj, Graph):
            return adj
        if not isinstance(adj, torch.Tensor):
            raise TypeError("adj must be a dense [N,N] tensor, an edge_index [2,E] tensor or a Graph")
        # keyed on the tensor OBJECT (a weak reference) and its version counter: an address is not an
        # identity -- the caching allocator hands a freed adjacency's address to the next one of that shape
        same = (self._ref is not None and self._ref() is adj and self._version == adj._version
                and self._graph.directed == bool(directed))
        if not same:
            require_cuda(adj, "adj")
            sparse = adj.layout != torch.strided        # checked before anything touches data_ptr()
            if sparse:
                coo = (adj.to_sparse_coo() if adj.layout != torch.sparse_coo else adj).coalesce()
                idx = coo.indices()[:, coo.values() != 0]
                rp_graph = _graph_from_entries(idx[0], idx[1], n_nodes, directed)
            elif adj.dim() == 2 and adj.shape[0] == 2 and not adj.is_floating_point():
                rp_graph = Graph.from_edge_index(adj, n_nodes, directed=directed)
            elif adj.dim() == 2 and adj.shape[0] == adj.shape[1] == n_nodes:
                rp_graph = Graph.from_dense(adj, directed=directed)
            else:
                raise ValueError(f"cannot interpret adj of shape {tuple(adj.shape)} for N={n_nodes}")
            self._ref, self._version, self._graph = weakref.ref(adj), adj._version, rp_graph
        return self._graph


def _graph_from_entries(row, col, n_nodes, directed=False):
    """Entries used as given (no symmetrisation): sort + unique through the edge kernel would
    symmetrise, so build the CSR from sorted keys with torch integer ops (one-off, tiny)."""
    key = torch.unique(row.to(torch.int64) * n_nodes + col.to(torch.int64))
    r, c = key // n_nodes, (key % n_nodes).to(torch.int32)
    rowptr = torch.zeros(n_nodes + 1, dtype=torch.int64, device=row.device)
    rowptr[1:] = torch.cumsum(torch.bincount(r, minlength=n_nodes), 0)
    return Graph(rowptr, c, n_nodes, directed=directed)


def is_dense_adj(adj: AdjLike, n_nodes: int) -> bool:
    return (isinstance(adj, torch.Tensor) and adj.layout == torch.strided and adj.dim() == 2
            and adj.shape[0] == adj.shape[1] == n_nodes and (adj.is_floating_point() or n_nodes != 2))


class Disentangle_layer(nn.Module):
    """[ref: model.py:49-77]  forward(Z: list of K [N,d] tensors, adj) ->
    (h_all_factor: list of K [N,d], alpha0 [K,N,N], att: list of K [N,N]).

    ``h_all_factor`` is differentiable w.r.t. Z.  ``alpha0`` and ``att`` are dense diagnostic
    views (detached) and are only materialised for N <= dense_limit; use ``sparse_forward`` for
    the per-entry form at scale."""

    def __init__(self, nfactor, beta, t=1, dense_limit: int = 8192):
        super().__init__()
        self.temperature = t
        self.nfactor = nfactor
        self.beta = beta
        self.dense_limit = dense_limit
        self._cache = _GraphCache()
        # how a tensor adj is read: "symmetric" (an undirected graph like the script's adj_sym; the backward
        # refuses a pattern that is not symmetric) or "directed" (any 0/1 pattern, used as given; the backward
        # gathers over its transpose).  A Graph handle carries its own mark (Graph.directed).
        self.adjacency = "symmetric"

    def _directed(self) -> bool:
        if self.adjacency not in ("symmetric", "directed"):
            raise ValueError(f"adjacency must be 'symmetric' or 'directed', got {self.adjacency!r}")
        return self.adjacency == "directed"

    def sparse_forward(self, Z: torch.Tensor, adj: AdjLike):
        """Z [N,K,d] -> (H [N,K,d], kstar u8 [nnz], w [nnz], s [N,K], graph)."""
        graph = self._cache.get(adj, Z.shape[0], self._directed())
        H, kstar, w, s = ops.factor_aggregate(Z, graph, self.beta, float(self.temperature),
                                              return_attention=True)
        return H, kstar, w, s, graph

    def forward(self, Z: List[torch.Tensor], adj: AdjLike):
        Zs = torch.stack(list(Z), dim=1)
        N = Zs.shape[0]
        H, kstar, w, s, graph = self.sparse_forward(Zs, adj)
        h_all_factor = [H[:, k, :] for k in range(self.nfactor)]
        if N > self.dense_limit:
            raise RuntimeError(
                f"Disentangle_layer.forward returns dense [K,N,N] tensors; N={N} exceeds "
                f"dense_limit={self.dense_limit}. Use sparse_forward().")
        alpha0 = ops.dense_alpha0(Zs, float(self.temperature))
        att = ops.dense_att(graph, kstar, w, s, self.nfactor)
        return h_all_factor, alpha0, [att[k] for k in range(self.nfactor)]


class Disentangle_out_layer(nn.Module):
    """Dead code in the reference (never instantiated); kept importable, plain torch.
    [ref: model.py:79-89]"""

    def __init__(self, beta, t=1):
        super().__init__()
        self.temperature = t
        self.beta = beta

    def forward(self, Z, adj):
        temp = torch.exp(torch.mm(Z, Z.t()) / self.temperature)
        alpha = temp / torch.sum(temp, dim=1)
        p_adj = alpha * adj
        return self.beta * Z + (1 - self.beta) * torch.mm(p_adj, Z), alpha


class LinkScorer:
    """Lazy stand-in for the dense ``link_pred`` [N,N] of model.py:113 when N is large.

    ``scorer(pairs)`` / ``scorer.score(batch)`` evaluate sigmoid(sum_k exp(z_u^k.z_v^k/T)
    (h_u^k.h_v^k)) on explicit pairs (differentiable).  ``scorer[mask]`` accepts a dense boolean
    [N,N] mask like the script's ``a_pred[pos_train_adj==1]`` and returns the scores in the same
    row-major order."""

    def __init__(self, Z: torch.Tensor, H: torch.Tensor, T: float):
        self.Z, self.H, self.T = Z, H, float(T)
        self.N = int(Z.shape[0])

    def score(self, batch: ops.PairBatch, as_prob: bool = True) -> torch.Tensor:
        return ops.pair_score(self.Z, self.H, batch, self.T, as_prob)

    def __call__(self, pairs, as_prob: bool = True) -> torch.Tensor:
        if not isinstance(pairs, ops.PairBatch):
            pairs = ops.PairBatch(pairs[0], pairs[1], self.N)
        return self.score(pairs, as_prob)

    def __getitem__(self, mask: torch.Tensor) -> torch.Tensor:
        if mask.dtype != torch.bool or tuple(mask.shape) != (self.N, self.N):
            raise IndexError("LinkScorer only supports dense boolean [N,N] masks or pair batches")
        idx = mask.nonzero(as_tuple=True)
        return self(idx)

    def dense(self) -> torch.Tensor:
        return ops.allpairs_score(self.Z, self.H, self.T)


class Disentangle(nn.Module):
    """[ref: model.py:91-114]"""

    def __init__(self, nfeat, nhid, nebed, nfactor, beta, t=1, dense_limit: int = 16384):
        super().__init__()
        if nhid == 1:
            self.factors = [Factor(nfeat, nebed) for _ in range(nfactor)]
        else:
            self.factors = [Factor2(nfeat, nhid, nebed) for _ in range(nfactor)]
        for i, factor in enumerate(self.factors):
            self.add_module('factor_{}'.format(i), factor)
        self.disentangle_layer1 = Disentangle_layer(nfactor, beta, t)
        self.disentangle_layer2 = Disentangle_layer(nfactor, beta, t)
        self.temperature = t
        self.nfactor = nfactor
        self.beta = beta
        self.dense_limit = dense_limit
        # "fp32": plain SGEMM (default, bit-compatible with the reference's nn.Linear on the same library);
        # "3xtf32": three TF32 tensor-core GEMMs per product, fp32-class accuracy (dense CUDA x only)
        self.projection = "fp32"

    @property
    def adjacency(self) -> str:
        """"symmetric" (default): a tensor adj is an undirected graph such as adj_sym, and the backward
        refuses a pattern that is not symmetric.  "directed": a dense, sparse or edge_index adj is used as
        given (edge_index columns are not symmetrised) and trains through the backward over its transpose,
        e.g. the directed train adjacency.  A Graph handle passed as adj carries its own mark."""
        return self.disentangle_layer1.adjacency

    @adjacency.setter
    def adjacency(self, value: str) -> None:
        self.disentangle_layer1.adjacency = value
        self.disentangle_layer2.adjacency = value

    def project(self, x: Union[torch.Tensor, SparseFeatures]) -> torch.Tensor:
        """Z [N,K,d] = the K factor MLPs of model.py:106, batched: one [N,F] x [F,K*nhid] GEMM for the
        K first layers (a sparse-dense product when x is a sparse tensor: bag-of-words features are
        ~1 % dense) and one batched [K] x ([N,nhid] x [nhid,d]) product for the second layers, written
        straight into the [N,K,d] layout.  The parameters stay the per-factor nn.Linear modules of
        the reference (same state_dict); the stacked weights are views rebuilt per call, so autograd
        routes the gradients back to them.  Library GEMMs, fp32 -- TF32 would break the 1e-5 parity
        target.  When x is a ``SparseFeatures`` handle the first layers (with their ReLU) run over its
        nonzeros in the project's kernels (ops.feature_projection); the second layers are unchanged."""
        K = len(self.factors)
        first = [f.mlp if isinstance(f, Factor) else f.mlp1 for f in self.factors]
        b1 = torch.cat([m.bias for m in first], dim=0)
        if isinstance(x, SparseFeatures):
            Wt = torch.cat([m.weight.t() for m in first], dim=1)      # [F, K*nhid]
            hid = ops.feature_projection(x, Wt, b1, relu=not isinstance(self.factors[0], Factor), blocks=K)
            if isinstance(self.factors[0], Factor):
                return hid.transpose(0, 1)                            # [N, K, d], contiguous
            return self._second_layer(hid, False)
        W1 = torch.cat([m.weight for m in first], dim=0)              # [K*nhid, F]
        tc = self.projection == "3xtf32" and x.is_cuda and x.layout == torch.strided
        if x.is_sparse or x.layout == torch.sparse_csr:
            hid = torch.sparse.mm(x, W1.t()) + b1
        elif tc:
            hid = mm_3xtf32(x, W1.t()) + b1
        else:
            hid = torch.addmm(b1, x, W1.t())                          # [N, K*nhid]
        N = hid.shape[0]
        if isinstance(self.factors[0], Factor):
            return hid.view(N, K, -1)
        hid = F.relu(hid).view(N, K, -1).transpose(0, 1)              # [K, N, nhid]
        return self._second_layer(hid, tc)

    def _second_layer(self, hid: torch.Tensor, tc: bool) -> torch.Tensor:
        """[K, N, nhid] hidden layers -> Z [N, K, d]."""
        W2 = torch.stack([f.mlp2.weight for f in self.factors], dim=0)  # [K, d, nhid]
        b2 = torch.stack([f.mlp2.bias for f in self.factors], dim=0)    # [K, d]
        if tc:
            Z = mm_3xtf32(hid.contiguous(), W2.transpose(1, 2)) + b2.unsqueeze(1)
        else:
            Z = torch.baddbmm(b2.unsqueeze(1), hid, W2.transpose(1, 2))   # [K, N, d]
        return Z.transpose(0, 1).contiguous()

    def embed(self, x: Union[torch.Tensor, SparseFeatures], adj: AdjLike):
        """-> (Z [N,K,d], H [N,K,d], graph)"""
        require_cuda(x, "x")
        Z = self.project(x)
        H, _, _, _, graph = self.disentangle_layer1.sparse_forward(Z, adj)
        return Z, H, graph

    def forward(self, x: Union[torch.Tensor, SparseFeatures], adj: AdjLike):
        Z, H, graph = self.embed(x, adj)
        N = Z.shape[0]
        T = float(self.temperature)
        if is_dense_adj(adj, N):
            if N > self.dense_limit:
                raise RuntimeError(
                    f"a dense adj asks for a dense [N,N] link_pred; N={N} exceeds dense_limit="
                    f"{self.dense_limit}. Pass a Graph / edge_index and use the LinkScorer.")
            link_pred = ops.allpairs_score(Z, H, T)
        else:
            link_pred = LinkScorer(Z, H, T)
        return H.reshape(N, -1), link_pred
