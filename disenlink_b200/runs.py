"""The reference's independent runs trained together: R models over R edge splits in one batched step.

main_disentangled.py:131-224 repeats its whole protocol ``for run in range(args.run)`` -- a fresh 85/10/5 split,
``adj_sym``, negatives and model per run -- and reports the mean and std of the test AUCs.  The runs share
nothing, so they are stacked instead of repeated:

  * node i of run r is node ``r*N + i`` of one union graph.  The union of the runs' train adjacencies is one CSR
    whose rows never reach another run's rows, and attention, aggregation, pair scoring and both backward
    passes are per row or per pair, so one call over the union gives every run exactly its own results;
  * ``DisentangleRuns`` holds R parameter sets of ``Disentangle`` stacked along a leading run axis and projects
    one shared ``x`` into the union's ``Z [R*N, K, d]``.  Adam and weight decay act element by element, so one
    optimizer over the stacked parameters takes the steps R optimizers would;
  * ``RunSet`` builds each run's split, negatives, loss / eval pairs, labels and weights exactly as
    examples/train_link.py's ``run()`` does for one seed, then offsets and concatenates them, with ``seg_ptr``
    marking each run's segment of every pair list (ops.link_bce_segments / ops.roc_auc_segments read them);
  * ``EarlyStopping`` keeps the script's per-run stopping rule on the device.

    runs = RunSet(edge_index, N, seeds=[0, 1, 2], m=5)
    model = DisentangleRuns(F, nhid, d, K, beta, t, runs=3).cuda()
    Z = model.project(x)                                        # [3N, K, d]
    loss, prob, H = ops.link_bce_loss(Z, runs.graph, runs.train, runs.train_labels, runs.train_weights, beta, t)
    per_run_loss = ops.link_bce_segments(prob, runs.train_labels, runs.train_weights, runs.train_ptr)
"""
from __future__ import annotations

from collections import OrderedDict
from typing import List, Sequence

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import data, ops
from ._lib import require_cuda
from .graph import Graph
from .model import Disentangle, Factor2


def edge_labels(u, v, edge_keys, n):
    """ori_adj[u, v] of the script: 1 where (u, v) is a column of the full edge set (edge_keys = the sorted
    unique u * n + v of its columns)."""
    k = u.long() * n + v.long()
    pos = torch.searchsorted(edge_keys, k).clamp_(max=edge_keys.numel() - 1)
    return (edge_keys[pos] == k).float()


class DisentangleRuns(nn.Module):
    """R parameter sets of ``Disentangle`` (the Factor2 branch, nhid > 1), stacked:
    ``W1 [R, K*nhid, F]``, ``b1 [R, K*nhid]``, ``W2 [R, K, d, nhid]``, ``b2 [R, K, d]``.

    A new module initialises run r as the r-th of R ``Disentangle(nfeat, nhid, nebed, nfactor, beta, t)``
    constructed one after another from the global RNG; ``from_models`` packs modules that exist already.
    ``run_state_dict(r)`` gives run r's weights under the reference's keys."""

    def __init__(self, nfeat, nhid, nebed, nfactor, beta, t=1, runs=1):
        super().__init__()
        if nhid == 1:
            raise ValueError("DisentangleRuns stacks the two-layer factors (nhid > 1); nhid == 1 is not supported")
        if runs < 1:
            raise ValueError(f"runs must be >= 1, got {runs}")
        self.runs, self.nfeat, self.nhid, self.nembed, self.nfactor = int(runs), int(nfeat), int(nhid), int(nebed), int(nfactor)
        self.beta, self.temperature = beta, t
        R, K = self.runs, self.nfactor
        self.W1 = nn.Parameter(torch.empty(R, K * nhid, nfeat))
        self.b1 = nn.Parameter(torch.empty(R, K * nhid))
        self.W2 = nn.Parameter(torch.empty(R, K, nebed, nhid))
        self.b2 = nn.Parameter(torch.empty(R, K, nebed))
        for r in range(R):
            self.load_run_state_dict(r, Disentangle(nfeat, nhid, nebed, nfactor, beta, t).state_dict())

    @classmethod
    def from_models(cls, models: Sequence[Disentangle]) -> "DisentangleRuns":
        """Stack existing ``Disentangle`` modules of one shape (run r = models[r]).  Leaves the global RNG as it was."""
        m0 = models[0]
        if not isinstance(m0.factors[0], Factor2):
            raise ValueError("DisentangleRuns stacks the two-layer factors (nhid > 1); nhid == 1 is not supported")
        f = m0.factors[0]
        with torch.random.fork_rng(devices=[]):
            out = cls(f.mlp1.in_features, f.mlp1.out_features, f.mlp2.out_features, m0.nfactor, m0.beta,
                      m0.temperature, runs=len(models))
        out = out.to(f.mlp1.weight.device)
        for r, m in enumerate(models):
            out.load_run_state_dict(r, m.state_dict())
        return out

    def _slices(self, r: int):
        """(key, view of the stacked parameter) of run r, in Disentangle.state_dict() order."""
        h = self.nhid
        for i in range(self.nfactor):
            yield f"factor_{i}.mlp1.weight", self.W1[r, i * h:(i + 1) * h]
            yield f"factor_{i}.mlp1.bias", self.b1[r, i * h:(i + 1) * h]
            yield f"factor_{i}.mlp2.weight", self.W2[r, i]
            yield f"factor_{i}.mlp2.bias", self.b2[r, i]

    def run_state_dict(self, r: int) -> "OrderedDict[str, torch.Tensor]":
        """Run r's weights (copies) under the keys of ``Disentangle.state_dict()`` (the reference's model.py)."""
        if not 0 <= r < self.runs:
            raise IndexError(f"run {r} of {self.runs}")
        return OrderedDict((k, v.detach().clone()) for k, v in self._slices(r))

    def load_run_state_dict(self, r: int, state_dict) -> None:
        """Inverse of ``run_state_dict``: the keys must be exactly those of ``Disentangle.state_dict()``."""
        if not 0 <= r < self.runs:
            raise IndexError(f"run {r} of {self.runs}")
        slices = OrderedDict(self._slices(r))
        if set(state_dict.keys()) != set(slices.keys()):
            missing = sorted(set(slices) - set(state_dict))
            unexpected = sorted(set(state_dict) - set(slices))
            raise KeyError(f"run state dict mismatch: missing {missing}, unexpected {unexpected}")
        with torch.no_grad():
            for k, dst in slices.items():
                src = state_dict[k]
                if tuple(src.shape) != tuple(dst.shape):
                    raise ValueError(f"{k}: shape {tuple(src.shape)}, expected {tuple(dst.shape)}")
                dst.copy_(src)

    def project(self, x: torch.Tensor) -> torch.Tensor:
        """Z [R*N, K, d] of a shared x [N, F]; row r*N + i is run r's node i (Disentangle.project per run).
        The first layers of all runs and factors are one [N,F] x [F, R*K*nhid] GEMM (torch.sparse.mm for a
        sparse x), the second layers one batched product over the R*K factors.  Library GEMMs, fp32."""
        R, K, h, d = self.runs, self.nfactor, self.nhid, self.nembed
        W1 = self.W1.reshape(R * K * h, self.nfeat)
        b1 = self.b1.reshape(R * K * h)
        if x.is_sparse or x.layout == torch.sparse_csr:
            hid = torch.sparse.mm(x, W1.t()) + b1
        else:
            hid = torch.addmm(b1, x, W1.t())                                  # [N, R*K*nhid]
        N = hid.shape[0]
        hid = F.relu(hid).view(N, R * K, h).transpose(0, 1)                   # [R*K, N, nhid]
        Z = torch.baddbmm(self.b2.reshape(R * K, 1, d), hid, self.W2.reshape(R * K, d, h).transpose(1, 2))
        return Z.view(R, K, N, d).transpose(1, 2).reshape(R * N, K, d)      # [R, N, K, d]


class RunSet:
    """The per-run data of main_disentangled.py:134-190 for R seeds, offset by r*N and concatenated.

    Run r is what examples/train_link.py's ``run()`` builds for ``--seed seeds[r]``: split
    ``data.split_edges(E, seeds[r])``, negatives ``ops.structured_negative_sampling(edge_index, N,
    seed=seeds[r]*1000 + m_index)`` against the full edge set, loss pairs ``pairs_exactly_once`` with the same
    labels and weights, eval pairs ``pairs_at_least_once``.

      graph                         union of the runs' train adjacencies (adj_sym, or adj if ``directed``)
      train / val / test            PairBatch over the R*N union ids
      train_labels, train_weights   per train pair; val_labels, test_labels per eval pair
      train_ptr / val_ptr / test_ptr  int64 [R+1] on the device: run r's pairs are [ptr[r], ptr[r+1])
    """

    def __init__(self, edge_index: torch.Tensor, n_nodes: int, seeds: Sequence[int], m: int, directed: bool = False):
        require_cuda(edge_index, "edge_index")
        N, R = int(n_nodes), len(seeds)
        if R < 1:
            raise ValueError("RunSet needs at least one seed")
        if R * N >= 2**31:
            raise ValueError(f"R*N = {R}*{N} must stay below 2^31 (int32 node ids of the union)")
        dev = edge_index.device
        E = int(edge_index.shape[1])
        self.N, self.R, self.seeds, self.directed = N, R, [int(s) for s in seeds], bool(directed)
        full = Graph.from_edges(edge_index[0], edge_index[1], N, symmetrize=False)
        edge_keys = torch.unique(edge_index[0].long() * N + edge_index[1].long())
        src, dst = [], []
        parts = {"train": ([], [], [], []), "val": ([], [], []), "test": ([], [], [])}
        for r, seed in enumerate(self.seeds):
            off = r * N
            tr, te, va = data.split_edges(E, seed, dev)
            train_edges = edge_index[:, tr]
            src.append(train_edges[0] + off)
            dst.append(train_edges[1] + off)
            neg = {"tr": [], "va": [], "te": []}
            for m_index in range(m):                                      # main_disentangled.py:159-163
                i, _, k = ops.structured_negative_sampling(edge_index, N, seed=seed * 1000 + m_index, graph=full)
                for name, idx in (("tr", tr), ("va", va), ("te", te)):
                    neg[name].append(torch.stack([i[idx], k[idx]]))
            neg = {k_: torch.cat(v_, dim=1) for k_, v_ in neg.items()}
            pu, pv = ops.pairs_exactly_once(train_edges[0], train_edges[1], N)     # :175-178,195
            nu, nv = ops.pairs_exactly_once(neg["tr"][0], neg["tr"][1], N)
            u, v, lab, wt = parts["train"]
            u.append(torch.cat([pu, nu]) + off)
            v.append(torch.cat([pv, nv]) + off)
            lab.append(torch.cat([edge_labels(pu, pv, edge_keys, N), edge_labels(nu, nv, edge_keys, N)]))
            wt.append(torch.cat([torch.full((pu.numel(),), 1.0 / max(pu.numel(), 1), device=dev),
                                 torch.full((nu.numel(),), 1.0 / (m * max(nu.numel(), 1)), device=dev)]))
            for name, pos_idx, negs in (("val", va, neg["va"]), ("test", te, neg["te"])):   # :188-190
                eu, ev = ops.pairs_at_least_once(torch.cat([edge_index[0][pos_idx], negs[0]]),
                                                 torch.cat([edge_index[1][pos_idx], negs[1]]), N)
                u, v, lab = parts[name]
                u.append(eu + off)
                v.append(ev + off)
                lab.append(edge_labels(eu, ev, edge_keys, N))
        self.graph = Graph.from_edges(torch.cat(src), torch.cat(dst), R * N, directed=self.directed)
        u, v, lab, wt = parts["train"]
        self.train, self.train_ptr = self._batch(u, v, dev)
        self.train_labels, self.train_weights = torch.cat(lab), torch.cat(wt)
        u, v, lab = parts["val"]
        self.val, self.val_ptr = self._batch(u, v, dev)
        self.val_labels = torch.cat(lab)
        u, v, lab = parts["test"]
        self.test, self.test_ptr = self._batch(u, v, dev)
        self.test_labels = torch.cat(lab)

    def _batch(self, us: List[torch.Tensor], vs: List[torch.Tensor], dev):
        ptr = [0]
        for u in us:
            ptr.append(ptr[-1] + int(u.numel()))
        return (ops.PairBatch(torch.cat(us), torch.cat(vs), self.R * self.N),
                torch.tensor(ptr, dtype=torch.int64, device=dev))


class EarlyStopping:
    """Per-run early stopping of main_disentangled.py:205-213 on the device, for parameters stacked along a
    leading run axis.  Per epoch, for every run that has not stopped:

        if auc > best_auc: best_auc = auc; stale = 0; snapshot = weights after the step
        else:              stale += 1
        if stale > patience: the run stops

    (a NaN AUC is no improvement).  A stopped run is frozen: its best_auc, stale and snapshot never change
    again, so its result is the one the script's ``break`` gives, while its rows may keep training in the
    union.  The snapshot starts as the weights given here, which a run that never improves keeps."""

    def __init__(self, params: Sequence[torch.Tensor], patience: int = 200):
        self.params = list(params)
        R, dev = int(self.params[0].shape[0]), self.params[0].device
        self.patience = int(patience)
        self.best_auc = torch.zeros(R, dtype=torch.float64, device=dev)
        self.stale = torch.zeros(R, dtype=torch.int64, device=dev)
        self.stopped = torch.zeros(R, dtype=torch.bool, device=dev)
        self.snapshot = [p.detach().clone() for p in self.params]

    @torch.no_grad()
    def update(self, auc: torch.Tensor) -> None:
        """One epoch: auc = float64 [R] validation AUC of every run (after the optimizer step)."""
        active = ~self.stopped
        improved = active & (auc > self.best_auc)
        self.best_auc.copy_(torch.where(improved, auc, self.best_auc))
        self.stale.copy_(torch.where(improved, torch.zeros_like(self.stale), self.stale + active.long()))
        for p, snap in zip(self.params, self.snapshot):
            mask = improved.view(-1, *([1] * (p.dim() - 1)))
            torch.where(mask, p.detach(), snap, out=snap)                # masked copy of the improved runs
        self.stopped |= active & (self.stale > self.patience)

    @torch.no_grad()
    def restore(self) -> None:
        """Copy every run's snapshot (its best weights) into the parameters."""
        for p, snap in zip(self.params, self.snapshot):
            p.copy_(snap)
