"""The training epoch of examples/train_link.py captured once as a CUDA graph and replayed, with early stopping
and model selection on the device and one device-to-host copy per chunk of epochs.

On the reference's small graphs (Cora, Citeseer, the WebKB sets, chameleon, squirrel) an epoch is a few dozen
launches whose host overhead exceeds the work they carry.  ``CapturedEpoch`` records everything one epoch does
-- projection, fused loss forward + backward, optimizer step, per-run losses, validation scores from the
training forward's H (main_disentangled.py:202), the AUC and the stopping update of ``runs.EarlyStopping`` --
with ``torch.cuda.graph`` and replays it.  Each replay writes the epoch's record (R losses, R validation AUCs,
R best AUCs, R stop flags: the row ``batched_epoch`` returns) into slot ``epoch % chunk`` of a static device
buffer through an epoch counter the graph increments itself; ``run`` reads the buffer back once per chunk.

    opt = torch.optim.Adam(model.parameters(), lr=0.01, weight_decay=5e-4, capturable=True)
    ce = CapturedEpoch(model, opt, x, graph, train, train_labels, train_weights, val, val_labels,
                       test, test_labels, beta, T, patience=200, chunk=50)
    out = ce.run(2000)          # per-run history, best validation AUC, test AUC with the best weights

Decided once, before capture, and held: the backward plan (``ops.bwd_plan``: scratch mode and buffers, which
otherwise depend on free memory at each call), and every lazily built cache (graph views, incidence lists,
scratch, library handles and workspaces), which one eager epoch on the capture stream builds.  That epoch is
undone afterwards: weights, optimizer state and stopping state are put back, so the first replay is epoch 0.
Inputs are read by address at every replay: weights loaded in place (``load_state_dict``) are what the next
replay trains.

Refused before capture (RuntimeError): a sparse ``x``, a row-partitioned graph (the partitioned steps check
indices with a host synchronisation), and an optimizer that is not capturable (Adam needs ``capturable=True``
or ``fused=True``).  ``ops.roc_auc`` reads its result on the host and raises inside a capture.
"""
from __future__ import annotations

import time
from typing import Callable, List, Sequence

import torch

from . import ops
from .graph import Graph
from .model import Disentangle
from .runs import DisentangleRuns, EarlyStopping


def run_chunks(step: Callable[[int], List[Sequence[float]]], epochs: int, chunk: int, R: int, log=None,
               log_every: int = 0):
    """The host side of ``CapturedEpoch.run``: calls ``step(n)`` (n epochs, n <= chunk; -> their n records of 4R
    values) until every run has stopped at a chunk's end or ``epochs`` epochs have run.  Run r's history holds
    (loss, validation AUC) of every epoch up to and including the one its stop flag is first set in.
    -> (history per run, epochs run)."""
    history: List[list] = [[] for _ in range(R)]
    active = [True] * R
    done = 0
    while done < epochs and any(active):
        n = min(chunk, epochs - done)
        rows = step(n)
        for i, row in enumerate(rows):
            for r in range(R):
                if active[r]:
                    history[r].append((row[r], row[R + r]))
                    active[r] = not row[3 * R + r]
            if log is not None and log_every and (done + i) % log_every == 0:
                log(f"epoch: {done + i} active runs: {sum(active)}/{R} loss: {sum(row[:R]) / R:.5f} (mean) "
                    f"val_auc: " + " ".join(f"{b:.4f}" for b in row[2 * R:3 * R]))
        done += n
    return history, done


def _capturable(opt: torch.optim.Optimizer) -> bool:
    return all(g.get("capturable") or g.get("fused") for g in opt.param_groups)


class CapturedEpoch:
    """One training epoch of ``model`` (``Disentangle``, R = 1, or ``DisentangleRuns``, R runs over a ``RunSet``
    union), captured as a CUDA graph (``capture=False``: the same epoch run eagerly, the reference the replay
    is held to).

    x                                  dense features [N, F] on the device
    graph                              the train adjacency (adj_sym, or a graph marked directed)
    train, train_labels, train_weights loss pairs; val / val_labels and test / test_labels eval pairs
    train_ptr, val_ptr, test_ptr       the RunSet's int64 [R+1] segment pointers (R > 1 only)
    patience, chunk                    stopping rule; epochs per host read (the record buffer's rows)
    """

    def __init__(self, model, opt: torch.optim.Optimizer, x: torch.Tensor, graph: Graph, train: ops.PairBatch,
                 train_labels, train_weights, val: ops.PairBatch, val_labels, test: ops.PairBatch, test_labels,
                 beta: float, T: float = 1.0, patience: int = 200, chunk: int = 1, train_ptr=None, val_ptr=None,
                 test_ptr=None, capture: bool = True):
        if isinstance(model, DisentangleRuns):
            self.R = model.runs
            if self.R > 1 and (train_ptr is None or val_ptr is None or test_ptr is None):
                raise ValueError("R > 1 runs need the RunSet's train_ptr, val_ptr and test_ptr")
        elif isinstance(model, Disentangle):
            self.R = 1
        else:
            raise TypeError("CapturedEpoch trains a Disentangle or a DisentangleRuns model")
        if int(chunk) < 1:
            raise ValueError(f"chunk must be >= 1, got {chunk}")
        if x.layout != torch.strided:
            raise RuntimeError("CapturedEpoch needs a dense x: the sparse projection (torch.sparse.mm) is not "
                               "captured; pass x.to_dense()")
        if graph.row_base != 0 or graph.n_global != graph.N:
            raise RuntimeError("CapturedEpoch needs a whole graph on one GPU: the row-partitioned steps check "
                               "indices with a host synchronisation and cannot be captured")
        if not _capturable(opt):
            raise RuntimeError("the optimizer must be capturable (Adam(..., capturable=True) or fused=True): the "
                               "default Adam keeps its step count on the host")
        self.model, self.opt, self.x, self.graph = model, opt, x, graph
        self.train, self.train_labels, self.train_weights = train, train_labels, train_weights
        self.val, self.val_labels, self.test, self.test_labels = val, val_labels, test, test_labels
        self.train_ptr, self.val_ptr, self.test_ptr = train_ptr, val_ptr, test_ptr
        self.beta, self.T, self.chunk = float(beta), float(T), int(chunk)
        dev = x.device
        stacked = isinstance(model, DisentangleRuns)
        self.stop = EarlyStopping(list(model.parameters()), patience=patience, stacked=stacked)
        K, d = model.nfactor, (model.nembed if stacked else model.factors[0].nhid)
        # the backward's scratch mode is taken once, here, not per call from the free memory of the moment
        self.plan = None if graph.directed else ops.bwd_plan(graph, K, d)
        self.records = torch.zeros(self.chunk, 4 * self.R, dtype=torch.float64, device=dev)
        self.counter = torch.zeros(1, dtype=torch.int64, device=dev)     # epochs replayed, advanced on the device
        self.epoch = 0                                                   # the same count on the host
        self.graph_exec = None
        self.capture_s = 0.0
        if capture:
            t0 = time.perf_counter()
            self._capture()
            self.capture_s = time.perf_counter() - t0

    # ------------------------------------------------------------------ the epoch
    def _epoch(self) -> None:
        m, R = self.model, self.R
        Z = m.project(self.x)
        loss, prob, H = ops.link_bce_loss(Z, self.graph, self.train, self.train_labels, self.train_weights,
                                          self.beta, self.T, plan=self.plan)
        self.opt.zero_grad()
        loss.backward()
        self.opt.step()
        with torch.no_grad():
            _, val_prob = ops.pair_score_fwd(Z.detach(), H, self.val, self.T, want_logit=False)
            if R == 1:                       # run()'s loss and ops.roc_auc's statistic, without the host reads
                run_loss = loss.detach().view(1)
                auc = ops.roc_auc_stats(val_prob, self.val_labels)[:1]
            else:
                run_loss = ops.link_bce_segments(prob, self.train_labels, self.train_weights, self.train_ptr)
                auc = ops.roc_auc_segments(val_prob, self.val_labels, self.val_ptr)[:, 0]
            self.stop.update(auc)
            row = torch.cat([run_loss.double(), auc, self.stop.best_auc, self.stop.stopped.double()])
            self.records.index_copy_(0, torch.remainder(self.counter, self.chunk), row.view(1, -1))
            self.counter += 1

    def _state(self):
        """Every tensor one epoch changes, for undoing the warm-up epoch."""
        opt_state = {id(p): {k: v for k, v in st.items() if torch.is_tensor(v)} for p, st in self.opt.state.items()}
        return ([p.detach().clone() for p in self.model.parameters()],
                {i: {k: v.clone() for k, v in st.items()} for i, st in opt_state.items()},
                [t.clone() for t in (self.stop.best_auc, self.stop.stale, self.stop.stopped, *self.stop.snapshot)])

    @torch.no_grad()
    def _restore(self, saved) -> None:
        params, opt_state, stop = saved
        for p, v in zip(self.model.parameters(), params):
            p.copy_(v)
        for p, st in self.opt.state.items():
            before = opt_state.get(id(p))
            for k, v in st.items():
                if torch.is_tensor(v):
                    # state the warm-up created (Adam's lazy init) goes back to its initial zeros
                    v.copy_(before[k]) if before is not None else v.zero_()
        for t, v in zip((self.stop.best_auc, self.stop.stale, self.stop.stopped, *self.stop.snapshot), stop):
            t.copy_(v)
        self.counter.zero_()
        self.records.zero_()

    def _capture(self) -> None:
        saved = self._state()
        s = torch.cuda.Stream(device=self.x.device)
        s.wait_stream(torch.cuda.current_stream(self.x.device))
        with torch.cuda.stream(s):
            self._epoch()                    # builds every lazy cache and workspace outside the graph
        torch.cuda.current_stream(self.x.device).wait_stream(s)
        self._restore(saved)
        self.opt.zero_grad(set_to_none=True)
        torch.cuda.synchronize(self.x.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            self._epoch()
        self.graph_exec = g
        # the graph holds raw addresses of the scratch buffers cached on the graph handles: keep them alive even if
        # a later eager call on these handles replaces a cache with a larger buffer
        handles = [self.graph, self.train.incidence()[0]]
        for view in (self.graph._sym, self.graph._sym_lower, self.graph._transpose):
            if view:
                handles.append(view[0])
        self._held = [getattr(h, a, None) for h in handles for a in ("_x_scratch", "_hub_ws", "_sr_scratch")]

    # ------------------------------------------------------------------ driving it
    def step(self, n: int) -> List[List[float]]:
        """Run n <= chunk epochs (replays, or eager epochs when not captured) -> their n records, in epoch order,
        read back in one device-to-host copy."""
        if not 1 <= n <= self.chunk:
            raise ValueError(f"step takes 1 <= n <= chunk = {self.chunk} epochs, got {n}")
        for _ in range(n):
            if self.graph_exec is not None:
                self.graph_exec.replay()
            else:
                self._epoch()
        host = self.records.cpu().tolist()
        first = self.epoch
        self.epoch += n
        return [host[(first + i) % self.chunk] for i in range(n)]

    def run(self, epochs: int, log=None, log_every: int = 0) -> dict:
        """The script's loop (main_disentangled.py:192-221) in chunks of ``chunk`` epochs, ending at the first chunk
        boundary after every run has stopped or after ``epochs`` epochs; then every run's best weights are
        restored and its test AUC is computed from them, as examples/train_link.py does.
        -> {"history": [R lists of (loss, val AUC)], "best_val_auc": [R], "test_auc": [R], "epochs": n}"""
        history, done = run_chunks(self.step, epochs, self.chunk, self.R, log=log, log_every=log_every)
        self.stop.restore()
        with torch.no_grad():
            Z = self.model.project(self.x)
            H = ops.factor_aggregate(Z, self.graph, self.beta, self.T)
            _, test_prob = ops.pair_score_fwd(Z, H, self.test, self.T, want_logit=False)
        if self.R == 1:
            test_auc = [ops.roc_auc(test_prob, self.test_labels)]
        else:
            test_auc = ops.roc_auc_segments(test_prob, self.test_labels, self.test_ptr)[:, 0].tolist()
        return {"history": history, "best_val_auc": self.stop.best_auc.tolist(), "test_auc": test_auc,
                "epochs": done}
