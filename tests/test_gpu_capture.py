"""The captured training epoch (disenlink_b200/capture.py) against the same epoch run eagerly: bitwise equal records,
weights, Adam state and snapshots on every step path; stops inside a chunk; inputs read at replay time; the
refused cases; examples/train_link.py --capture against the default eager loops."""
import argparse
import copy
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden
from disenlink_b200 import _lib, ops
from disenlink_b200.capture import CapturedEpoch
from disenlink_b200.graph import Graph
from disenlink_b200.model import Disentangle
from disenlink_b200.runs import DisentangleRuns, RunSet

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
sys.path.insert(0, os.path.join(ROOT, "examples"))
F_IN, NHID = 96, 64


def _cora():
    g = load_golden("cora_K3_d32")
    ei = torch.stack([torch.as_tensor(g["src"]), torch.as_tensor(g["dst"])]).to(DEV)
    return ei, int(g["N"]), float(g["beta"]), float(g["T"])


def _features(N, F=F_IN, seed=0):
    gx = torch.Generator().manual_seed(seed)
    return (torch.rand(N, F, generator=gx) < 0.05).float().to(DEV)


def _model(R, K, d, seed=0):
    torch.manual_seed(seed)
    if R == 1:
        return Disentangle(F_IN, NHID, d, nfactor=K, beta=0.7).to(DEV)
    return DisentangleRuns(F_IN, NHID, d, K, 0.7, runs=R).to(DEV)


def _pair(runs, x, R, K, d, beta, T, chunk, patience=200, lr=0.01, seed=0):
    """(eager, captured) CapturedEpochs from the same initial weights and fresh capturable Adams."""
    base = _model(R, K, d, seed)
    out = []
    for capture in (False, True):
        m = copy.deepcopy(base)
        opt = torch.optim.Adam(m.parameters(), lr=lr, weight_decay=5e-4, capturable=True)
        ptrs = dict(train_ptr=runs.train_ptr, val_ptr=runs.val_ptr, test_ptr=runs.test_ptr) if R > 1 else {}
        out.append(CapturedEpoch(m, opt, x, runs.graph, runs.train, runs.train_labels, runs.train_weights, runs.val,
                                 runs.val_labels, runs.test, runs.test_labels, beta, T, patience=patience,
                                 chunk=chunk, capture=capture, **ptrs))
    return out


def _bits(t):
    return t.detach().contiguous().view(torch.int64 if t.element_size() == 8 else
                                        torch.int32 if t.element_size() == 4 else torch.uint8)


def _assert_same_state(a: CapturedEpoch, b: CapturedEpoch):
    assert torch.equal(_bits(a.records), _bits(b.records))
    for pa, pb in zip(a.model.parameters(), b.model.parameters()):
        assert torch.equal(_bits(pa), _bits(pb))
        sa, sb = a.opt.state[pa], b.opt.state[pb]
        assert sa.keys() == sb.keys()
        for k in sa:
            assert torch.equal(_bits(sa[k]), _bits(sb[k])), k
    for ta, tb in zip(a.stop.snapshot, b.stop.snapshot):
        assert torch.equal(_bits(ta), _bits(tb))
    for name in ("best_auc", "stale", "stopped"):
        assert torch.equal(getattr(a.stop, name), getattr(b.stop, name)), name


PATHS = {                                    # name -> (R, directed, flags, symmetric attention, K, d)
    "sym_fl_K5d32": (1, False, 0, True, 5, 32),
    "fl": (1, False, _lib.DL_F_NO_SYM, False, 5, 32),
    "stream": (1, False, _lib.DL_F_NO_FL, False, 3, 32),
    "generic": (1, False, _lib.DL_F_NO_STREAM, False, 3, 32),
    "directed": (1, True, 0, False, 3, 32),
    "runs3_sym": (3, False, 0, True, 5, 32),
    "runs3_directed": (3, True, 0, False, 3, 32),
}


@pytest.mark.parametrize("path", list(PATHS))
def test_replay_equals_eager(path):
    R, directed, flags, sym, K, d = PATHS[path]
    ei, N, beta, T = _cora()
    runs = RunSet(ei, N, list(range(R)), m=2, directed=directed)
    runs.graph.flags = flags
    if sym:
        runs.graph.sym_min_nnz = 0
    x = _features(N)
    eager, cap = _pair(runs, x, R, K, d, beta, T, chunk=5)
    if sym:
        assert cap.plan["mode"] == "sym"
    rows_e = eager.step(5)
    rows_c = cap.step(5)
    _assert_same_state(eager, cap)
    assert np.array_equal(np.array(rows_e), np.array(rows_c), equal_nan=True)
    assert all(np.isfinite(r[0]) for r in rows_c)


def test_two_replays_from_one_state_are_equal():
    ei, N, beta, T = _cora()
    runs = RunSet(ei, N, [0], m=2)
    _, cap = _pair(runs, _features(N), 1, 3, 32, beta, T, chunk=4)
    saved = cap._state()
    a = cap.step(3)
    cap._restore(saved)
    cap.epoch = 0
    b = cap.step(3)
    assert a == b


def test_weights_loaded_in_place_are_read_by_the_next_replay():
    ei, N, beta, T = _cora()
    runs = RunSet(ei, N, [0], m=2)
    x = _features(N)
    eager, cap = _pair(runs, x, 1, 3, 32, beta, T, chunk=2)
    fresh, _ = _pair(runs, x, 1, 3, 32, beta, T, chunk=2)
    other = _model(1, 3, 32, seed=7).state_dict()
    eager.model.load_state_dict(other)
    cap.model.load_state_dict(other)
    ours, theirs, orig = cap.step(2), eager.step(2), fresh.step(2)
    assert ours == theirs
    assert ours[0][0] != orig[0][0]
    _assert_same_state(eager, cap)


def _check_stopped_runs(eager, cap, epochs, chunk):
    a, b = eager.run(epochs), cap.run(epochs)
    assert len(a["history"]) == len(b["history"])
    for ha, hb in zip(a["history"], b["history"]):                           # NaN AUCs compare equal here
        assert np.array_equal(np.array(ha, dtype=float).reshape(-1, 2), np.array(hb, dtype=float).reshape(-1, 2),
                              equal_nan=True)
    assert a["best_val_auc"] == b["best_val_auc"] and a["test_auc"] == b["test_auc"] and a["epochs"] == b["epochs"]
    for pa, pb in zip(eager.model.parameters(), cap.model.parameters()):     # restored best weights
        assert torch.equal(_bits(pa), _bits(pb))
    longest = max(len(h) for h in b["history"])
    assert b["epochs"] == min(epochs, -(-longest // chunk) * chunk)          # ends at the chunk boundary after
    return b


@pytest.mark.parametrize("labels", ["random", "one_class"])
def test_single_run_stops_inside_a_chunk(labels):
    ei, N, beta, T = _cora()
    runs = RunSet(ei, N, [0], m=2)
    g = torch.Generator(device=DEV).manual_seed(5)
    if labels == "random":                   # validation AUC that stops improving
        runs.val_labels = (torch.rand(runs.val.P, device=DEV, generator=g) < 0.5).float()
    else:                                    # NaN AUC: never an improvement, stops at epoch patience
        runs.val_labels = torch.zeros(runs.val.P, device=DEV)
    eager, cap = _pair(runs, _features(N), 1, 3, 32, beta, T, chunk=8, patience=2, lr=0.05)
    init = [p.detach().clone() for p in cap.model.parameters()]
    out = _check_stopped_runs(eager, cap, 64, 8)
    n = len(out["history"][0])
    assert n < 64
    if labels == "one_class":
        assert n == 3 and out["best_val_auc"] == [0.0]
        assert all(torch.equal(p, q) for p, q in zip(cap.model.parameters(), init))


def test_runs_stop_independently_inside_a_chunk():
    ei, N, beta, T = _cora()
    runs = RunSet(ei, N, [0, 1, 2], m=2)
    vp = runs.val_ptr.tolist()
    runs.val_labels[vp[1]:vp[2]] = 0.0       # run 1: one class, NaN AUC, stops at epoch 3
    eager, cap = _pair(runs, _features(N), 3, 3, 32, beta, T, chunk=8, patience=3)
    out = _check_stopped_runs(eager, cap, 24, 8)
    lens = [len(h) for h in out["history"]]
    assert lens[1] == 4 and max(lens[0], lens[2]) > 4, lens                   # the others keep training
    assert out["best_val_auc"][1] == 0.0 and cap.stop.stale[1].item() == 4      # frozen after its stop
    init = _model(3, 3, 32)                                  # run 1 never improved: restored to its initial weights
    assert all(torch.equal(p[1], q[1]) for p, q in zip(cap.model.parameters(), init.parameters()))


def test_refused_before_capture():
    ei, N, beta, T = _cora()
    runs = RunSet(ei, N, [0], m=2)
    x = _features(N)
    m = _model(1, 3, 32)
    adam = torch.optim.Adam(m.parameters(), lr=0.01, capturable=True)
    args = (runs.train, runs.train_labels, runs.train_weights, runs.val, runs.val_labels, runs.test,
            runs.test_labels, beta, T)
    with pytest.raises(RuntimeError, match="dense x"):
        CapturedEpoch(m, adam, x.to_sparse(), runs.graph, *args)
    g = runs.graph
    rank_local = Graph(g.rowptr, g.col, g.N, n_global=2 * g.N)
    with pytest.raises(RuntimeError, match="whole graph"):
        CapturedEpoch(m, adam, x, rank_local, *args)
    with pytest.raises(RuntimeError, match="capturable"):
        CapturedEpoch(m, torch.optim.Adam(m.parameters(), lr=0.01), x, g, *args)
    score = torch.rand(64, device=DEV)
    lab = (torch.arange(64, device=DEV) % 2).float()
    graph = torch.cuda.CUDAGraph()
    with pytest.raises(RuntimeError, match="cannot be captured"):
        with torch.cuda.graph(graph):
            score.mul(2.0)
            ops.roc_auc(score, lab)


# ---- examples/train_link.py --------------------------------------------------------------------------------
@pytest.mark.parametrize("extra", [[], ["--run", "3"], ["--directed"], ["--run", "3", "--directed"]])
def test_example_capture(extra):
    cmd = [sys.executable, os.path.join(ROOT, "examples", "train_link.py"), "--dataset", "synthetic",
           "--capture", "10", "--epochs", "30", "--nhidden", "64"] + extra
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    assert "test auc" in out.stdout


def test_captured_loop_against_the_default_eager_loops():
    """20 epochs: the captured loop (capturable Adam: bias correction on the device) against run() and
    run_batched(R = 3) with the default Adam, on test_gpu_runs.py's synthetic graph and shapes; best validation
    and test AUC within the 0.02 that test uses."""
    import train_link
    x, ei, _ = train_link.synthetic(n=2000, seed=0)
    args = argparse.Namespace(nfactor=4, nhidden=64, nembed=16, beta=0.7, temperature=1, m=2, lr=0.01, epochs=20,
                              seed=3, log_every=1000, standardize=True, run=1, capture=None)
    quiet = lambda *_: None                                                # noqa: E731
    drift = []
    for R in (1, 3):
        ref = []
        for capture in (None, 10):
            torch.manual_seed(args.seed)
            a = argparse.Namespace(**{**vars(args), "run": R, "capture": capture})
            out = (train_link.run if R == 1 else train_link.run_batched)(a, x, ei, torch.device(DEV), log=quiet)
            ref.append(out["runs"] if R > 1 else [out])
        for r, (e, c) in enumerate(zip(*ref)):
            assert len(c["history"]) == len(e["history"]) == 20
            d = (abs(e["best_val_auc"] - c["best_val_auc"]), abs(e["test_auc"] - c["test_auc"]))
            drift.append(d)
            assert max(d) <= 0.02, (R, r, e["best_val_auc"], c["best_val_auc"], e["test_auc"], c["test_auc"])
    print("captured vs eager (best val AUC, test AUC) differences: " +
          ", ".join(f"{a:.2e}/{b:.2e}" for a, b in drift))
