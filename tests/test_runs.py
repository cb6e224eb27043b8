"""Batched independent runs (disenlink_b200/runs.py) on the CPU: the stacked projection against each run's own
Disentangle, the per-run state dicts, per-run gradients of the summed losses, and the per-run early stopping
against a plain restatement of main_disentangled.py's rule."""
import math

import pytest
import torch

from disenlink_b200.model import Disentangle
from disenlink_b200.runs import DisentangleRuns, EarlyStopping

F_, NHID, D, K = 37, 12, 8, 3


def _models(R, seed0=0):
    out = []
    for r in range(R):
        torch.manual_seed(seed0 + r)
        out.append(Disentangle(F_, NHID, D, K, 0.7, 1))
    return out


def test_project_matches_each_run():
    models = _models(4)
    runs = DisentangleRuns.from_models(models)
    x = torch.randn(50, F_)
    Z = runs.project(x)
    assert Z.shape == (4 * 50, K, D)
    for r, m in enumerate(models):
        ref = m.project(x)
        got = Z[r * 50:(r + 1) * 50]
        assert (got - ref).abs().max() <= 1e-6 * ref.abs().max()


def test_project_sparse_x():
    models = _models(2)
    runs = DisentangleRuns.from_models(models)
    x = torch.randn(30, F_) * (torch.rand(30, F_) < 0.1)
    Z = runs.project(x.to_sparse())
    for r, m in enumerate(models):
        ref = m.project(x)
        assert (Z[r * 30:(r + 1) * 30] - ref).abs().max() <= 1e-6 * ref.abs().max()


def test_state_dict_round_trip():
    models = _models(3, seed0=10)
    runs = DisentangleRuns.from_models(models)
    for r, m in enumerate(models):
        sd = runs.run_state_dict(r)
        ref = m.state_dict()
        assert list(sd.keys()) == list(ref.keys())
        for k in ref:
            assert torch.equal(sd[k], ref[k]), k
        fresh = Disentangle(F_, NHID, D, K, 0.7, 1)
        fresh.load_state_dict(sd, strict=True)
    other = DisentangleRuns(F_, NHID, D, K, 0.7, 1, runs=3)
    for r in range(3):
        other.load_run_state_dict(r, models[r].state_dict())
    for a, b in zip(other.parameters(), runs.parameters()):
        assert torch.equal(a, b)
    bad = dict(models[0].state_dict())
    bad.pop("factor_0.mlp1.bias")
    with pytest.raises(KeyError):
        other.load_run_state_dict(0, bad)


def test_from_models_leaves_rng_and_default_init_matches_sequential_models():
    torch.manual_seed(5)
    a = DisentangleRuns(F_, NHID, D, K, 0.7, 1, runs=2)
    torch.manual_seed(5)
    seq = [Disentangle(F_, NHID, D, K, 0.7, 1) for _ in range(2)]
    for r in range(2):
        for k, v in seq[r].state_dict().items():
            assert torch.equal(a.run_state_dict(r)[k], v)
    torch.manual_seed(7)
    DisentangleRuns.from_models(seq)
    after = torch.rand(4)
    torch.manual_seed(7)
    assert torch.equal(after, torch.rand(4))


def test_nhid_one_refused():
    with pytest.raises(ValueError):
        DisentangleRuns(F_, 1, D, K, 0.7, 1, runs=2)


def test_gradients_of_summed_losses_are_per_run():
    models = _models(3, seed0=20)
    runs = DisentangleRuns.from_models(models)
    x = torch.randn(40, F_)
    C = torch.randn(3, 40, K, D)
    Z = runs.project(x).view(3, 40, K, D)
    (torch.tanh(Z) * C).sum().backward()
    for r, m in enumerate(models):
        (torch.tanh(m.project(x)) * C[r]).sum().backward()
        h = NHID
        for i, f in enumerate(m.factors):
            pairs = [(runs.W1.grad[r, i * h:(i + 1) * h], f.mlp1.weight.grad),
                     (runs.b1.grad[r, i * h:(i + 1) * h], f.mlp1.bias.grad),
                     (runs.W2.grad[r, i], f.mlp2.weight.grad), (runs.b2.grad[r, i], f.mlp2.bias.grad)]
            for got, want in pairs:
                assert (got - want).abs().max() <= 1e-5 * want.abs().max()


# ---- early stopping ---------------------------------------------------------------------------------------
def _script_rule(aucs, patience):
    """main_disentangled.py's loop for one run: -> (best_auc, stale, epoch of the last snapshot, stop epoch)."""
    best, stale, snap, stop = 0.0, 0, None, None
    for e, auc in enumerate(aucs):
        if auc > best:
            best, stale, snap = auc, 0, e
        else:
            stale += 1
        if stale > patience:
            stop = e
            break
    return best, stale, snap, stop


@pytest.mark.parametrize("patience", [0, 2, 3])
def test_early_stopping_matches_script_rule(patience):
    nan = math.nan
    seqs = [
        [0.5, 0.6, 0.6, 0.6, 0.6, 0.6, 0.7, 0.7, 0.7, 0.7, 0.7, 0.7],       # ties are no improvement
        [nan, 0.4, nan, nan, 0.5, 0.45, 0.45, 0.9, nan, nan, nan, nan],     # NaN is no improvement
        [0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9, 0.91, 0.92, 0.93],    # never stops
        [0.9, 0.1, 0.1, 0.1, 0.95, 0.1, 0.1, 0.1, 0.1, 0.1, 0.1, 0.99],     # stops before the late best
        [0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0],       # never improves on 0
    ]
    R, T = len(seqs), len(seqs[0])
    W = torch.zeros(R, 3, 2)                      # a stacked "parameter": run r's slice holds the epoch number
    b = torch.zeros(R, 5)
    es = EarlyStopping([W, b], patience=patience)
    snap_epoch = [None] * R
    stopped_at = [None] * R
    for e in range(T):
        W.fill_(float(e))
        b.fill_(float(-e))
        before = es.snapshot[0].clone()
        es.update(torch.tensor([s[e] for s in seqs], dtype=torch.float64))
        for r in range(R):
            if stopped_at[r] is not None:         # frozen: the snapshot no longer changes
                assert torch.equal(es.snapshot[0][r], before[r])
            if not torch.equal(es.snapshot[0][r], before[r]):
                snap_epoch[r] = e
            if es.stopped[r] and stopped_at[r] is None:
                stopped_at[r] = e
    for r, s in enumerate(seqs):
        best, stale, snap, stop = _script_rule(s, patience)
        assert es.best_auc[r].item() == best, r
        assert es.stale[r].item() == stale, r
        assert stopped_at[r] == stop, r
        if snap is None:                          # never improved: the initial weights stay
            assert torch.equal(es.snapshot[0][r], torch.zeros(3, 2))
        else:
            assert torch.equal(es.snapshot[0][r], torch.full((3, 2), float(snap)))
            assert torch.equal(es.snapshot[1][r], torch.full((5,), float(-snap)))
    es.restore()
    assert torch.equal(W, es.snapshot[0]) and torch.equal(b, es.snapshot[1])


def test_early_stopping_runs_stop_at_different_epochs():
    es = EarlyStopping([torch.zeros(3, 1)], patience=1)
    stops = []
    for e, aucs in enumerate([(0.5, 0.5, 0.5), (0.4, 0.6, 0.6), (0.4, 0.4, 0.7), (0.4, 0.4, 0.4), (0.9, 0.9, 0.4)]):
        es.update(torch.tensor(aucs, dtype=torch.float64))
        stops.append(es.stopped.tolist())
    assert stops[2] == [True, False, False]
    assert stops[3] == [True, True, False]
    assert stops[4] == [True, True, True]
    assert es.best_auc.tolist() == [0.5, 0.6, 0.7]          # the late 0.9 reaches no stopped run
