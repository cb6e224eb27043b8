"""Host side of the captured epoch (disenlink_b200/capture.py) without a GPU: the chunk bookkeeping of
run_chunks driven by a fake record source, and examples/train_link.py's --capture argument."""
import os
import sys

import pytest

from disenlink_b200.capture import run_chunks

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples"))


class FakeRecords:
    """Epoch e of run r: loss 100 r + e, AUC e / 1000, best AUC = AUC, stop flag from epoch stop[r] on."""

    def __init__(self, stop, chunk):
        self.stop, self.chunk, self.epoch, self.calls = stop, chunk, 0, []

    def __call__(self, n):
        assert 1 <= n <= self.chunk
        self.calls.append(n)
        R = len(self.stop)
        rows = []
        for e in range(self.epoch, self.epoch + n):
            rows.append([100.0 * r + e for r in range(R)] + [e / 1000] * R + [e / 1000] * R +
                        [float(s is not None and e >= s) for s in self.stop])
        self.epoch += n
        return rows


def test_history_ends_at_each_runs_stop_epoch():
    src = FakeRecords(stop=[3, None, 10], chunk=4)
    history, done = run_chunks(src, epochs=20, chunk=4, R=3)
    assert [len(h) for h in history] == [4, 20, 11]
    assert history[0][-1] == (3.0, 0.003)
    assert history[2] == [(200.0 + e, e / 1000) for e in range(11)]
    assert done == 20 and src.calls == [4] * 5


def test_ends_at_the_first_chunk_boundary_after_every_run_stopped():
    src = FakeRecords(stop=[2, 5], chunk=4)
    history, done = run_chunks(src, epochs=100, chunk=4, R=2)
    assert done == 8 and src.calls == [4, 4]
    assert [len(h) for h in history] == [3, 6]


def test_partial_last_chunk():
    src = FakeRecords(stop=[None], chunk=8)
    history, done = run_chunks(src, epochs=19, chunk=8, R=1)
    assert src.calls == [8, 8, 3] and done == 19
    assert [a for _, a in history[0]] == [e / 1000 for e in range(19)]


def test_stop_in_the_last_epoch_of_a_chunk():
    src = FakeRecords(stop=[7], chunk=8)
    history, done = run_chunks(src, epochs=40, chunk=8, R=1)
    assert done == 8 and len(history[0]) == 8


def test_capture_argument():
    import train_link
    assert train_link.parse_args([]).capture is None
    assert train_link.parse_args(["--capture", "50", "--run", "3"]).capture == 50
    for bad in ("0", "-2"):
        with pytest.raises(SystemExit):
            train_link.parse_args(["--capture", bad])
