"""Times the training epoch run eagerly against the same epoch replayed as a CUDA graph (disenlink_b200/capture.py,
examples/train_link.py --capture E), per epoch, on one GPU.

    python tools/capture_bench.py [--runs 1,10] [--epochs 50] [--warmup 5] [--rounds 3] [--out FILE]

Graphs and shapes are those of tools/runs_bench.py: the train edge columns stored in tests/golden used as the full
edge set (85/10/5 split, m = 5), random binary bag-of-words features at Cora's density; Cora K = 3, nhid 512,
d = 32 and the tuned K = 10, nhid 256, d = 64; chameleon K = 5, nhid 512, d = 32; squirrel K = 5, nhid 512,
d = 64.  R = 1 trains a Disentangle, R > 1 a DisentangleRuns over a RunSet union.  Every leg uses Adam with
capturable=True and does the whole epoch: projection, fused loss forward + backward, Adam, per-run losses,
validation AUC, stopping update, the record row.

  eager        the epoch's ops launched one by one, one device-to-host copy of the record per epoch
  captured_1   one graph replay and one copy per epoch (E = 1)
  captured_50  fifty replays, then one copy of the fifty records (E = 50)

Each leg runs --warmup epochs, then --epochs epochs between two device synchronisations (host clock); the legs
alternate for --rounds rounds in one process and the median per-epoch time is reported.  capture_ms is the time
CapturedEpoch's constructor spends on the warm-up epoch and the capture.  Prints one JSON object with the card's
name, power limit and max SM clock read in the same run; writes only the --out file.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "examples"))
import train_link  # noqa: E402
from runs_bench import WORKLOADS, gpu_info, load_graph  # noqa: E402
from disenlink_b200.capture import CapturedEpoch  # noqa: E402
from disenlink_b200.model import Disentangle  # noqa: E402
from disenlink_b200.runs import RunSet  # noqa: E402

LEGS = (("eager", False, 1), ("captured_1", True, 1), ("captured_50", True, 50))


def ms_per_epoch(ce: CapturedEpoch, n: int) -> float:
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    done = 0
    while done < n:
        k = min(ce.chunk, n - done)
        ce.step(k)
        done += k
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / n * 1e3


def bench_workload(wl, runs_list, a, dev):
    ei, N, beta, T = load_graph(wl["golden"], dev)
    gx = torch.Generator().manual_seed(0)
    x = (torch.rand(N, wl["F"], generator=gx) < 0.0127).float().to(dev)     # bag-of-words density of Cora
    args = argparse.Namespace(nfactor=wl["K"], nhidden=wl["nhid"], nembed=wl["d"], beta=beta, temperature=T, m=5,
                              lr=0.01)
    res = {"N": N, "edge_columns": int(ei.shape[1]), "F": wl["F"], "K": wl["K"], "nhid": wl["nhid"], "d": wl["d"],
           "by_R": {}}
    for R in runs_list:
        seeds = list(range(R))
        union = RunSet(ei, N, seeds, args.m)
        legs = {}
        for name, capture, chunk in LEGS:
            if R == 1:
                torch.manual_seed(0)
                model = Disentangle(wl["F"], wl["nhid"], wl["d"], nfactor=wl["K"], beta=beta, t=T).to(dev)
                ptrs = {}
            else:
                model = train_link.batched_model(args, wl["F"], seeds).to(dev)
                ptrs = dict(train_ptr=union.train_ptr, val_ptr=union.val_ptr, test_ptr=union.test_ptr)
            opt = torch.optim.Adam(model.parameters(), lr=args.lr, weight_decay=5e-4, capturable=True)
            torch.cuda.synchronize()
            legs[name] = CapturedEpoch(model, opt, x, union.graph, union.train, union.train_labels,
                                       union.train_weights, union.val, union.val_labels, union.test,
                                       union.test_labels, beta, T, patience=10**9, chunk=chunk, capture=capture,
                                       **ptrs)
        for ce in legs.values():
            ms_per_epoch(ce, a.warmup)
        times = {name: [] for name in legs}
        for _ in range(a.rounds):
            for name, ce in legs.items():
                times[name].append(ms_per_epoch(ce, a.epochs))
        med = {name: float(np.median(t)) for name, t in times.items()}
        row = {"union_nnz": union.graph.nnz, "train_pairs": union.train.P, "val_pairs": union.val.P}
        for name in legs:
            row[f"{name}_ms_per_epoch"] = round(med[name], 3)
            row[f"{name}_ms_all"] = [round(t, 3) for t in times[name]]
        row["speedup_1"] = round(med["eager"] / med["captured_1"], 2)
        row["speedup_50"] = round(med["eager"] / med["captured_50"], 2)
        row["capture_ms"] = round(legs["captured_50"].capture_s * 1e3, 1)
        # epochs after which the capture has paid for itself at E = 50 (None: it does not pay)
        gain = med["eager"] - med["captured_50"]
        row["break_even_epochs"] = round(row["capture_ms"] / gain) if gain > 0 else None
        res["by_R"][str(R)] = row
        print(json.dumps({wl["golden"]: {str(R): row}}), file=sys.stderr)
        del union, legs
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", default="1,10")
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--epochs", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("capture_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    runs_list = [int(r) for r in a.runs.split(",")]
    out = {"gpu": gpu_info(), "epochs": a.epochs, "warmup": a.warmup, "rounds": a.rounds, "workloads": {}}
    for name in a.workloads.split(","):
        out["workloads"][name] = bench_workload(WORKLOADS[name], runs_list, a, dev)
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
