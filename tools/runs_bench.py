"""Times R independent runs trained one after another against the same R runs trained together as one union
(disenlink_b200/runs.py, examples/train_link.py --run R), per epoch, on one GPU.

    python tools/runs_bench.py [--runs 1,2,4,10] [--epochs 30] [--warmup 5] [--rounds 3] [--out FILE]

Graphs: the train edge columns stored in tests/golden (Cora, chameleon, squirrel; the datasets themselves are
not shipped), used as the full edge set of the script's protocol (85/10/5 split, m = 5 negative rounds).
Features are random binary bag-of-words rows (seeded) with the datasets' widths and Cora's density.  Shapes:
Cora at K = 3, d = 32 (nhid 512) and at the tuned K = 10, nhid = 256, d = 64; chameleon K = 5, nhid = 512,
d = 32; squirrel K = 5, nhid = 512, d = 64.

  sequential  R single-run epochs as examples/train_link.py's run() makes them: projection, fused loss forward +
              backward, Adam, validation scores, roc_auc, with its two host syncs (loss.item(), the AUC)
  batched     one epoch of examples/train_link.py's batched_epoch over the union: the same steps for all runs,
              plus the per-run losses, segmented AUC and stopping update, one device-to-host copy
Each leg runs --warmup epochs, then --epochs epochs between two device synchronisations; the legs alternate for
--rounds rounds and the median per-epoch time is reported.  Also timed, at R = 10 on every graph: one
roc_auc_segments call against 10 roc_auc_stats calls over the same validation pairs (CUDA events, median of 50).
Prints one JSON object with the card's name and power limit read in the same run; writes only the --out file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "examples"))
import train_link  # noqa: E402
from disenlink_b200 import ops  # noqa: E402
from disenlink_b200.model import Disentangle  # noqa: E402
from disenlink_b200.runs import EarlyStopping, RunSet  # noqa: E402

WORKLOADS = {
    "cora_k3": dict(golden="cora_K3_d32", F=1433, K=3, nhid=512, d=32),
    "cora_tuned": dict(golden="cora_K3_d32", F=1433, K=10, nhid=256, d=64),
    "chameleon": dict(golden="chameleon_K5_d32", F=2325, K=5, nhid=512, d=32),
    "squirrel": dict(golden="squirrel_K8_d16", F=2089, K=5, nhid=512, d=64),
}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def load_graph(name, dev):
    g = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
    ei = torch.stack([torch.as_tensor(g["src"].astype(np.int64)), torch.as_tensor(g["dst"].astype(np.int64))])
    return ei.to(dev), int(g["N"]), float(g["beta"]), float(g["T"])


def ms_per_epoch(fn, n):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / n * 1e3


def event_ms(fn, reps=50):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts))


def bench_workload(name, wl, runs_list, a, dev):
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
        bmodel = train_link.batched_model(args, wl["F"], seeds).to(dev)
        bopt = torch.optim.Adam(bmodel.parameters(), lr=args.lr, weight_decay=5e-4)
        stop = EarlyStopping(list(bmodel.parameters()), patience=200)
        singles = []
        for s in seeds:
            rs = RunSet(ei, N, [s], args.m)
            torch.manual_seed(s)
            m = Disentangle(wl["F"], wl["nhid"], wl["d"], nfactor=wl["K"], beta=beta, t=T).to(dev)
            singles.append((rs, m, torch.optim.Adam(m.parameters(), lr=args.lr, weight_decay=5e-4)))

        def sequential():
            for rs, m, opt in singles:                    # run()'s epoch body, examples/train_link.py
                Z = m.project(x)
                loss, _, H = ops.link_bce_loss(Z, rs.graph, rs.train, rs.train_labels, rs.train_weights, beta, T)
                opt.zero_grad()
                loss.backward()
                opt.step()
                _, vp = ops.pair_score_fwd(Z.detach(), H, rs.val, T, want_logit=False)
                ops.roc_auc_stats(vp, rs.val_labels).tolist()     # = ops.roc_auc without its NaN / one-class raise
                loss.item()

        def batched():
            train_link.batched_epoch(args, x, union, bmodel, bopt, stop)

        ms_per_epoch(sequential, a.warmup)
        ms_per_epoch(batched, a.warmup)
        seq_ms, bat_ms = [], []
        for _ in range(a.rounds):
            seq_ms.append(ms_per_epoch(sequential, a.epochs))
            bat_ms.append(ms_per_epoch(batched, a.epochs))
        seq, bat = float(np.median(seq_ms)), float(np.median(bat_ms))
        row = {"union_nnz": union.graph.nnz, "train_pairs": union.train.P, "val_pairs": union.val.P,
               "sequential_ms_per_epoch": round(seq, 3), "batched_ms_per_epoch": round(bat, 3),
               "speedup": round(seq / bat, 2), "sequential_ms_all": [round(t, 3) for t in seq_ms],
               "batched_ms_all": [round(t, 3) for t in bat_ms]}
        if R == 10:
            with torch.no_grad():
                Z = bmodel.project(x)
                H = ops.factor_aggregate(Z, union.graph, beta, T)
                _, val_scores = ops.pair_score_fwd(Z, H, union.val, T, want_logit=False)
            seg_ms = event_ms(lambda: ops.roc_auc_segments(val_scores, union.val_labels, union.val_ptr))
            bounds = union.val_ptr.tolist()
            pieces = [(val_scores[bounds[r]:bounds[r + 1]], union.val_labels[bounds[r]:bounds[r + 1]]) for r in range(R)]
            sep_ms = event_ms(lambda: [ops.roc_auc_stats(s, l) for s, l in pieces])
            row["auc_segments_ms"] = round(seg_ms, 4)
            row["auc_stats_x10_ms"] = round(sep_ms, 4)
        res["by_R"][str(R)] = row
        print(json.dumps({name: {str(R): row}}), file=sys.stderr)
        del union, bmodel, bopt, stop, singles
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", default="1,2,4,10")
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--epochs", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("runs_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    runs_list = [int(r) for r in a.runs.split(",")]
    out = {"gpu": gpu_info(), "epochs": a.epochs, "warmup": a.warmup, "rounds": a.rounds, "workloads": {}}
    for name in a.workloads.split(","):
        out["workloads"][name] = bench_workload(name, WORKLOADS[name], runs_list, a, dev)
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
