"""Times DirectedPartitionedLinkStep (training on directed edge columns, node-partitioned) on bench.py's graph
generator, one process per GPU.

    python -m torch.distributed.run --nproc-per-node G tools/directed_partition_bench.py [--workload c4] \\
        [--steps 5] [--warmup 2] [--out FILE]

Every rank builds the same edge columns (bench.gen_edges, same seed), the same pair batch and its own rows of Z
(bench.gen_Z).  After --warmup steps, --steps steps are timed with CUDA events at every phase boundary of the
step (its `mark` hook: ag_Z, attn_fwd, ag_s, ag_rec = the kstar and w record pushes, spmm_fwd, ... , bwd_gather =
pass 1, bwd_out = pass 2 out-side, ag_dw = the dw record push, bwd_in = pass 2 in-side).  Per phase the mean over
the timed steps is reported for the slowest rank (a phase ends for everyone with the barrier of the next push)
and per rank; with it the exchange volume per rank, record bytes included.  Rank 0 prints one JSON line (and
appends it to --out).  The card name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from disenlink_b200.partition import DirectedPartitionedLinkStep  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def make_inputs(wl, seed, device):
    """-> (src, dst, u, v, labels, weights): the same on every rank."""
    N, E, P = wl["N"], wl["E"], wl["P"]
    src, dst = bench.gen_edges(N, E, seed, device)
    g = torch.Generator(device=device).manual_seed(seed + 3)
    u = torch.randint(0, N, (P,), generator=g, device=device)
    v = torch.randint(0, N, (P,), generator=g, device=device)
    lab = (torch.rand(P, generator=g, device=device) < 0.2).float()
    wts = torch.full((P,), 1.0 / P, device=device)
    return src, dst, u, v, lab, wts


def build_step(wl, seed, device, world, rank, mark=None):
    src, dst, u, v, lab, wts = make_inputs(wl, seed, device)
    step = DirectedPartitionedLinkStep(src, dst, wl["N"], u, v, lab, wts, wl["K"], wl["d"], wl["beta"], wl["T"],
                                       world=world, rank=rank, device=device, mark=mark)
    del src, dst, u, v, lab, wts
    bench.gen_Z(step.n_own, wl["K"], wl["d"], seed, device, row0=step.part.lo, out=step.Z_own)
    return step


class Marks:
    def __init__(self):
        self.on, self.ev = False, []

    def __call__(self, name):
        if self.on:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            self.ev.append((name, e))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c4", choices=list(bench.WORKLOADS))
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    wl = bench.WORKLOADS[args.workload]
    marks = Marks()
    t0 = time.perf_counter()
    step = build_step(wl, args.seed, dev, world, rank, mark=marks)
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t0
    for _ in range(args.warmup):
        step.run()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    marks.on = True
    for _ in range(args.steps):
        step.run()
    torch.cuda.synchronize()
    phases, total = {}, 0.0
    per_step = [marks.ev[i:i + len(marks.ev) // args.steps] for i in range(0, len(marks.ev), len(marks.ev) // args.steps)]
    for ev in per_step:
        for (a, ea), (b, eb) in zip(ev[:-1], ev[1:]):
            phases[b] = phases.get(b, 0.0) + ea.elapsed_time(eb) / args.steps
        total += ev[0][1].elapsed_time(ev[-1][1]) / args.steps
    vol = step.exchange_volume()
    vol.update(record_bytes_out=vol["record_bytes_out_fwd"] + vol["record_bytes_out_bwd"], nnz_own=step.graph.nnz,
               in_entries=step.tgraph.nnz, peer_push=bool(step.pushed))
    mine = {"rank": rank, "phases_ms": {k: round(x, 3) for k, x in phases.items()}, "step_ms": round(total, 3),
            "volume": vol, "setup_s": round(setup_s, 1)}
    ranks = [None] * world
    if world > 1:
        dist.all_gather_object(ranks, mine)
    else:
        ranks = [mine]
    step.close()
    if rank == 0:
        names = list(ranks[0]["phases_ms"])
        out = {"gpu": gpu_info(), "gpus": world, "workload": args.workload, "N": wl["N"], "E": wl["E"], "P": wl["P"],
               "K": wl["K"], "d": wl["d"], "steps": args.steps, "warmup": args.warmup,
               "step_ms_max": max(r["step_ms"] for r in ranks),
               "phases_ms_max": {k: max(r["phases_ms"][k] for r in ranks) for k in names},
               "ranks": ranks}
        line = json.dumps(out)
        print(line, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "a") as f:
                f.write(line + "\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
