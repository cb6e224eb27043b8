"""Parity of DirectedPartitionedLinkStep on G GPUs with the same step on one GPU, over two steps (Z changed in
between), on bench.py's generator (power-law degrees: in- and out-hubs).

    python -m torch.distributed.run --nproc-per-node G tools/directed_partition_parity.py [--workload tiny] [--out FILE]

Every rank also runs the world-1 step on its own GPU with the same inputs and compares its owned part:
  integers   kstar of the own entries and of the record tail, the routed-mask-driven r == 0 pattern: bitwise
  halo       Z rows of the halo against the owners' rows: bitwise
  records    w and dw (own prefix and tail) against the one-GPU entries: bitwise count and max relative error
  floats     s, r, dZ of the owned rows, prob and loss: bitwise share and max |diff| / max |one GPU|
The directed kernels walk a row the same way on a rank-local graph (hub segments depend on the degree only), so
everything downstream of identical attention outputs is bitwise equal; the attention's s may differ in the last
bits where the streaming kernels cut ranges at other places of a smaller graph.  Rank 0 prints one JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from directed_partition_bench import build_step, gpu_info  # noqa: E402


def cmp(a, b):
    a, b = a.reshape(-1), b.reshape(-1)
    if a.numel() == 0:
        return {"n": 0, "bitwise": True, "share_equal": 1.0, "max_rel": 0.0}
    if a.dtype == torch.float32:
        eq = a.view(torch.int32) == b.view(torch.int32)
        rel = float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))
    else:
        eq = a == b
        rel = 0.0
    return {"n": int(a.numel()), "bitwise": bool(eq.all()), "share_equal": round(float(eq.float().mean()), 6),
            "max_rel": rel}


def compare(step, one, n):
    lo, hi, n_own, nnz = step.part.lo, step.part.hi, step.n_own, step.graph.nnz
    dev = step.Z.device
    e0, e1 = int(one.graph.rowptr[lo]), int(one.graph.rowptr[hi])
    gid = torch.cat([torch.arange(lo, hi, device=dev), step.plan.halo])
    # global CSR index of every tail record
    tperm = step.tperm.long()
    j = torch.repeat_interleave(torch.arange(n_own, device=dev), step.tgraph.rowptr[1:] - step.tgraph.rowptr[:-1]) + lo
    i = gid[step.tgraph.col.long()]
    rows1 = torch.repeat_interleave(torch.arange(n, device=dev), one.graph.rowptr[1:] - one.graph.rowptr[:-1])
    key1 = rows1 * n + one.graph.col.long()
    tail = tperm >= nnz
    tail_glob = torch.empty(step.n_tail, dtype=torch.int64, device=dev)
    tail_glob[tperm[tail] - nnz] = torch.searchsorted(key1, i[tail] * n + j[tail])
    rec = torch.cat([torch.arange(e0, e1, device=dev), tail_glob])
    n_rec = nnz + step.n_tail
    P = step.P
    return {
        "kstar": cmp(step.kstar[:n_rec], one.kstar[rec]),
        "r_zero_pattern": cmp((step.r[:n_own] == 0).to(torch.uint8), (one.r[lo:hi] == 0).to(torch.uint8)),
        "Z_halo": cmp(step.Z[n_own:], one.Z[step.plan.halo]),
        "w": cmp(step.w[:n_rec], one.w[rec]),
        "dw": cmp(step.dw[:n_rec], one.dw[rec]),
        "s": cmp(step.s[:n_own], one.s[lo:hi]),
        "r": cmp(step.r[:n_own], one.r[lo:hi]),
        "dZ": cmp(step.dZ, one.dZ[lo:hi]),
        "prob": cmp(step.prob[:P], one.prob[:P]),
        "loss": cmp(step.loss.reshape(1), one.loss.reshape(1)),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="tiny", choices=list(bench.WORKLOADS))
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
    step = build_step(wl, args.seed, dev, world, rank)
    one = build_step(wl, args.seed, dev, 1, 0)
    res = {}
    for k in range(2):
        if k == 1:                                         # the second step: another Z
            bench.gen_Z(step.n_own, wl["K"], wl["d"], args.seed + 11, dev, row0=step.part.lo, out=step.Z_own)
            bench.gen_Z(one.n_own, wl["K"], wl["d"], args.seed + 11, dev, row0=0, out=one.Z_own)
        step.run()
        one.run()
        torch.cuda.synchronize()
        res[f"step{k + 1}"] = compare(step, one, wl["N"])
    mine = {"rank": rank, "n_own": step.n_own, "n_halo": step.plan.n_halo, "n_tail": step.n_tail,
            "peer_push": bool(step.pushed), **res}
    ranks = [None] * world
    if world > 1:
        dist.all_gather_object(ranks, mine)
    else:
        ranks = [mine]
    step.close()
    one.close()
    if rank == 0:
        summary = {}
        for s_ in ("step1", "step2"):
            for k in ranks[0][s_]:
                summary[f"{s_}.{k}.bitwise"] = all(r[s_][k]["bitwise"] for r in ranks)
                summary[f"{s_}.{k}.max_rel"] = max(r[s_][k]["max_rel"] for r in ranks)
        out = {"gpu": gpu_info(), "gpus": world, "workload": args.workload, "summary": summary, "ranks": ranks}
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
