"""Times the directed backward (ops.factor_bwd_directed, csrc/bwd_dir.cu) against the symmetric backward
(ops.factor_bwd) on one GPU, on bench.py's graph generator at C4 size (N = 2 923 922, 13 975 788 edge columns,
K = 8, d = 16 by default).

    python tools/directed_bench.py [--workload c4] [--reps 10] [--out FILE]

Three backward calls, each after one forward (attention + aggregation) on the same Z and G:
  sym        the symmetrised graph, unmarked: the symmetric backward (pass 1 + one-sided pass 2)
  marked     the same symmetric pattern marked directed: the directed backward
  one_way    a graph with the same nnz and no reciprocal entry (every edge column oriented one way), marked
Reported per case: ms (CUDA events, median of --reps calls after 2 warm-up calls), the algorithmic bytes of
the backward in DESIGN.md section 4's terms (every gather counted at full size, no cache credit) and their
rate as a fraction of the copy bandwidth measured in the same run (a 4 GiB device-to-device copy).  After the
timed calls, one more call per case runs under torch.profiler (CUDA activity only) and the per-kernel device
times are reported ("kernels_ms"), so the directed passes can be compared with the symmetric ones entry for
entry (e.g. the in-side of pass 2, which recomputes the softmax, against the symmetric phase B, which reads it).
Prints one JSON object; writes only the --out file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (graph and Z generators, the symmetric backward's algorithmic bytes)
from disenlink_b200 import ops  # noqa: E402
from disenlink_b200.graph import Graph  # noqa: E402


def directed_bytes(nnz, N, K, d):
    """Algorithmic bytes of the directed backward: mask, pass 1 (in-view), pass 2 out-side, pass 2 in-side."""
    D = K * d
    return {
        "mask": nnz * 1 + N * 4 + 8 * (N + 1),
        "pass1": nnz * (4 + 4 + 1 + 4 + 4 * d) + N * (16 * D + 8 * K + 4) + 8 * (N + 1),
        "pass2_out": nnz * (4 + 1 + 4 * D + 4 + 4) + N * (16 * D + 4 * K) + 8 * (N + 1),
        "pass2_in": nnz * (4 + 4 + 1 + 4 + 4 * D) + N * 12 * D + 8 * (N + 1),
    }


def one_way_edges(N, nnz, seed, device, max_rounds=64):
    """nnz distinct (src, dst) columns of the same power-law generator, no self-loops, none whose reverse is
    present: each unordered pair is oriented by the parity of src + dst.  The generator repeats pairs often
    (hub endpoints), so batches of nnz draws are added until nnz distinct pairs exist."""
    key = torch.empty(0, dtype=torch.int64, device=device)
    for rnd in range(max_rounds):
        src, dst = bench.gen_edges(N, nnz, seed + 17 + 1000 * rnd, device)
        keep = src != dst
        lo, hi = torch.minimum(src[keep], dst[keep]), torch.maximum(src[keep], dst[keep])
        key = torch.unique(torch.cat([key, lo * N + hi]))
        del src, dst, keep, lo, hi
        if key.numel() >= nnz:
            break
    else:
        raise SystemExit(f"one-way generator produced {key.numel()} edges after {max_rounds} rounds, {nnz} needed")
    g = torch.Generator(device=device).manual_seed(seed + 18)
    key = key[torch.randperm(key.numel(), generator=g, device=device)[:nnz]]
    lo, hi = key // N, key % N
    flip = ((lo + hi) & 1) == 1
    return torch.where(flip, hi, lo), torch.where(flip, lo, hi)


def timed(fn, reps):
    for _ in range(2):
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
    ts.sort()
    return ts[len(ts) // 2], ts


def copy_peak_gbs(device, reps=10):
    n = 1 << 30                                                           # 4 GiB of fp32 each way
    a = torch.empty(n, dtype=torch.float32, device=device).fill_(1.0)
    b = torch.empty_like(a)
    ms, _ = timed(lambda: b.copy_(a), reps)
    del a, b
    return 2 * 4 * n / (ms * 1e-3) / 1e9


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def kernel_times(fn):
    """Device time per kernel name (ms) of one call of fn, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0.0)
        if t > 0:
            out[ev.key[:120]] = round(t / 1e3, 3)
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c4", choices=["c4", "c4k5", "c4k5d64", "tiny"])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None, help="also write the JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("directed_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    wl = bench.WORKLOADS[args.workload]
    N, E, K, d, beta, T = wl["N"], wl["E"], wl["K"], wl["d"], wl["beta"], wl["T"]
    src, dst = bench.gen_edges(N, E, args.seed, dev)
    Z = bench.gen_Z(N, K, d, args.seed, dev)
    G = bench.gen_Z(N, K, d, args.seed + 5, dev)
    graphs = {
        "sym": Graph.from_edges(src, dst, N),
        "marked": Graph.from_edges(src, dst, N, symmetrize=True, directed=True),
    }
    nnz = graphs["sym"].nnz
    a, b = one_way_edges(N, nnz, args.seed, dev)
    graphs["one_way"] = Graph.from_edges(a, b, N, directed=True)
    del src, dst, a, b
    peak = copy_peak_gbs(dev)
    out = {"gpu": gpu_info(), "workload": args.workload, "N": N, "K": K, "d": d, "copy_peak_GBps": round(peak, 1),
           "cases": {}}
    sym_b = bench.alg_bytes(nnz, N, K, d, 0)
    for name, g in graphs.items():
        kstar, w, s = ops.edge_attn_fwd(g, Z, T)
        dZ = torch.zeros_like(Z)
        if g.directed:
            g.transpose_view()
            fn = lambda g=g, kstar=kstar, w=w, s=s: ops.factor_bwd_directed(g, Z, G, kstar, w, s, beta, T, dZ=dZ.zero_())
            byts = sum(directed_bytes(g.nnz, N, K, d).values())
        else:
            fn = lambda g=g, kstar=kstar, w=w, s=s: ops.factor_bwd(g, Z, G, kstar, w, s, beta, T, dZ=dZ.zero_())
            byts = sym_b["bwd_gather"] + sym_b["bwd_edges"]
        ms, ts = timed(fn, args.reps)
        tg = g.transpose_view()[0] if g.directed else None
        out["cases"][name] = {
            "nnz": g.nnz, "ms": round(ms, 3), "ms_all": [round(x, 3) for x in ts], "alg_bytes": int(byts),
            "alg_GBps": round(byts / (ms * 1e-3) / 1e9, 1), "frac_of_copy_peak": round(byts / (ms * 1e-3) / 1e9 / peak, 4),
            "max_out_degree": int(g.degrees().max().item()),
            "max_in_degree": int(tg.degrees().max().item()) if tg is not None else None,
            "dZ_absmax": float(dZ.abs().max().item()), "dZ_finite": bool(torch.isfinite(dZ).all().item()),
            "kernels_ms": kernel_times(fn),
        }
        del kstar, w, s
    out["ratio_marked_over_sym"] = round(out["cases"]["marked"]["ms"] / out["cases"]["sym"]["ms"], 3)
    out["ratio_one_way_over_sym"] = round(out["cases"]["one_way"]["ms"] / out["cases"]["sym"]["ms"], 3)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
