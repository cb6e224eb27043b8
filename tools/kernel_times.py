"""Per-kernel device time of the single-GPU PartitionedLinkStep, from torch.profiler (CUDA activities).

    python tools/kernel_times.py --workload mid [--steps 3] [--warmup 1] [--out FILE.json]

Builds bench.py's workload (same generators, same seeds), runs `warmup` untimed steps, then profiles `steps`
steps and prints one line per kernel name: total milliseconds per step, launches per step, and for the two
kernels of the symmetric backward pass 2 (phase A k_bwd_edges_fl on the primary view, phase B k_bwd_sym_lower
on the secondary view) nanoseconds per entry of their view.  bench.py's "bwd_edges" phase is phase A +
phase B (+ their small carry fix-ups); "attn_fwd" is k_attn_fl + k_sym_expand (+ fix-ups).  Run it in a
process of its own: tracing slows the host, so its step times are not the benchmark's.
"""
import argparse
import json
import os
import re
import sys
from collections import defaultdict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")   # as bench.py on one GPU

import bench  # noqa: E402


def short_name(name: str) -> str:
    """Kernel name without the anonymous namespace, argument list and return type."""
    name = re.sub(r"\(anonymous namespace\)::", "", name)
    name = re.sub(r"^void ", "", name)
    depth, out = 0, []
    for ch in name:                          # drop the trailing "(...)" argument list, keep template args
        if ch == "(" and depth == 0 and out:
            break
        depth += ch == "<"
        depth -= ch == ">"
        out.append(ch)
    return "".join(out).strip()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workload", default="mid", choices=list(bench.WORKLOADS))
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the table as JSON here")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
    from disenlink_b200 import _lib
    from disenlink_b200.partition import PartitionedLinkStep

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    _lib.lib()
    wl = bench.WORKLOADS[args.workload]
    N, E, K, d, P, beta, T = (wl[k] for k in ("N", "E", "K", "d", "P", "beta", "T"))
    src, dst = bench.gen_edges(N, E, 0, dev)
    u, v, lab, wts = bench.gen_pairs_from_edges(src, dst, N, E, P, dev)
    step = PartitionedLinkStep(src, dst, N, u, v, lab, wts, K, d, beta, T, world=1, rank=0, device=dev)
    del src, dst
    torch.cuda.empty_cache()
    bench.gen_Z(step.part.n_local, K, d, 0, dev, row0=step.part.lo, out=step.Z_own)
    for _ in range(args.warmup):
        step.run()
    torch.cuda.synchronize(dev)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.steps):
            step.run()
        torch.cuda.synchronize(dev)

    tot, cnt = defaultdict(float), defaultdict(int)
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA and ev.device_time_total > 0:
            nm = short_name(ev.name)
            tot[nm] += ev.device_time_total / 1e3          # us -> ms
            cnt[nm] += 1
    plan = step.plan_bwd or {}
    n_entries = {"k_bwd_edges_fl": plan["upper"].nnz if plan.get("mode") == "sym" else step.graph.nnz,
                 "k_bwd_sym_lower": plan["lower"].nnz if plan.get("mode") == "sym" else 0}
    rows = []
    for nm in sorted(tot, key=lambda k: -tot[k]):
        ms = tot[nm] / args.steps
        base = nm.split("<")[0]
        per = n_entries.get(base)
        rows.append({"kernel": nm, "ms_per_step": round(ms, 4), "launches_per_step": cnt[nm] / args.steps,
                     "entries": per, "ns_per_entry": round(ms * 1e6 / per, 4) if per else None})
    props = torch.cuda.get_device_properties(dev)
    head = {"workload": args.workload, "device": props.name, "nnz": step.graph.nnz, "steps": args.steps,
            "pass2_mode": plan.get("mode"), "a_kept": bool(plan.get("mode") == "sym" and
                                                           not (step.graph.flags & _lib.DL_F_NO_KEEPA)),
            "DL_FLAGS": os.environ.get("DL_FLAGS", "")}
    print(json.dumps(head))
    print(f"{'ms/step':>10} {'launch':>6} {'ns/entry':>9}  kernel")
    for r in rows:
        npe = f"{r['ns_per_entry']:9.4f}" if r["ns_per_entry"] is not None else " " * 9
        print(f"{r['ms_per_step']:10.4f} {r['launches_per_step']:6.1f} {npe}  {r['kernel']}")
    a = [r for r in rows if r["kernel"].startswith("k_bwd_edges_fl")]
    b = [r for r in rows if r["kernel"].startswith("k_bwd_sym_lower")]
    if a and b and a[0]["ns_per_entry"] and b[0]["ns_per_entry"]:
        print(f"phase A / phase B time per entry: {a[0]['ns_per_entry'] / b[0]['ns_per_entry']:.3f}")
    if args.out:
        with open(args.out, "w") as f:
            json.dump({**head, "kernels": rows}, f, indent=1)
    step.close()


if __name__ == "__main__":
    main()
