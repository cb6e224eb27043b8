"""Times the first layer of the factor MLPs from sparse bag-of-words features (SparseFeatures, csrc/feat_proj.cu)
against the dense SGEMM and torch.sparse.mm, alone and inside the captured training epoch, on one GPU.

    python tools/sparse_features_bench.py [--iters 20] [--epochs 50] [--rounds 3] [--out FILE]

  layer   forward + weight gradient of relu(x W1^T + b1) (autograd.grad with a fixed cotangent), three ways:
          dense (torch.addmm, SGEMM), torch_sparse (torch.sparse.mm on a COO x) and sparse_kernels
          (ops.feature_projection, Wt = W1^T made contiguous inside the timed call as the model does).  Widths J =
          K nhid R: Cora K=3 nhid 512 (1536) and the tuned K=10 nhid 256 (2560), at R = 1 and R = 10.  Inputs:
          binary rows at Cora's shape and density (2708 x 1433, 1.27 %) with Zipf column popularity, and a denser
          one at Pubmed's shape (19717 x 500, 10 %, uniform).  CUDA events around --iters calls after warm-up,
          implementations alternating for --rounds rounds, median.  gathered_GBps = the 2 nnz J 4 bytes of Wt and
          G' rows the kernels gather, over their time; wt_fits_l2 = F J 4 bytes below the 126 MB of L2.
  epoch   capture_bench.ms_per_epoch of the captured epoch (E = 50) with dense x against SparseFeatures of the
          same x, on capture_bench's Cora workloads (uniform binary features at 1.27 %) at R = 1 and R = 10;
          plus the max abs / relative difference of Z and of every parameter gradient of Z.backward(C) (one fixed
          cotangent C) between the two paths, from the same initial weights.
Prints one JSON object with the card's name, power limit and max SM clock read in the same run; writes only the
--out file.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch
import torch.nn.functional as Fn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "examples"))

L2_BYTES = 126e6
SHAPES = {"cora_k3": 1536, "cora_tuned": 2560, "cora_k3_R10": 15360, "cora_tuned_R10": 25600}
INPUTS = {"cora_zipf_1.27pct": dict(N=2708, F=1433, density=0.0127, zipf=1.0),
          "pubmed_shape_10pct": dict(N=19717, F=500, density=0.10, zipf=0.0)}


def zipf_bag_of_words(N, F, density, s=1.0, cap=0.5, seed=0):
    """Binary [N, F] with column f present in a row with probability min(cap, c (rank f)^-s) (ranks shuffled over
    the columns), c set so that the expected density is `density`.  s = 0: uniform."""
    g = torch.Generator().manual_seed(seed)
    w = (torch.arange(F, dtype=torch.float64) + 1.0) ** -s
    w = w[torch.randperm(F, generator=g)]
    lo, hi = 0.0, 1.0 / float(w.min())
    for _ in range(100):                                   # bisection on c
        c = 0.5 * (lo + hi)
        lo, hi = (c, hi) if float(torch.clamp(c * w, max=cap).mean()) < density else (lo, c)
    p = torch.clamp(0.5 * (lo + hi) * w, max=cap).float()
    return (torch.rand(N, F, generator=g) < p).float()


def event_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def bench_layer(a, dev):
    from disenlink_b200 import ops
    from disenlink_b200.features import SparseFeatures
    out = {}
    for iname, spec in INPUTS.items():
        x = zipf_bag_of_words(spec["N"], spec["F"], spec["density"], s=spec["zipf"]).to(dev)
        feats = SparseFeatures.from_dense(x)
        xs = x.to_sparse().coalesce()
        N, F, nnz = spec["N"], spec["F"], feats.nnz
        for sname, J in SHAPES.items():
            g = torch.Generator(device=dev).manual_seed(1)
            W1 = (torch.randn(J, F, device=dev, generator=g) / F ** 0.5).requires_grad_()
            b = (0.1 * torch.randn(J, device=dev, generator=g)).requires_grad_()
            C = torch.randn(N, J, device=dev, generator=g)

            def dense():
                torch.autograd.grad(Fn.relu(torch.addmm(b, x, W1.t())), (W1, b), C)

            def torch_sparse():
                torch.autograd.grad(Fn.relu(torch.sparse.mm(xs, W1.t()) + b), (W1, b), C)

            def kernels():
                A = ops.feature_projection(feats, W1.t().contiguous(), b, relu=True)
                torch.autograd.grad(A, (W1, b), C.view(1, N, J))

            legs = {"dense": dense, "torch_sparse": torch_sparse, "sparse_kernels": kernels}
            for fn in legs.values():
                for _ in range(3):
                    fn()
            torch.cuda.synchronize()
            times = {k: [] for k in legs}
            for _ in range(a.rounds):
                for k, fn in legs.items():
                    times[k].append(event_ms(fn, a.iters))
            med = {k: float(np.median(v)) for k, v in times.items()}
            row = {"N": N, "F": F, "J": J, "nnz": nnz, "density": round(nnz / (N * F), 5),
                   "n_heavy_columns": feats.n_heavy, "wt_MB": round(F * J * 4 / 1e6, 1),
                   "wt_fits_l2": F * J * 4 < L2_BYTES}
            for k in legs:
                row[f"{k}_ms"] = round(med[k], 4)
                row[f"{k}_ms_all"] = [round(t, 4) for t in times[k]]
            row["dense_TFLOPs"] = round(4 * N * F * J / (med["dense"] * 1e-3) / 1e12, 2)
            row["sparse_kernels_gathered_GBps"] = round(2 * nnz * J * 4 / (med["sparse_kernels"] * 1e-3) / 1e9, 1)
            row["speedup_vs_dense"] = round(med["dense"] / med["sparse_kernels"], 2)
            row["speedup_vs_torch_sparse"] = round(med["torch_sparse"] / med["sparse_kernels"], 2)
            out[f"{iname}/{sname}"] = row
            print(json.dumps({f"{iname}/{sname}": row}), file=sys.stderr)
            del W1, b, C
            torch.cuda.empty_cache()
    return out


def _diff(a, b):
    d = float((a - b).abs().max())
    return {"max_abs": d, "max_rel": d / max(float(b.abs().max()), 1e-30)}


def bench_epoch(a, dev):
    import train_link
    from capture_bench import ms_per_epoch
    from runs_bench import WORKLOADS, load_graph
    from disenlink_b200.capture import CapturedEpoch
    from disenlink_b200.features import SparseFeatures
    from disenlink_b200.model import Disentangle
    from disenlink_b200.runs import RunSet
    out = {}
    for name in ("cora_k3", "cora_tuned"):
        wl = WORKLOADS[name]
        ei, N, beta, T = load_graph(wl["golden"], dev)
        gx = torch.Generator().manual_seed(0)
        x = (torch.rand(N, wl["F"], generator=gx) < 0.0127).float().to(dev)   # capture_bench's features
        feats = SparseFeatures.from_dense(x)
        args = argparse.Namespace(nfactor=wl["K"], nhidden=wl["nhid"], nembed=wl["d"], beta=beta, temperature=T, m=5,
                                  lr=0.01)
        for R in (1, 10):
            seeds = list(range(R))
            union = RunSet(ei, N, seeds, args.m)

            def fresh_model():
                if R == 1:
                    torch.manual_seed(0)
                    return Disentangle(wl["F"], wl["nhid"], wl["d"], nfactor=wl["K"], beta=beta, t=T).to(dev)
                return train_link.batched_model(args, wl["F"], seeds).to(dev)

            # differences of the two paths from the same (initial) weights
            model = fresh_model()
            g = torch.Generator(device=dev)
            res = {}
            for leg, xin in (("dense_x", x), ("sparse_features", feats)):
                model.zero_grad(set_to_none=True)
                Z = model.project(xin)
                C = torch.randn(Z.shape, device=dev, generator=g.manual_seed(2))
                Z.backward(C)
                res[leg] = (Z.detach(), {n: p.grad.clone() for n, p in model.named_parameters()})
            diffs = {"diff_Z": _diff(res["sparse_features"][0], res["dense_x"][0]),
                     "diff_grad": {n: _diff(res["sparse_features"][1][n], res["dense_x"][1][n]) for n in res["dense_x"][1]}}
            del model, res
            legs = {}
            for leg, xin in (("dense_x", x), ("sparse_features", feats)):
                model = fresh_model()
                ptrs = {} if R == 1 else dict(train_ptr=union.train_ptr, val_ptr=union.val_ptr, test_ptr=union.test_ptr)
                opt = torch.optim.Adam(model.parameters(), lr=args.lr, weight_decay=5e-4, capturable=True)
                legs[leg] = CapturedEpoch(model, opt, xin, union.graph, union.train, union.train_labels,
                                          union.train_weights, union.val, union.val_labels, union.test,
                                          union.test_labels, beta, T, patience=10**9, chunk=50, **ptrs)
            for ce in legs.values():
                ms_per_epoch(ce, a.warmup)
            times = {k: [] for k in legs}
            for _ in range(a.rounds):
                for k, ce in legs.items():
                    times[k].append(ms_per_epoch(ce, a.epochs))
            med = {k: float(np.median(v)) for k, v in times.items()}
            row = {f"{k}_ms_per_epoch": round(med[k], 3) for k in legs}
            row.update({f"{k}_ms_all": [round(t, 3) for t in times[k]] for k in legs})
            row["speedup"] = round(med["dense_x"] / med["sparse_features"], 2)
            row.update(diffs)
            out[f"{name}/R{R}"] = row
            print(json.dumps({f"{name}/R{R}": row}), file=sys.stderr)
            del union, legs, model
            torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--epochs", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--parts", default="layer,epoch")
    ap.add_argument("--out", default=None, help="also write the JSON here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sparse_features_bench.py needs a CUDA device")
    from runs_bench import gpu_info
    dev = torch.device("cuda:0")
    out = {"gpu": gpu_info(), "iters": a.iters, "epochs": a.epochs, "warmup": a.warmup, "rounds": a.rounds}
    parts = a.parts.split(",")
    if "layer" in parts:
        out["layer"] = bench_layer(a, dev)
    if "epoch" in parts:
        out["epoch"] = bench_epoch(a, dev)
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
