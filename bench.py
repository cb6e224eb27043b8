#!/usr/bin/env python
"""bench.py -- factor-aggregation edges/s (fwd+bwd) and link-pair scores/s on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c5|c6|c4|c4k5|c4k5d64|mid|tiny] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over the whole graph and pair batch:
    attention -> aggregation -> pair scoring -> BCE gradient -> decoder backward -> factor backward
`value` = nnz / (t_attention + t_aggregation + t_factor_backward)  [edges/s, BASELINE.json metric],
with inputs resident in HBM; per-kernel CUDA-event times and the HBM roofline of the dominant
kernel are reported next to it.  `e2e` runs the same pass through the public autograd API
(`ops.link_bce_loss` + backward) with Z copied from pinned host memory and the loss / scores read
back every step.  `cpu_baseline` times the CPU oracle (a port of the reference's math, the dense
reference itself cannot run at these sizes) on a bounded sample on the box's host cores.
N > 1 (torchrun): the same graph is node-partitioned across the ranks (strong scaling) with NCCL
all-gathers between the kernels (disenlink_b200/partition.py).
"""
import argparse
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# c5 keeps ~160 GB of 25.6-GB tensors live: let the caching allocator map segments instead of carving
# fixed blocks, or fragmentation alone (26 GiB "reserved but unallocated") runs the device out of memory
# (one GPU only: expandable segments cannot be exported with CUDA IPC, which the multi-GPU exchange needs)
if int(os.environ.get("WORLD_SIZE", "1")) == 1:
    os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")

WORKLOADS = {
    # BASELINE.json configs[4]: synthetic power-law graph 50M nodes / 500M edges, K=8, D=128, 100M pairs
    "c5": dict(N=50_000_000, E=500_000_000, K=8, d=16, P=100_000_000, beta=0.5, T=1.0,
               name="synthetic power-law 50M nodes / 500M directed edges, K=8, d=16 (D=128), 100M link pairs"),
    # 1.6 x c5: the node arrays alone (4 x 41 GB) exceed one B200 -- only runs node-partitioned (--gpus 8)
    "c6": dict(N=80_000_000, E=800_000_000, K=8, d=16, P=100_000_000, beta=0.5, T=1.0,
               name="synthetic power-law 80M nodes / 800M directed edges, K=8, d=16 (does not fit one GPU)"),
    # BASELINE.json configs[3] scale: snap-patents-sized synthetic
    "c4": dict(N=2_923_922, E=13_975_788, K=8, d=16, P=16_000_000, beta=0.5, T=1.0,
               name="snap-patents-scale synthetic 2.92M nodes / 13.98M directed edges, K=8, d=16"),
    "c4k5": dict(N=2_923_922, E=13_975_788, K=5, d=32, P=16_000_000, beta=0.5, T=1.0,
                 name="snap-patents-scale synthetic 2.92M nodes / 13.98M directed edges, K=5, d=32"),
    "c4k5d64": dict(N=2_923_922, E=13_975_788, K=5, d=64, P=16_000_000, beta=0.5, T=1.0,
                    name="snap-patents-scale synthetic 2.92M nodes / 13.98M directed edges, K=5, d=64"),
    "mid": dict(N=5_000_000, E=50_000_000, K=8, d=16, P=10_000_000, beta=0.5, T=1.0,
                name="synthetic power-law 5M nodes / 50M directed edges, K=8, d=16 (1/10 of c5)"),
    "tiny": dict(N=200_000, E=2_000_000, K=8, d=16, P=400_000, beta=0.5, T=1.0,
                 name="synthetic power-law 200k nodes / 2M directed edges (smoke)"),
}
CPU_SAMPLE = dict(N=5_000_000, E=50_000_000, P=10_000_000)   # 1/10 of c5 (= the "mid" workload), same generator:
#                                                              ~20 s of oracle time on 16 host threads, ~15 GB of host RAM
M_NEG = 5
POWER = 3.0   # endpoint rank ~ N * U^3  ->  degree(rank) ~ rank^(-2/3), degree exponent alpha = 2.5


# ------------------------------------------------------------------------------------------------
# synthetic inputs (torch ops; same code on cpu and cuda)
# ------------------------------------------------------------------------------------------------
def gen_edges(N, E, seed, device):
    import torch
    g = torch.Generator(device=device).manual_seed(seed)
    src = torch.empty(E, dtype=torch.int64, device=device)
    dst = torch.empty(E, dtype=torch.int64, device=device)
    A, B = 7919, 104729   # affine node-id shuffle (A coprime to N) so hubs are spread over the id range
    while math.gcd(A, N) != 1:
        A += 2
    chunk = 1 << 26
    for out in (src, dst):
        for a in range(0, E, chunk):
            b = min(E, a + chunk)
            u = torch.rand(b - a, generator=g, device=device, dtype=torch.float64)
            ids = (u.pow_(POWER) * N).to(torch.int64).clamp_(max=N - 1)
            out[a:b] = (ids * A + B) % N
    return src, dst


def gen_pairs(rowptr, col, N, P, seed, device):
    """P = P_pos * (1 + M_NEG): positives drawn from CSR entries, M_NEG uniform negatives sharing u
    with each positive (main_disentangled.py:159-163), sorted by u."""
    import torch
    g = torch.Generator(device=device).manual_seed(seed + 1)
    nnz = int(col.numel())
    P_pos = max(P // (1 + M_NEG), 1)
    e = torch.randint(0, max(nnz, 1), (P_pos,), generator=g, device=device)
    pu = torch.searchsorted(rowptr, e, right=True) - 1
    pv = col[e].to(torch.int64)
    nu = pu.repeat(M_NEG)
    nv = torch.randint(0, N, (P_pos * M_NEG,), generator=g, device=device)
    u = torch.cat([pu, nu])
    v = torch.cat([pv, nv])
    lab = torch.cat([torch.ones(P_pos, device=device), torch.zeros(P_pos * M_NEG, device=device)])
    wts = torch.cat([torch.full((P_pos,), 1.0 / P_pos, device=device),
                     torch.full((P_pos * M_NEG,), 1.0 / (M_NEG * P_pos * M_NEG), device=device)])
    order = torch.sort(u, stable=True).indices
    return u[order], v[order], lab[order], wts[order]


Z_CHUNK = 1 << 22


def gen_Z(n_rows, K, d, seed, device, row0=0, out=None):
    """Rows [row0, row0 + n_rows) of the synthetic factor embeddings.  Every block of Z_CHUNK rows has its
    own generator seed, so a rank of a node-partitioned run draws exactly the rows it owns and they are
    the rows a single-GPU run draws."""
    import torch
    Z = out if out is not None else torch.empty(n_rows, K, d, dtype=torch.float32, device=device)
    scale = d ** -0.25                                                      # q = O(1)
    c0, c1 = row0 // Z_CHUNK, (row0 + n_rows + Z_CHUNK - 1) // Z_CHUNK
    for c in range(c0, c1):
        g = torch.Generator(device=device).manual_seed((seed + 2) * 1_000_003 + c)
        blk = torch.randn(Z_CHUNK, K, d, generator=g, device=device)
        a, b = max(row0, c * Z_CHUNK), min(row0 + n_rows, (c + 1) * Z_CHUNK)
        Z[a - row0:b - row0] = blk[a - c * Z_CHUNK:b - c * Z_CHUNK] * scale
        del blk
    return Z


# ------------------------------------------------------------------------------------------------
# algorithmic bytes (SURVEY.md section 8d)
# ------------------------------------------------------------------------------------------------
def alg_bytes(nnz, N, K, d, P):
    D = K * d
    return {
        "attn_fwd": nnz * (4 + 4 * D + 5) + N * (4 * D + 4 * K) + 8 * (N + 1),
        "spmm_fwd": nnz * (4 + 5 + 4 + 4 * d) + N * (8 * D + 4 * K) + 8 * (N + 1),
        "bwd_gather": nnz * (9 + 4 * d) + N * (12 * D + 8 * K) + 8 * (N + 1),
        "bwd_edges": nnz * (17 + 4 * D + 4 * d) + N * (12 * D + 8 * K) + 8 * (N + 1),
        "pair_fwd": P * (16 * D + 12),
        "pair_bwd": P * (32 * D + 16),
    }


# ------------------------------------------------------------------------------------------------
# clocks during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
               0x4: "sw_power_cap", 0x80: "hw_power_brake", 0x2: "applications_clocks_setting"}

    def __init__(self, index=0):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(
                    nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def start(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr is not None:
            self._thr.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port on a bounded sample (all host threads)
# ------------------------------------------------------------------------------------------------
def dense_reference_leg(device=None):
    """The reference's OWN dense path (baseline/_ref/model.py, unmodified, staged by
    tools/stage_reference.sh) timed on the host cores on the configs it can run -- chameleon
    (hyperparameters_setting:2: K=5, nhid=512, d=32, beta=.7) and Cora (argparse defaults: K=3,
    nhid=512, d=32, beta=.9) -- next to this repository's module on the same x / adj_sym / weights on
    the GPU: model(x, adj_sym) forward and forward + backward of a BCE over all N^2 scores
    (model.py:105-114).  3 warm-up + 5 timed calls, median."""
    import numpy as np
    import torch
    import torch.nn.functional as F
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.exists(os.path.join(ref_dir, "model.py")):
        return {"unavailable": "baseline/_ref/model.py not staged (tools/stage_reference.sh needs /root/reference)"}
    import importlib.util
    spec = importlib.util.spec_from_file_location("_ref_model", os.path.join(ref_dir, "model.py"))
    refmodel = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(refmodel)
    from disenlink_b200 import data as dl_data
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    out = {"cores": threads, "what": "model(x, adj_sym) of the unmodified reference model.py on the host cores vs "
                                     "disenlink_b200.model.Disentangle on the same inputs on the GPU; 3 warm-up + 5 timed, median"}
    cases = []
    cham = os.path.join(ref_dir, "data_pre_false", "chameleon", "raw", "chameleon.npz")
    if os.path.exists(cham):
        x, ei, _ = dl_data.read_wikipedia_npz(cham)
        cases.append(("chameleon_K5_d32", dl_data.row_standardize(x), ei, dict(nhid=512, d=32, K=5, beta=0.7)))
    cora = os.path.join(ref_dir, "data", "cora", "raw")
    if os.path.exists(cora):
        x, ei, _ = dl_data.read_planetoid(cora, "cora")
        cases.append(("cora_K3_d32", x, ei, dict(nhid=512, d=32, K=3, beta=0.9)))

    def timed(fn, sync=None, warm=3, reps=5):
        ts = []
        for i in range(warm + reps):
            if sync:
                sync()
            t0 = time.perf_counter()
            fn()
            if sync:
                sync()
            if i >= warm:
                ts.append(time.perf_counter() - t0)
        return sorted(ts)[len(ts) // 2]

    for name, x, ei, hp in cases:
        n = x.shape[0]
        tr = dl_data.split_edges(ei.shape[1], seed=0)[0]            # main_disentangled.py:134-142
        adj = torch.zeros(n, n)
        adj[ei[0][tr], ei[1][tr]] = 1
        adj_sym = ((adj + adj.t()) != 0).float()
        nnz = int(adj_sym.sum().item())
        torch.manual_seed(0)
        ref = refmodel.Disentangle(x.shape[1], hp["nhid"], hp["d"], nfactor=hp["K"], beta=hp["beta"], t=1)

        def ref_fwd():
            with torch.no_grad():
                ref(x, adj_sym)

        def ref_fwd_bwd():
            ref.zero_grad()
            _, a = ref(x, adj_sym)
            F.binary_cross_entropy(a, adj_sym).backward()
        rec = {"N": n, "nnz_sym": nnz, **hp, "ref_cpu_fwd_ms": 1e3 * timed(ref_fwd), "ref_cpu_fwd_bwd_ms": 1e3 * timed(ref_fwd_bwd)}
        rec["ref_cpu_edges_per_s"] = nnz / (rec["ref_cpu_fwd_bwd_ms"] * 1e-3)
        if device is not None:
            from disenlink_b200.model import Disentangle
            ours = Disentangle(x.shape[1], hp["nhid"], hp["d"], nfactor=hp["K"], beta=hp["beta"], t=1)
            ours.load_state_dict(ref.state_dict(), strict=True)
            ours = ours.to(device)
            xg, ag = x.to(device), adj_sym.to(device)
            sync = lambda: torch.cuda.synchronize(device)

            def our_fwd():
                with torch.no_grad():
                    ours(xg, ag)

            def our_fwd_bwd():
                ours.zero_grad()
                _, a = ours(xg, ag)
                F.binary_cross_entropy(a, ag).backward()
            rec["gpu_fwd_ms"] = 1e3 * timed(our_fwd, sync)
            rec["gpu_fwd_bwd_ms"] = 1e3 * timed(our_fwd_bwd, sync)
            rec["gpu_edges_per_s"] = nnz / (rec["gpu_fwd_bwd_ms"] * 1e-3)
            with torch.no_grad():
                Hr, ar = ref(x, adj_sym)
                Ho, ao = ours(xg, ag)
            rec["max_abs_diff_link_pred"] = float((ao.cpu() - ar).abs().max())
            rec["max_rel_diff_H"] = float((Ho.cpu() - Hr).abs().max() / Hr.abs().max())
        out[name] = {k: ((round(v, 4) if abs(v) >= 1e-2 else float(f"{v:.3e}")) if isinstance(v, float) else v)
                     for k, v in rec.items()}
    return out


def cpu_baseline(K, d, beta, T, steps=2, warmup=1):
    import numpy as np
    import torch
    from oracle import oracle
    threads = os.cpu_count() or 1
    oracle.set_num_threads(threads)
    torch.set_num_threads(threads)     # torchrun exports OMP_NUM_THREADS=1: the (untimed) input generation would crawl
    cs = CPU_SAMPLE
    src, dst = gen_edges(cs["N"], cs["E"], 0, "cpu")
    rowptr, col = oracle.csr_from_edges(src.numpy(), dst.numpy(), cs["N"])
    u, v, lab, wts = gen_pairs(torch.from_numpy(rowptr), torch.from_numpy(col), cs["N"], cs["P"], 0, "cpu")
    Z = gen_Z(cs["N"], K, d, 0, "cpu").numpy()
    u, v, lab, wts = u.numpy(), v.numpy(), lab.numpy(), wts.numpy()
    nnz = int(col.size)
    t_factor, t_pair_fwd, t_all = [], [], []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        ks, w, s = oracle.edge_attn_fwd(rowptr, col, Z, T)
        H = oracle.factor_spmm_fwd(rowptr, col, Z, ks, w, s, beta)
        t1 = time.perf_counter()
        _, prob = oracle.pair_score_fwd(u, v, Z, H, T)
        t2 = time.perf_counter()
        dS = ((prob - lab) * wts).astype(np.float32)
        dZp, dH = oracle.pair_score_bwd(u, v, Z, H, dS, T)
        t3 = time.perf_counter()
        oracle.factor_bwd(rowptr, col, Z, dH, ks, w, s, beta, T, dZ_init=dZp)
        t4 = time.perf_counter()
        if it >= warmup:
            t_factor.append((t1 - t0) + (t4 - t3))
            t_pair_fwd.append(t2 - t1)
            t_all.append(t4 - t0)
    tf = sum(t_factor) / len(t_factor)
    return {"value": nnz / tf, "unit": "edges/s", "cores": threads, "kind": "port",
            "pair_scores_per_s": cs["P"] / (sum(t_pair_fwd) / len(t_pair_fwd)),
            "ms_per_step": 1e3 * sum(t_all) / len(t_all),
            "sample": f"same power-law generator at 1/10 scale: N={cs['N']}, E={cs['E']} directed edges "
                      f"(nnz={nnz}), P={cs['P']} pairs, K={K}, d={d}; {steps} timed steps after {warmup} "
                      f"warm-up; C oracle (oracle/disen_oracle.c, OpenMP, {threads} threads)"}


def run_reference(args):
    """--impl reference: the reference's own CPU math.  The dense model.py path needs
    (9K+6) N^2 4 bytes (121 GB already at N = 19 717), so on this arm's config it is the oracle port of
    the same math that is timed -- all host threads, bounded sample (1/10 scale); the unmodified dense
    model.py itself is timed where it can run (chameleon, Cora) and reported under "dense_reference"."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    cb = cpu_baseline(wl["K"], wl["d"], wl["beta"], wl["T"], steps=args.steps, warmup=args.warmup)
    line = {"impl": "reference", "metric": "factor-agg edges/s (fwd+bwd)", "value": cb["value"],
            "unit": "edges/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["name"], "K": wl["K"], "d": wl["d"]},
            "pair_scores_per_s": cb["pair_scores_per_s"],
            "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": cb["value"], "unit": "edges/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0}, "gpu_launches": 0,
            "dense_reference": dense_reference_leg(None)}
    emit(line)



# ------------------------------------------------------------------------------------------------
# the other BASELINE.json configs, measured the same way (device-timed phases, one GPU)
# ------------------------------------------------------------------------------------------------
def measure_config(name, src, dst, N, K, d, beta, dev, peak, steps=10, warmup=3, P=None, note=""):
    """One BASELINE config through the same PartitionedLinkStep as the headline workload (world = 1):
    -> {nnz, value (edges/s fwd+bwd), ms per phase, HBM roofline fraction on SURVEY's bytes}."""
    import torch
    from disenlink_b200.partition import PartitionedLinkStep
    E = int(src.numel())
    g = torch.Generator(device=dev).manual_seed(1)
    P_pos = max((P or min(E, 4_000_000)) // (1 + M_NEG), 1)
    e = torch.randint(0, E, (P_pos,), generator=g, device=dev)
    pu, pv = src[e], dst[e]
    u = torch.cat([pu, pu.repeat(M_NEG)])
    v = torch.cat([pv, torch.randint(0, N, (P_pos * M_NEG,), generator=g, device=dev)])
    lab = torch.cat([torch.ones(P_pos, device=dev), torch.zeros(P_pos * M_NEG, device=dev)])
    wts = torch.cat([torch.full((P_pos,), 1.0 / P_pos, device=dev),
                     torch.full((P_pos * M_NEG,), 1.0 / (M_NEG * P_pos * M_NEG), device=dev)])
    order = torch.sort(u, stable=True).indices
    u, v, lab, wts = u[order], v[order], lab[order], wts[order]
    events = []

    def mark(nm):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(torch.cuda.current_stream(dev))
        events.append((nm, ev))
    step = PartitionedLinkStep(src, dst, N, u, v, lab, wts, K, d, beta, 1.0, world=1, rank=0, device=dev, mark=mark)
    gen_Z(N, K, d, 0, dev, out=step.Z_own)
    for _ in range(warmup):
        step.run()
    torch.cuda.synchronize(dev)
    events.clear()
    for _ in range(steps):
        step.run()
    torch.cuda.synchronize(dev)
    ph = {p: 0.0 for p in PHASES}
    for (n0, e0), (n1, e1) in zip(events[:-1], events[1:]):
        if n1 != "begin":
            ph[n1] += e0.elapsed_time(e1)
    ph = {p: v / steps for p, v in ph.items()}
    nnz = step.graph.nnz
    t_factor = ph["attn_fwd"] + ph["spmm_fwd"] + ph["bwd_gather"] + ph["bwd_edges"]
    ab = alg_bytes(nnz, N, K, d, int(u.numel()))
    fb = ab["attn_fwd"] + ab["spmm_fwd"] + ab["bwd_gather"] + ab["bwd_edges"]
    out = {"N": int(N), "nnz": int(nnz), "K": K, "d": d, "P": int(u.numel()),
           "value_edges_per_s": nnz / (t_factor * 1e-3), "pair_scores_per_s": int(u.numel()) / (ph["pair_fwd"] * 1e-3),
           "ms": {k: round(ph[k], 4) for k in KERNEL_PHASES},
           "factor_agg_fwd_bwd": {"alg_bytes": int(fb), "GB/s": round(fb / (t_factor * 1e-3) / 1e9, 1),
                                  "frac": round(fb / (t_factor * 1e-3) / 1e9 / peak, 4)},
           "working_set": "exceeds L2" if N * K * d * 4 > 2 * 126e6 else "fits L2 (launch / latency bound: not roofline evidence)",
           "loss": float(step.loss.item())}
    if note:
        out["note"] = note
    del step
    torch.cuda.empty_cache()
    return out


def other_configs(dev, peak):
    """BASELINE.json configs[0..3] on one GPU: real graphs where the reference ships them (staged in
    baseline/_ref or committed as a fixture), synthetic snap-patents-scale otherwise."""
    import numpy as np
    import torch
    from disenlink_b200 import data as dl_data
    out = {}
    ref_dir = os.path.join(ROOT, "baseline", "_ref")

    def real(name, ei, N, shapes, note):
        tr = dl_data.split_edges(ei.shape[1], seed=0)[0]
        src, dst = ei[0][tr].to(dev), ei[1][tr].to(dev)
        for (K, d, beta) in shapes:
            try:
                out[f"{name}_K{K}_d{d}"] = measure_config(name, src, dst, N, K, d, beta, dev, peak, steps=20, note=note)
            except Exception as ex:                      # never lose the headline line to a side config
                out[f"{name}_K{K}_d{d}"] = {"error": repr(ex)[:200]}
    cora = os.path.join(ref_dir, "data", "cora", "raw")
    if os.path.exists(cora):
        _, ei, _ = dl_data.read_planetoid(cora, "cora")
        real("c1_cora", ei, 2708, [(3, 32, 0.9), (10, 64, 0.6)], "real Cora graph, 85 % train columns; Z ~ N(0, d^-1/2)")
    cham = os.path.join(ref_dir, "data_pre_false", "chameleon", "raw", "chameleon.npz")
    if os.path.exists(cham):
        x, ei, _ = dl_data.read_wikipedia_npz(cham)
        real("c2_chameleon", ei, int(x.shape[0]), [(5, 32, 0.7)], "real chameleon graph (72 202 stored columns)")
    sq = os.path.join(ref_dir, "data", "squirrel", "geom_gcn", "raw", "out1_graph_edges.txt")
    if os.path.exists(sq):
        e = torch.from_numpy(np.loadtxt(sq, skiprows=1, dtype=np.int64).T.copy())
        real("c2_squirrel", e, int(e.max()) + 1, [(5, 64, 0.5)], "real squirrel graph (hyperparameters_setting:3)")
    pm = os.path.join(ROOT, "tests", "golden", "pubmed_graph.npz")
    if os.path.exists(pm):
        gd = np.load(pm)
        ei = torch.from_numpy(np.stack([gd["src"], gd["dst"]]).astype(np.int64))
        real("c3_pubmed", ei, int(gd["N"]), [(8, 8, 0.6), (8, 64, 0.6)], "real Pubmed graph, K=8, both readings of d=64 (D=64, D=512)")
    for key, K, d in (("c4_K8_d16", 8, 16), ("c4_K5_d32", 5, 32), ("c4_K5_d64", 5, 64)):
        try:
            wl = WORKLOADS["c4"]
            src, dst = gen_edges(wl["N"], wl["E"], 0, dev)
            out[key] = measure_config(key, src, dst, wl["N"], K, d, 0.5, dev, peak, steps=10, P=wl["P"],
                                      note="snap-patents-scale synthetic power-law graph")
            del src, dst
        except Exception as ex:
            out[key] = {"error": repr(ex)[:200]}
    return out



def projection_bench(dev):
    """The factor projection X W (model.py:16-27,106; the one tensor-core contraction of the path) at the
    sizes of configs[0] and configs[2]: plain fp32 SGEMM against 3xTF32 on the tensor cores, accuracy
    against fp64."""
    import torch
    from disenlink_b200.model import Disentangle
    out = {}
    for name, (n, F_, nhid, d, K) in {"cora_F1433_K3_nhid512_d32": (2708, 1433, 512, 32, 3),
                                      "pubmed_F500_K8_nhid512_d64": (19717, 500, 512, 64, 8)}.items():
        torch.manual_seed(0)
        x = torch.randn(n, F_, device=dev)
        m = Disentangle(F_, nhid, d, nfactor=K, beta=0.5, t=1).to(dev)
        m64 = Disentangle(F_, nhid, d, nfactor=K, beta=0.5, t=1).double().to(dev)
        m64.load_state_dict({k: v.double() for k, v in m.state_dict().items()})
        with torch.no_grad():
            ref = m64.project(x.double())
        flops = 2.0 * n * F_ * K * nhid + 2.0 * n * K * nhid * d
        rec = {"N": n, "F": F_, "K": K, "nhid": nhid, "d": d, "gflop": round(flops / 1e9, 2)}
        for mode in ("fp32", "3xtf32"):
            m.projection = mode
            with torch.no_grad():
                for _ in range(3):
                    Z = m.project(x)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize(dev)
                a.record()
                for _ in range(10):
                    Z = m.project(x)
                b.record()
                torch.cuda.synchronize(dev)
            ms = a.elapsed_time(b) / 10
            rec[mode] = {"ms": round(ms, 4), "TFLOP/s": round(flops / (ms * 1e-3) / 1e12, 2),
                         "max_rel_err_vs_fp64": float((Z.double() - ref).abs().max() / ref.abs().max())}
        out[name] = rec
    return out

# ------------------------------------------------------------------------------------------------
# N > 1: the partitioned step against a single-GPU step on the same inputs (every rank checks its rows)
# ------------------------------------------------------------------------------------------------
def multi_gpu_parity(world, rank, dev, workload="mid"):
    import torch
    import torch.distributed as dist
    from disenlink_b200.partition import PartitionedLinkStep
    wl = WORKLOADS[workload]
    N, E, K, d, P, beta, T = (wl[k] for k in ("N", "E", "K", "d", "P", "beta", "T"))
    src, dst = gen_edges(N, E, 0, dev)
    u, v, lab, wts = gen_pairs_from_edges(src, dst, N, E, P, dev)
    part_step = PartitionedLinkStep(src, dst, N, u, v, lab, wts, K, d, beta, T, world=world, rank=rank, device=dev)
    lo, hi = part_step.part.lo, part_step.part.hi
    gen_Z(hi - lo, K, d, 0, dev, row0=lo, out=part_step.Z_own)
    # Two steps, Z changed in between (exchange ordering, ADVICE r1).  The compared step runs on Z / 4: with the
    # full-scale Z the hub rows of H reach |H| ~ 10^2, and their ABSOLUTE fp32 error (6e-7 relative, from range
    # cuts that depend on the partition) goes through exp(q) <H_u, H_v> into the scores of the many pairs that
    # have a hub endpoint -- |d prob| up to 8e-4 at 8 ranks with every forward quantity equal to 6e-7.
    for it in range(2):
        if it == 1:
            part_step.Z_own.mul_(0.25)
        part_step.run()
    # the single-GPU side runs the kernel paths a rank runs (two-sided attention and pass 2; the aggregation
    # pre-scaled or not as the ranks chose), so that what is compared is the partition and the exchange and not two
    # roundings of the same quantity -- the logits of this workload reach the hundreds and amplify those
    old_flags = os.environ.get("DL_FLAGS")
    os.environ["DL_FLAGS"] = "NO_SYM" + ("" if part_step.prescale else ",NO_PRESCALE")
    try:
        single = PartitionedLinkStep(src, dst, N, u, v, lab, wts, K, d, beta, T, world=1, rank=0, device=dev)
    finally:
        if old_flags is None:
            del os.environ["DL_FLAGS"]
        else:
            os.environ["DL_FLAGS"] = old_flags
    gen_Z(N, K, d, 0, dev, out=single.Z_own)
    single.Z_own.mul_(0.25)
    single.run()
    torch.cuda.synchronize(dev)
    e0, e1 = int(single.graph.rowptr[lo]), int(single.graph.rowptr[hi])
    nl = part_step.graph.nnz
    halo = part_step.plan.halo
    col_g = torch.where(part_step.graph.col.long() < part_step.n_own, part_step.graph.col.long() + lo,
                        halo[(part_step.graph.col.long() - part_step.n_own).clamp_(min=0)]) if nl else None
    ok_int = (e1 - e0 == nl) and bool(torch.equal(col_g.int(), single.graph.col[e0:e1]))
    ok_int = ok_int and bool(torch.equal(part_step.kstar[:nl], single.kstar[e0:e1]))
    ok_int = ok_int and bool(torch.equal(part_step.w[:nl], single.w[e0:e1]))
    pos = torch.arange(e0, e1, device=dev, dtype=torch.int64) % 1_000_003 + 1
    khash = (part_step.kstar[:nl].long() * pos).sum()
    khash_single = (single.kstar[:single.graph.nnz].long() *
                    (torch.arange(single.graph.nnz, device=dev, dtype=torch.int64) % 1_000_003 + 1)).sum()

    def rel(a, b):
        return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))
    n = part_step.n_own
    errs = {"s": rel(part_step.s[:n], single.s[lo:hi]), "H": rel(part_step.H[:n], single.H[lo:hi]),
            "r": rel(part_step.r[:n], single.r[lo:hi]), "dZ": rel(part_step.dZ, single.dZ[lo:hi]),
            "dH": rel(part_step.dH[:n], single.dH[lo:hi]),
            "prob": float((part_step.prob[:part_step.P] - single.prob[:part_step.P]).abs().max())}
    # the exchange itself, on the device: halo rows of Z must be bit-identical copies of the owners' rows, halo rows
    # of H (pair endpoints) and s equal to the single-GPU values row by row
    def rowrel(a, b):
        den = b.abs().amax(dim=tuple(range(1, b.dim()))).clamp_min(1e-20)
        return float(((a - b).abs().amax(dim=tuple(range(1, b.dim()))) / den).max()) if a.numel() else 0.0
    pair_loc = torch.cat([part_step.plan.recv_pair[q] for q in range(world) if q != rank]) if world > 1 else None
    diag = {"Z_halo_bitwise": bool(torch.equal(part_step.Z[n:], single.Z[halo])),
            "s_halo_rowrel": rowrel(part_step.s[n:], single.s[halo]),
            "H_pair_halo_rowrel": rowrel(part_step.H[pair_loc], single.H[halo[pair_loc - n]]) if pair_loc is not None else 0.0,
            "H_own_rowrel": rowrel(part_step.H[:n], single.H[lo:hi])}
    dp = (part_step.prob[:part_step.P] - single.prob[:part_step.P]).abs()
    worst = int(dp.argmax())
    deg = single.graph.degrees()
    diag["worst_pair"] = {"u_degree": int(deg[u[worst]]), "v_degree": int(deg[v[worst]]),
                          "prob": float(part_step.prob[worst]), "prob_single_gpu": float(single.prob[worst])}
    dflag = torch.tensor([float(diag["Z_halo_bitwise"]), -diag["s_halo_rowrel"], -diag["H_pair_halo_rowrel"],
                          -diag["H_own_rowrel"]], dtype=torch.float64, device=dev)
    dist.all_reduce(dflag, op=dist.ReduceOp.MIN)
    diag.update(Z_halo_bitwise=bool(dflag[0].item() == 1.0), s_halo_rowrel=-float(dflag[1]),
                H_pair_halo_rowrel=-float(dflag[2]), H_own_rowrel=-float(dflag[3]))
    vol = part_step.exchange_volume()
    t = torch.tensor([float(ok_int)] + [-e for e in errs.values()], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    hs = khash.clone()
    dist.all_reduce(hs)
    out = {"workload": wl["name"], "steps": 2,
           "integers_and_routing_bitwise_equal": bool(t[0].item() == 1.0),
           "kstar_hash": int(hs.item()), "kstar_hash_single_gpu": int(khash_single.item()),
           "max_rel_err_vs_single_gpu": {k: -float(x) for k, x in zip(errs.keys(), t[1:].tolist())},
           "loss": float(part_step.loss.item()), "loss_single_gpu": float(single.loss.item()),
           "exchange_check": diag,
           "rank0_rows": vol, "exchange": "NVLink peer push" if part_step.pushed else "torch.distributed p2p"}
    # Bars.  Integers and routing: bitwise.  s, H (computed directly from Z): 1e-5 of the tensor's max-abs.  The
    # scores and everything behind them (dH, r, dZ) inherit the ABSOLUTE error of the hub rows of H -- 5e-7 of
    # |H| ~ 10^1..10^2, from range cuts that depend on the partition -- through exp(q) <H_u, H_v> of the many pairs
    # with a hub endpoint: observed 5e-5 (2, 4 ranks) to 2e-4 (8 ranks) in prob and up to 7e-4 in r; the host
    # logic (halo lists, exchange order) is bitwise equal to one process at world 2, 4 and 8 on the CPU backend.
    tol = {"s": 1e-5, "H": 1e-5, "r": 2e-3, "dZ": 2e-3, "dH": 2e-3, "prob": 1e-3}
    out["tolerance"] = tol
    out["ok"] = (out["integers_and_routing_bitwise_equal"] and out["kstar_hash"] == out["kstar_hash_single_gpu"]
                 and diag["Z_halo_bitwise"] and diag["s_halo_rowrel"] < 1e-5 and diag["H_pair_halo_rowrel"] < 1e-5
                 and all(e < tol[k] for k, e in out["max_rel_err_vs_single_gpu"].items()))
    part_step.close()
    del part_step, single
    torch.cuda.empty_cache()
    return out


def gen_pairs_from_edges(src, dst, N, E, P, dev):
    """every rank draws the same pairs: positives are directed edge columns (each is an entry of adj_sym),
    M_NEG uniform negatives share u with their positive (main_disentangled.py:159-163); sorted by u so the
    (1 + M_NEG) pairs of one u are adjacent"""
    import torch
    gp = torch.Generator(device=dev).manual_seed(1)
    P_pos = max(P // (1 + M_NEG), 1)
    e = torch.randint(0, E, (P_pos,), generator=gp, device=dev)
    pu, pv = src[e], dst[e]
    nu = pu.repeat(M_NEG)
    nv = torch.randint(0, N, (P_pos * M_NEG,), generator=gp, device=dev)
    u, v = torch.cat([pu, nu]), torch.cat([pv, nv])
    lab = torch.cat([torch.ones(P_pos, device=dev), torch.zeros(P_pos * M_NEG, device=dev)])
    wts = torch.cat([torch.full((P_pos,), 1.0 / P_pos, device=dev),
                     torch.full((P_pos * M_NEG,), 1.0 / (M_NEG * P_pos * M_NEG), device=dev)])
    order = torch.sort(u, stable=True).indices
    return u[order], v[order], lab[order], wts[order]

# ------------------------------------------------------------------------------------------------
# native arm
# ------------------------------------------------------------------------------------------------
PHASES = ["wait", "ag_Z", "attn_fwd", "ag_s", "spmm_fwd", "ag_H", "pair_fwd", "ag_prob", "loss", "pair_bwd",
          "ag_dH", "bwd_gather", "ag_r", "bwd_edges"]
KERNEL_PHASES = ["attn_fwd", "spmm_fwd", "pair_fwd", "pair_bwd", "bwd_gather", "bwd_edges"]
DUMP_PAIRS = 1 << 20     # sampled link scores
DUMP_ROWS = 1 << 14      # sampled node rows of H and dL/dZ (K*d floats each): 20 MB in all at K*d = 128


def dump_outputs(out_dir, step):
    """What the last timed step handed its caller, as float .npy files in out_dir: loss [1] (float64),
    prob [<= DUMP_PAIRS] (link scores), H and dZ [<= DUMP_ROWS, K, d] (embeddings and dL/dZ of the
    nodes).  Larger outputs are sampled at indices drawn from a fixed seed, so two builds run with the
    same arguments dump the same entries."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(0)
    pick = lambda n, k: torch.from_numpy(np.sort(rng.choice(n, size=min(n, k), replace=False))).to(step.device)
    pairs, rows = pick(step.P, DUMP_PAIRS), pick(step.n_own, DUMP_ROWS)
    out = {"loss": np.array([float(step.loss.item())], dtype=np.float64),
           "prob": step.prob[:step.P][pairs].cpu().numpy(),
           "H": step.H[:step.n_own][rows].cpu().numpy(),
           "dZ": step.dZ[rows].cpu().numpy()}
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_native(args):
    import torch
    import torch.distributed as dist
    from disenlink_b200 import _lib, ops
    from disenlink_b200.partition import PartitionedLinkStep

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # stdout carries exactly one JSON line
        dist.init_process_group("nccl", device_id=dev)
    _lib.lib()  # fail loudly if the extension is missing

    wl = dict(WORKLOADS[args.workload])
    N, E, K, d, P, beta, T = (wl[k] for k in ("N", "E", "K", "d", "P", "beta", "T"))
    D = K * d
    parity = None
    if world > 1 and not args.no_parity:
        parity = multi_gpu_parity(world, rank, dev)
    # memory guard (one GPU; a partitioned run holds own + halo rows only): ~4 [N,K,d] fp32 buffers + graph + pairs
    free_b, total_b = torch.cuda.mem_get_info(dev)
    need = max(int(4.4 * N * D * 4) + 2 * E * 10 + P * 50, 16 * E + 56 * E) + (4 << 30)
    if world == 1 and need > free_b:
        raise SystemExit(f"workload {args.workload} needs ~{need / 2**30:.0f} GiB, {free_b / 2**30:.0f} GiB free")

    t_setup = time.perf_counter()
    src, dst = gen_edges(N, E, 0, dev)
    from disenlink_b200.graph import Graph
    u, v, lab, wts = gen_pairs_from_edges(src, dst, N, E, P, dev)
    P = int(u.numel())

    events = []

    def mark(name):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(torch.cuda.current_stream(dev))
        events.append((name, ev))

    step = PartitionedLinkStep(src, dst, N, u, v, lab, wts, K, d, beta, T, world=world, rank=rank,
                               device=dev, mark=mark)
    del src, dst
    torch.cuda.empty_cache()
    part = step.part
    nnz_local = step.graph.nnz
    nnz_global = nnz_local
    if world > 1:
        t = torch.tensor([nnz_local], dtype=torch.int64, device=dev)
        dist.all_reduce(t)
        nnz_global = int(t.item())
    gen_Z(part.n_local, K, d, 0, dev, row0=part.lo, out=step.Z_own)   # every rank draws the rows it owns
    pushed = step.pushed                     # exchanges as NVLink pushes when the ranks can map each other
    volume = step.exchange_volume()
    torch.cuda.synchronize(dev)
    t_setup = time.perf_counter() - t_setup

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-timed loop ----
    for _ in range(args.warmup):
        step.run()
    barrier()
    events.clear()
    launches0 = _lib.launches
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev_a, ev_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    torch.cuda.profiler.start()      # ncu --profile-from-start off captures exactly the timed steps
    ev_a.record(torch.cuda.current_stream(dev))
    for _ in range(args.steps):
        step.run()
    ev_b.record(torch.cuda.current_stream(dev))
    torch.cuda.profiler.stop()
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, step)
    abi_calls = _lib.launches - launches0
    total_ms = ev_a.elapsed_time(ev_b)
    # per-phase times from consecutive events
    phase_ms = {p: 0.0 for p in PHASES}
    for (n0, e0), (n1, e1) in zip(events[:-1], events[1:]):
        if n1 != "begin":
            phase_ms[n1] += e0.elapsed_time(e1)
    phase_ms = {p: v / args.steps for p, v in phase_ms.items()}
    loss_val = float(step.loss.item())
    per_rank = None
    if world > 1:
        tt = torch.tensor([total_ms] + [phase_ms[p] for p in PHASES], dtype=torch.float64, device=dev)
        allt = [torch.empty_like(tt) for _ in range(world)]
        dist.all_gather(allt, tt)
        per_rank = {p: [round(float(a[1 + i]), 3) for a in allt] for i, p in enumerate(PHASES)}
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        total_ms = float(tt[0].item())
        phase_ms = {p: float(x) for p, x in zip(PHASES, tt[1:].tolist())}
    ms_per_step = total_ms / args.steps
    t_factor = phase_ms["attn_fwd"] + phase_ms["spmm_fwd"] + phase_ms["bwd_gather"] + phase_ms["bwd_edges"]
    # the same definition at every N: the four factor kernels plus the exchanges THEY need (Z, s, the routed
    # dH slices, r; all zero on one GPU).  The H and prob exchanges serve the pair scoring and count there.
    t_comm_factor = phase_ms["wait"] + phase_ms["ag_Z"] + phase_ms["ag_s"] + phase_ms["ag_dH"] + phase_ms["ag_r"]
    value = nnz_global / ((t_factor + t_comm_factor) * 1e-3)
    pair_rate = P / ((phase_ms["pair_fwd"] + phase_ms["ag_H"] + phase_ms["ag_prob"]) * 1e-3)

    # ---- roofline of the dominant kernel (per-rank bytes / per-rank time) ----
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (measured copy)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    ab = alg_bytes(nnz_local, part.n_local, K, d, 0)
    ab["pair_fwd"] = (step.p_hi - step.p_lo) * (16 * D + 12)
    # node-major decoder backward: per incidence the other endpoint's Z and H rows + 3 ids/floats,
    # per node 2 rows in and 2 rows out (less than SURVEY's scatter-form P*(32D+16): see DESIGN.md)
    ab["pair_bwd"] = int(step.inc.nnz) * (8 * D + 12) + part.n_local * 16 * D
    # kernels of libdisenlink_b200.so per step (streaming path): attention = routing + row sums + chain +
    # empty rows (3; one GPU, symmetric: upper-triangle routing + expand + chain + empty rows = 4); aggregation =
    # gather + chain + empty rows (3; + the Z/s streaming pass on one GPU); pair scoring fwd (1); weighted BCE (2);
    # decoder backward = stream + chain + empty nodes (3); backward pass 1 (3); backward pass 2 = (s,r) pack +
    # stream + chain (3)
    # (checked against the ncu launch list of the same command: profiles/r02_launches_mid.csv, 22 per step)
    launches_per_step = 18
    try:
        g_ = step.graph
        sym_attn = bool(getattr(g_, "_sym", None)) and g_.nnz >= g_.sym_min_nnz      # + k_sym_expand
        sym_bwd = bool(step.plan_bwd) and step.plan_bwd.get("mode") == "sym"          # + k_bwd_sym_lower + its chain
        launches_per_step += int(sym_attn) + int(bool(step.prescale)) + 2 * int(sym_bwd)
    except Exception:
        launches_per_step += 2 if world == 1 else 0
    if world > 1 and pushed:                                  # + need-masks, pushes of Z, s, H, dH, r, prob
        launches_per_step += 7
    kernels = {}
    for kname in KERNEL_PHASES:
        ms = phase_ms[kname]
        gbs = ab[kname] / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
        kernels[kname] = {"ms": round(ms, 4), "alg_bytes": int(ab[kname]), "GB/s": round(gbs, 1),
                          "frac": round(gbs / peak, 4)}
    # second bound for the two slice gathers: one random <=128-byte access per entry cannot go faster than the
    # device's random-access rate, measured by tools/gather_probe.cu (profiles/r02_gather_probe.jsonl)
    probe_path = os.path.join(ROOT, "profiles", "r02_gather_probe.jsonl")
    if os.path.exists(probe_path):
        try:
            rows = [json.loads(l) for l in open(probe_path) if l.strip()]
            ceil = max(r["objects_per_s"] for r in rows if r.get("object_bytes") == 64 and r.get("array_gb", 0) > 20
                       and r.get("method") in ("ldg", "cpasync"))
            for kname in ("spmm_fwd", "bwd_gather"):
                if phase_ms[kname] > 0:
                    rate = nnz_local / (phase_ms[kname] * 1e-3)
                    kernels[kname]["random_access_bound"] = {
                        "accesses_per_s": rate, "ceiling": ceil, "frac": round(rate / ceil, 4),
                        "note": "one random 64-B slice per entry; ceiling = measured random 64-B gathers/s over a "
                                "25.6 GB array (profiles/r02_gather_probe.jsonl); the phase also streams 8ND bytes"}
        except Exception:
            pass
    # SURVEY's P(16D+12) counts four full rows per pair; the pairs are sorted by u and come in groups of
    # 1 + M_NEG sharing u, so z_u / h_u are read once per group: the honest floor is P(8D(1 + 1/(1+m)) + 12)
    pf_ms = phase_ms["pair_fwd"]
    pf_sorted = (step.p_hi - step.p_lo) * (8 * D * (1 + 1.0 / (1 + M_NEG)) + 12)
    kernels["pair_fwd"]["alg_bytes_u_sorted"] = int(pf_sorted)
    kernels["pair_fwd"]["frac_u_sorted"] = round(pf_sorted / (pf_ms * 1e-3) / 1e9 / peak, 4) if pf_ms > 0 else 0.0
    kernels["pair_fwd"]["note"] = ("frac uses SURVEY 8(d)'s P(16D+12) (no credit for the u-sorted 1+m groups) and reads "
                                   "above 1; frac_u_sorted uses P(8D(1+1/(1+m))+12), the bytes a read-only stream must move")
    dom = max(KERNEL_PHASES, key=lambda k: phase_ms[k])
    fwd_bwd_bytes = ab["attn_fwd"] + ab["spmm_fwd"] + ab["bwd_gather"] + ab["bwd_edges"]
    roofline = {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["GB/s"], "peak": peak, "unit": "GB/s",
                "frac": kernels[dom]["frac"], "traffic": None, "peak_source": peak_src,
                "factor_agg_fwd_bwd": {"alg_bytes": int(fwd_bwd_bytes),
                                       "GB/s": round(fwd_bwd_bytes / (t_factor * 1e-3) / 1e9, 1),
                                       "frac": round(fwd_bwd_bytes / (t_factor * 1e-3) / 1e9 / peak, 4)}}
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(prof):
        try:   # ncu dram bytes per entry (captured at the mid size) x the entries of this launch
            per = json.load(open(prof))[dom]["per_entry"]
            units = (step.p_hi - step.p_lo) if dom.startswith("pair") else nnz_local
            roofline["traffic"] = int(per * units)
            roofline["traffic_source"] = "profiles/traffic.json: ncu --set full dram bytes per entry at nnz=1e8, scaled"
        except Exception:
            pass

    # ---- end to end through the public autograd API, host buffers ----
    e2e = None
    if world == 1 and not args.no_e2e:
        Z_host = torch.empty(N, K, d, dtype=torch.float32).pin_memory()
        Z_host.copy_(step.Z_own)
        del step
        torch.cuda.empty_cache()
        g_full = Graph.from_edges(*gen_edges(N, E, 0, dev), N)
        batch = ops.PairBatch(u, v, N)
        batch.incidence()
        torch.cuda.empty_cache()
        prob_host = torch.empty(P, dtype=torch.float32).pin_memory()
        # Input staging: Z comes from pinned host memory every step.  Two device buffers and a copy
        # stream let the upload of step t+1 overlap the kernels of step t (every timed step still
        # issues, and the timed region completes, one 4*N*D-byte upload and one P-float read-back);
        # with a single buffer (not enough memory for two) the upload is serial with the kernels.
        Zbufs = [torch.empty(N, K, d, dtype=torch.float32, device=dev)]
        try:
            Zbufs.append(torch.empty(N, K, d, dtype=torch.float32, device=dev))
        except torch.cuda.OutOfMemoryError:
            pass
        nb = len(Zbufs)
        copy_stream = torch.cuda.Stream(dev)
        ready = [torch.cuda.Event() for _ in range(nb)]
        free = [torch.cuda.Event() for _ in range(nb)]
        for ev in free:
            ev.record(torch.cuda.current_stream(dev))
        last = {}

        def upload(slot):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(free[slot])          # the kernels that read this buffer are done
                Zbufs[slot].copy_(Z_host, non_blocking=True)
                ready[slot].record(copy_stream)

        def e2e_step(i):
            cur = torch.cuda.current_stream(dev)
            slot = i % nb
            if nb == 1:
                upload(0)
            else:
                upload((i + 1) % nb)                        # next step's input
            cur.wait_event(ready[slot])
            Zg = Zbufs[slot].requires_grad_(True)
            loss, prob, H = ops.link_bce_loss(Zg, g_full, batch, lab, wts, beta, T)
            del H                                           # 25.6 GB the backward does not need
            loss.backward()
            free[slot].record(cur)
            prob_host.copy_(prob, non_blocking=True)
            last["prob"] = prob
            val = loss.item()
            Zg.grad = None
            Zbufs[slot].requires_grad_(False)
            return val

        def e2e_run(n_steps, i0):
            for i in range(i0, i0 + n_steps):
                val = e2e_step(i)
            torch.cuda.synchronize(dev)                     # all streams: the last upload included
            return val

        oom = False
        try:
            if nb > 1:
                upload(0)
            n_warm = max(args.warmup, 1)
            e2e_run(n_warm, 0)
            t0 = time.perf_counter()
            e2e_loss = e2e_run(args.steps, n_warm)
            e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
        except torch.cuda.OutOfMemoryError:
            oom = True                       # handled outside the handler: the traceback pins the failed step's buffers
        if oom:
            # the second input buffer did not leave room for the step's own buffers: serial staging
            import gc
            torch.cuda.synchronize(dev)
            del Zbufs[1:]
            nb = 1
            last.clear()
            Zbufs[0].grad = None
            Zbufs[0].requires_grad_(False)
            gc.collect()
            torch.cuda.empty_cache()
            e2e_run(max(args.warmup, 1), 0)
            t0 = time.perf_counter()
            e2e_loss = e2e_run(args.steps, 0)
            e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
        e2e = {"value": g_full.nnz / (e2e_ms * 1e-3), "unit": "edges/s", "ms_per_step": round(e2e_ms, 3),
               "h2d_bytes_per_step": int(N * D * 4), "d2h_bytes_per_step": int(P * 4 + 4),
               "api": "ops.link_bce_loss(Z, graph, pairs, labels, weights).backward(); Z from pinned host "
                      "memory, loss + P scores read back",
               "input_staging": ("double-buffered on a copy stream: the upload of step t+1 overlaps the kernels "
                                 "of step t" if nb > 1 else "single buffer: upload serial with the kernels"),
               "loss": e2e_loss}

    # ---- N > 1: end to end through the partitioned step's public API: every rank uploads the embeddings of
    # the nodes it owns from pinned host memory (a staging buffer on a copy stream takes step t+1's upload
    # while step t runs), runs the step and reads back the loss and its share of the scores ----
    if world > 1 and not args.no_e2e:
        n_own = step.n_own
        Zh = torch.empty(n_own, K, d, dtype=torch.float32).pin_memory()
        Zh.copy_(step.Z_own)
        lo_p = rank * step.p_per
        n_p = step.p_hi - step.p_lo
        prob_host = torch.empty(max(n_p, 1), dtype=torch.float32).pin_memory()
        stage = torch.empty(n_own, K, d, dtype=torch.float32, device=dev)
        copy_stream = torch.cuda.Stream(dev)
        ready, free = torch.cuda.Event(), torch.cuda.Event()
        free.record(torch.cuda.current_stream(dev))

        def upload():
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(free)
                stage.copy_(Zh, non_blocking=True)
                ready.record(copy_stream)

        def e2e_multi(n_steps):
            val = 0.0
            for _ in range(n_steps):
                cur = torch.cuda.current_stream(dev)
                cur.wait_event(ready)
                step.Z_own.copy_(stage)
                free.record(cur)
                upload()                                        # next step's input, overlapped with this step
                step.run()
                prob_host.copy_(step.prob[lo_p:lo_p + n_p] if n_p else step.prob[:1], non_blocking=True)
                val = step.loss.item()
            torch.cuda.synchronize(dev)
            return val
        upload()
        e2e_multi(max(args.warmup, 1))
        barrier()
        t0 = time.perf_counter()
        e2e_loss = e2e_multi(args.steps)
        barrier()
        tt = torch.tensor([(time.perf_counter() - t0) * 1e3 / args.steps], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_ms = float(tt.item())
        e2e = {"value": nnz_global / (e2e_ms * 1e-3), "unit": "edges/s", "ms_per_step": round(e2e_ms, 3),
               "h2d_bytes_per_step": int(N * D * 4), "d2h_bytes_per_step": int(P * 4 + 4 * world),
               "api": "PartitionedLinkStep.run(Z_own) on every rank; Z_own from pinned host memory (N*D*4 bytes over all "
                      "ranks), loss + the rank's share of the P scores read back; wall clock between barriers, max over ranks",
               "input_staging": "staging buffer on a copy stream: the upload of step t+1 overlaps the kernels of step t",
               "loss": e2e_loss}
        step.close()

    # ---- the evaluation-side kernels of SURVEY 8(f) on the same data: AUC of the P scores, one
    # round of structured negative sampling against the resident CSR (device-timed, outside the step) ----
    extras = None
    if e2e is not None and world == 1:
        def timed(fn, reps=2):
            fn()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            a.record()
            for _ in range(reps):
                out = fn()
            b.record()
            torch.cuda.synchronize(dev)
            return a.elapsed_time(b) / reps, out
        prob_d = last["prob"]
        auc_ms, auc_out = timed(lambda: ops.roc_auc_stats(prob_d, lab))
        n_src = min(g_full.nnz, 100_000_000)
        src64 = g_full.erow[:n_src].to(torch.int64)
        ei = torch.stack([src64, g_full.col[:n_src].to(torch.int64)])
        ns_ms, ns_out = timed(lambda: ops.structured_negative_sampling(ei, N, seed=1, graph=g_full))
        extras = {"roc_auc": {"pairs": P, "ms": round(auc_ms, 3), "pairs_per_s": P / (auc_ms * 1e-3),
                              "auc": float(auc_out[0].item())},
                  "structured_negative_sampling": {"edges": n_src, "ms": round(ns_ms, 3),
                                                   "edges_per_s": n_src / (ns_ms * 1e-3)}}
        del ei, src64, ns_out
        try:
            extras["projection"] = projection_bench(dev)
        except Exception as ex:                       # a side measurement never costs the headline line
            extras["projection"] = {"error": repr(ex)[:200]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    configs = None
    if world == 1 and not args.no_configs:
        # drop the headline workload's buffers (rebinding also clears the cells the e2e closures hold)
        g_full = batch = Zbufs = Z_host = prob_host = last = step = Z = prob_d = None  # noqa: F841
        torch.cuda.empty_cache()
        configs = other_configs(dev, peak)
    cb = cpu_baseline(K, d, beta, T) if (world == 1 and not args.no_cpu) else None
    if cb is not None:
        cb["dense_reference"] = dense_reference_leg(dev)

    line = {
        "metric": "factor-agg edges/s (fwd+bwd)", "value": value, "unit": "edges/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": wl["name"], "N": N, "E_directed": E, "nnz": nnz_global, "K": K, "d": d, "P": P,
                   "beta": beta, "T": T, "parallelism": "1 GPU" if world == 1 else (
                       f"node-partitioned x{world} (nnz-balanced ranges, rank-local storage = own + halo rows); owners push "
                       "what the reader reads over NVLink peer memory: halo rows of Z, s, r, H rows of the pair endpoints, "
                       "routed slices of dH" if pushed
                       else f"node-partitioned x{world}, torch.distributed point-to-point halo exchange"),
                   "l2": f"inputs exceed L2: Z alone is {N * D * 4 / 2**30:.1f} GiB vs 126 MB L2 (no flush needed)",
                   "value_definition": "nnz / (attention + aggregation + both backward passes + the halo exchanges they "
                                       "need: Z, s, routed dH slices, r, and the wait for the slowest rank -- all zero on one GPU); the same at every N"},
        "pair_scores_per_s": pair_rate,
        "phases_ms": {k: round(v, 4) for k, v in phase_ms.items()},
        "kernels": kernels, "roofline": roofline, "clocks": clocks,
        "gpu_launches": launches_per_step * args.steps, "abi_calls_per_step": abi_calls // max(args.steps, 1),
        "loss": loss_val, "setup_s": round(t_setup, 2),
    }
    if e2e is not None:
        line["e2e"] = e2e
    if parity is not None:
        line["parity"] = parity
    if world > 1:
        line["partition"] = {"bounds": part.bounds, "rank0": volume}
        line["phases_ms_per_rank"] = per_rank
    if extras is not None:
        line["next_rows"] = extras
    if cb is not None:
        line["cpu_baseline"] = cb
    if configs is not None:
        line["other_configs"] = configs
    emit(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line of the contract, on the process's real stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    # stdout carries exactly one JSON line: whatever libraries print there (NCCL's version banner, warnings)
    # is sent to stderr for the duration of the run
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default=os.environ.get("DL_BENCH_WORKLOAD", "c5"), choices=list(WORKLOADS))
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="N > 1: skip the comparison with a single-GPU step")
    ap.add_argument("--no-configs", action="store_true", help="skip the side measurements of BASELINE configs[0..3]")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's loss, scores, H and dL/dZ (seeded samples) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "native" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs: native arm on one GPU only")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
