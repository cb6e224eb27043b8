"""CPU suite of the node-partitioned step on directed edge columns (partition.DirectedPartitionedLinkStep).

The in-view of every rank (directed_in_view: the in-entries of its nodes, tperm into [own CSR | record tail]) and
the record send lists are checked against the global transposed pattern of the directed hard-case generator of
test_directed.py, for world 2, 4 and 8 and a rank that owns no node.  The step itself runs over torch.distributed
(gloo) with a CPU test double: the oracle for attention, aggregation and scoring (as in test_partition_gloo.py) and
numpy float32 statements of the three directed backward phases (csrc/bwd_dir.cu), which sum every node's entries in
the kernels' order.  The ranks must reproduce one process bit for bit; one process is checked against the float64
directed reference.
"""
import os
import socket
from functools import lru_cache

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from disenlink_b200.partition import (DirectedPartitionedLinkStep, NodePartition, directed_in_view, entry_send_lists,
                                      owned_out_entries)
from test_directed import RefDir64, csr_of, directed_cases, directed_graph, transpose_of
from test_gpu_kernel_paths import BETA, TEMP, check_outputs
from test_partition_gloo import OracleBackend, _LocalGraph


# ------------------------------------------------------------------------------------------
# numpy statement of the directed phases (float32, the kernels' per-node summation order)
# ------------------------------------------------------------------------------------------
def _dot(a, b):
    """sum over the last axis in index order (no pairwise reduction: the same bits for every row count)."""
    acc = np.zeros(a.shape[:-1], np.float32)
    for x in range(a.shape[-1]):
        acc = acc + a[..., x] * b[..., x]
    return acc


def _softmax(zr, zc, T):
    """a[e, :] of the entries with row slices zr and column slices zc ([E, K, d])."""
    q = _dot(zr, zc) / np.float32(T)
    e = np.exp(q - q.max(1, keepdims=True))
    return e / e.sum(1, keepdims=True)


def _rows(rowptr, n):
    return np.repeat(np.arange(n), np.diff(rowptr[:n + 1]))


def directed_phase(g, gt, tperm, Z, G, kstar, w, s, beta, T, dZ, r, dw, routed, phase):
    """One phase of dl_factor_bwd_directed_phase on numpy arrays; writes the owned rows of dZ / r and dw[:g.nnz]."""
    n, K = g.n_own, Z.shape[1]
    beta32, omb = np.float32(beta), np.float32(1.0 - beta)
    if phase == 1:
        has = np.zeros((n, K), bool)
        has[_rows(g.rowptr, n), kstar[:g.nnz].astype(np.int64)] = True
        j = _rows(gt.rowptr, n)
        e = tperm[:gt.nnz].astype(np.int64)
        k = kstar[e].astype(np.int64)
        acc = np.zeros((n,) + Z.shape[1:], np.float32)
        np.add.at(acc, (j, k), w[e][:, None] * G[gt.col.astype(np.int64), k])
        Tin = (omb / s[:n])[:, :, None] * acc
        r[:n] = np.where(has, _dot(Z[:n], Tin) / s[:n], np.float32(0))
        dZ[:n] += beta32 * G[:n] + Tin
        return
    if phase == 2:
        v, u, e = _rows(g.rowptr, n), g.col.astype(np.int64), np.arange(g.nnz)
    else:
        v, u, e = _rows(gt.rowptr, n), gt.col.astype(np.int64), tperm[:gt.nnz].astype(np.int64)
    k = kstar[e].astype(np.int64)
    a = _softmax(Z[u], Z[v], T) if phase == 3 else _softmax(Z[v], Z[u], T)
    if phase == 2:
        c = omb * _dot(G[v, k], Z[u, k])
        dw[e] = c / s[u, k] - r[v, k]
    dwv = dw[e]
    basec = dwv * a[np.arange(e.size), k] / np.float32(T)
    coef = basec[:, None] * (np.eye(K, dtype=np.float32)[k] - a)
    acc = np.zeros((n,) + Z.shape[1:], np.float32)
    np.add.at(acc, v, coef[:, :, None] * Z[u])
    dZ[:n] += acc


class DirectedOracleBackend(OracleBackend):
    """OracleBackend plus the directed CSR and the numpy directed phases."""

    def build_csr_directed(self, src, dst, part):
        rows, cols = owned_out_entries(src, dst, part)
        key = np.unique(rows.numpy() * part.n_global + cols.numpy())
        r, c = key // part.n_global, key % part.n_global
        rowptr = np.zeros(part.n_local + 1, np.int64)
        np.cumsum(np.bincount(r, minlength=part.n_local), out=rowptr[1:])
        return torch.from_numpy(rowptr), torch.from_numpy(c.astype(np.int32))

    def factor_bwd_directed_phase(self, g, gt, tperm, Z, G, kstar, w, s, beta, T, dZ, r, dw, routed, phase):
        dz = dZ.numpy()
        directed_phase(g, gt, tperm.numpy(), Z.numpy(), G.numpy(), kstar.numpy(), w.numpy(), s.numpy(), beta, T,
                       dz, r.numpy(), dw.numpy(), routed, phase)


# ------------------------------------------------------------------------------------------
# inputs: the directed hard cases
# ------------------------------------------------------------------------------------------
N_NODES = 6000


@lru_cache(maxsize=None)
def hard_directed():
    src, dst = directed_graph(N_NODES, 20000, 11)
    rowptr, col = csr_of(src, dst, N_NODES)
    directed_cases(rowptr, col)
    return src, dst, rowptr, col


def make_inputs(K=4, d=8, P=3000, seed=0):
    src, dst, _, _ = hard_directed()
    rng = np.random.default_rng(seed)
    u = rng.integers(0, N_NODES, P)
    v = rng.integers(0, N_NODES, P)
    lab = (rng.random(P) < 0.3).astype(np.float32)
    Z = (rng.standard_normal((N_NODES, K, d)) * 0.4).astype(np.float32)
    tt = torch.from_numpy
    return tt(src), tt(dst), tt(u), tt(v), tt(lab), torch.full((P,), 1.0 / P), tt(Z)


def split_points(world, empty_rank):
    src, dst, _, _ = hard_directed()
    b = NodePartition.nnz_balanced(torch.from_numpy(src), torch.from_numpy(dst), N_NODES, world, 0).bounds
    if empty_rank:                                    # rank world // 2 owns no node
        b[world // 2 + 1] = b[world // 2]
    return b


# ------------------------------------------------------------------------------------------
# in-view structure
# ------------------------------------------------------------------------------------------
def rank_view(src, dst, bounds, rank):
    part = NodePartition(N_NODES, len(bounds) - 1, rank, list(bounds))
    be = DirectedOracleBackend()
    rowptr, col_g = be.build_csr_directed(src, dst, part)
    trowptr, tsrc, tperm, tail_off = directed_in_view(src, dst, part, rowptr, col_g)
    rows = torch.repeat_interleave(torch.arange(part.n_local), rowptr[1:] - rowptr[:-1]) + part.lo
    key = (rows * N_NODES + col_g.to(torch.int64)).numpy()                  # (i, j) of every own CSR entry
    return dict(part=part, rowptr=rowptr, col_g=col_g, key=key, trowptr=trowptr.numpy(), tsrc=tsrc.numpy(),
                tperm=tperm.numpy(), tail_off=tail_off, send=[t.numpy() for t in entry_send_lists(col_g, part)])


@pytest.mark.parametrize("world,empty_rank", [(2, False), (4, True), (8, False), (8, True)])
def test_in_views_cover_the_transposed_pattern(world, empty_rank):
    src_np, dst_np, rowptr, col = hard_directed()
    src, dst = torch.from_numpy(src_np), torch.from_numpy(dst_np)
    bounds = split_points(world, empty_rank)
    views = [rank_view(src, dst, bounds, q) for q in range(world)]
    if empty_rank:
        assert views[world // 2]["part"].n_local == 0
    trowptr, tcol, tp = transpose_of(rowptr, col)
    # the union of the in-views is the global transposed pattern, in its order
    assert np.array_equal(np.concatenate([np.diff(v["trowptr"]) for v in views]), np.diff(trowptr))
    assert np.array_equal(np.concatenate([v["tsrc"] for v in views]), tcol)
    assert sum(v["key"].size for v in views) == col.size
    for p, v in enumerate(views):
        lo, n_own, nnz = v["part"].lo, v["part"].n_local, v["key"].size
        # tail: sender q's block = q's send list to p, in q's CSR order
        tail = np.concatenate([views[q]["key"][views[q]["send"][p]] for q in range(world) if q != p] +
                              [np.empty(0, np.int64)])
        for q in range(world):
            blk = tail[v["tail_off"][q]:v["tail_off"][q + 1]]
            want = views[q]["key"][views[q]["send"][p]] if q != p else np.empty(0, np.int64)
            assert np.array_equal(blk, want), (p, q)
            assert np.all(np.diff(blk) > 0)
        assert v["tail_off"][-1] - v["tail_off"][0] == tail.size
        # every tperm resolves to its (i, j) through [own CSR | tail]
        records = np.concatenate([v["key"], tail])
        j = np.repeat(np.arange(n_own), np.diff(v["trowptr"])) + lo
        assert v["tperm"].size == 0 or v["tperm"].max() < nnz + tail.size
        assert np.array_equal(records[v["tperm"]], v["tsrc"] * N_NODES + j)
        own = (v["tsrc"] >= lo) & (v["tsrc"] < lo + n_own)
        assert np.all(v["tperm"][own] < nnz) and np.all(v["tperm"][~own] >= nnz)


def test_world1_in_view_is_the_transpose():
    src_np, dst_np, rowptr, col = hard_directed()
    v = rank_view(torch.from_numpy(src_np), torch.from_numpy(dst_np), [0, N_NODES], 0)
    trowptr, tcol, tp = transpose_of(rowptr, col)
    assert np.array_equal(v["trowptr"], trowptr)
    assert np.array_equal(v["tsrc"], tcol)
    assert np.array_equal(v["tperm"], tp)
    assert v["tail_off"] == [0, 0]


# ------------------------------------------------------------------------------------------
# the step over gloo
# ------------------------------------------------------------------------------------------
def run_step(world, rank, bounds=None):
    src, dst, u, v, lab, wts, Z = make_inputs()
    n, K, d = Z.shape
    step = DirectedPartitionedLinkStep(src, dst, n, u, v, lab, wts, K, d, BETA, TEMP, world=world, rank=rank,
                                       backend=DirectedOracleBackend(), device=torch.device("cpu"), bounds=bounds)
    part = step.part
    step.Z_own.copy_(Z[part.lo:part.hi])
    step.run()
    step.Z_own.mul_(0.9)                              # a second step with other Z over the same buffers
    step.run()
    return step


def _worker(rank, world, port, out_dir, bounds):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        step = run_step(world, rank, bounds)
        n = step.n_own
        torch.save({"dZ": step.dZ.clone(), "prob": step.prob.clone(), "loss": step.loss.clone(),
                    "kstar": step.kstar[:step.graph.nnz].clone(), "w": step.w[:step.graph.nnz].clone(),
                    "r": step.r[:n].clone(), "halo": step.plan.halo.clone(), "Zhalo": step.Z[n:].clone(),
                    "n_own": n, "n_tail": step.n_tail, "vol": step.exchange_volume()},
                   os.path.join(out_dir, f"rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


@lru_cache(maxsize=None)
def single_process():
    return run_step(1, 0)


@pytest.mark.parametrize("world,empty_rank", [(2, False), (4, True), (8, False)])
def test_gloo_directed_ranks_equal_single_process(tmp_path, world, empty_rank):
    single = single_process()
    bounds = split_points(world, empty_rank)
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    mp.spawn(_worker, args=(world, port, str(tmp_path), bounds), nprocs=world, join=True)
    outs = [torch.load(os.path.join(tmp_path, f"rank{r}.pt")) for r in range(world)]
    if empty_rank:
        assert any(o["n_own"] == 0 for o in outs)
    assert sum(o["vol"]["records_out"] for o in outs) == sum(o["n_tail"] for o in outs) > 0
    assert torch.equal(torch.cat([o["kstar"] for o in outs]), single.kstar[:single.graph.nnz])
    assert torch.equal(torch.cat([o["w"] for o in outs]), single.w[:single.graph.nnz])
    assert torch.equal(torch.cat([o["r"] for o in outs]), single.r)
    assert torch.equal(torch.cat([o["dZ"] for o in outs]), single.dZ)
    for o in outs:
        assert torch.equal(o["prob"][:single.P], single.prob[:single.P])
        assert torch.equal(o["loss"], single.loss)
        assert torch.equal(o["Zhalo"], single.Z[o["halo"]])


def test_directed_step_trains_on_the_columns_as_given():
    """One process: the step's CSR is the directed one (not its symmetrisation) and its in-view the transpose."""
    step = single_process()
    _, _, rowptr, col = hard_directed()
    assert np.array_equal(step.graph.rowptr[:N_NODES + 1], rowptr) and np.array_equal(step.graph.col, col)
    trowptr, tcol, tp = transpose_of(rowptr, col)
    assert np.array_equal(step.tgraph.col, tcol) and np.array_equal(step.tperm.numpy(), tp)
    assert step.n_tail == 0


def test_numpy_phases_match_the_float64_reference():
    """The test double's three phases on the whole graph against RefDir64 (per-element bounds of
    test_gpu_kernel_paths.py), and against the closed form's clamp rule (r exactly 0)."""
    from oracle import oracle as O
    from test_directed import in_only_pairs
    from test_gpu_kernel_paths import case_inputs
    src, dst, rowptr, col = hard_directed()
    n, K, d = N_NODES, 4, 8
    Z, G, _, _, _ = case_inputs(n, K, d, 0, 41)
    o_k, o_w, o_s = O.edge_attn_fwd(rowptr, col, Z, TEMP)
    ref = RefDir64(rowptr, col, Z, o_k, BETA, TEMP)
    res = ref.forward_dict()
    res.update(ref.factor_bwd(G))
    g = _LocalGraph(torch.from_numpy(rowptr), torch.from_numpy(col), n, n)
    trowptr, tcol, tp = transpose_of(rowptr, col)
    gt = _LocalGraph(torch.from_numpy(trowptr), torch.from_numpy(tcol), n, n)
    dZ = np.zeros_like(Z)
    r = np.zeros((n, K), np.float32)
    dw = np.zeros(col.size, np.float32)
    for phase in (1, 2, 3):
        directed_phase(g, gt, tp, Z, G, o_k, o_w, o_s, BETA, TEMP, dZ, r, dw, None, phase)
    check_outputs("numpy directed phases", dict(r=r, dZ=dZ), res, names=("r", "dZ"))
    clamp = in_only_pairs(rowptr, col, o_k, K)
    assert clamp.size and np.all(r[clamp[:, 0], clamp[:, 1]] == 0.0)
