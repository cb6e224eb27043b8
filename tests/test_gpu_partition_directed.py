"""GPU suite of the node-partitioned step on directed edge columns: the phase entry point of the directed backward
(dl_factor_bwd_directed_phase), the record push (dl_push_entries), one rank of DirectedPartitionedLinkStep on one GPU
with its halo rows and record tails filled from a checked single-GPU run, and the step at world 1."""
import numpy as np
import pytest
import torch

from test_directed import transpose_of
from test_gpu_directed import dir_case, dir_graph
from test_gpu_kernel_paths import BETA, TEMP, check_outputs
from test_gpu_parity import ORA_TOL, dl, relerr, t  # noqa: F401  (dl is a fixture)

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
SENTINEL = -7.25e30
K_, D_ = 8, 16


def bits(x):
    return x.contiguous().view(torch.int32).cpu().numpy() if x.dtype == torch.float32 else x.cpu().numpy()


def full_run(ops, Graph, K=K_, d=D_):
    """Single-GPU directed run of dir_graph(): attention, then the three phases with their per-entry dw kept."""
    src, dst, n, rowptr, col, cases = dir_graph()
    c = dir_case(K, d)
    g = Graph.from_edges(t(src), t(dst), n, directed=True)
    tg, tperm = g.transpose_view()
    Z, G = t(c["Z"]), t(c["G"])
    kstar, w, s = ops.edge_attn_fwd(g, Z, TEMP)
    dZ = torch.zeros_like(Z)
    r = torch.empty(n, K, dtype=torch.float32, device=DEV)
    dw = torch.empty(g.nnz, dtype=torch.float32, device=DEV)
    routed = torch.empty(n, dtype=torch.int32, device=DEV)
    for phase in (1, 2, 3):
        ops.factor_bwd_directed_phase(g, tg, tperm, Z, G, kstar, w, s, BETA, TEMP, dZ, r, dw, routed, phase)
    return dict(g=g, tg=tg, tperm=tperm, Z=Z, G=G, kstar=kstar, w=w, s=s, dZ=dZ, r=r, dw=dw, c=c)


# ------------------------------------------------------------------------------------------
# the phase entry point
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,d", [(8, 16), (5, 32), (1, 16), (7, 20)])
def test_phases_equal_the_whole_backward(dl, K, d):
    ops, Graph = dl
    f = full_run(ops, Graph, K, d)
    dZ, r = ops.factor_bwd_directed(f["g"], f["Z"], f["G"], f["kstar"], f["w"], f["s"], BETA, TEMP)
    assert np.array_equal(bits(dZ), bits(f["dZ"])) and np.array_equal(bits(r), bits(f["r"]))
    check_outputs(f"directed phases K={K} d={d}", dict(dZ=f["dZ"].cpu().numpy(), r=f["r"].cpu().numpy()),
                  f["c"]["ref"], names=("r", "dZ"))


def test_phase_bounds_are_checked(dl):
    from disenlink_b200._lib import lib, ptr, stream_of
    DL_EINVAL = -1
    ops, Graph = dl
    f = full_run(ops, Graph)
    g, tg, tperm = f["g"], f["tg"], f["tperm"]
    n, nnz = g.N, g.nnz
    K, d = K_, D_
    dZ = torch.zeros_like(f["Z"])
    dw = torch.empty(nnz, dtype=torch.float32, device=DEV)
    routed = torch.empty(n, dtype=torch.int32, device=DEV)
    ws, wst = g.hub_scratch(K * d), tg.hub_scratch(K * d)

    def call(phase, n_tot=n, n_rec=nnz, gg=g, tt=tg, tp=tperm):
        return lib().dl_factor_bwd_directed_phase(gg.ref, tt.ref, ptr(tp), ptr(f["Z"]), ptr(f["G"]), ptr(f["kstar"]),
                                                  ptr(f["w"]), ptr(f["s"]), K, d, BETA, 1.0 - BETA, TEMP, n_tot, n_rec,
                                                  ptr(dZ), ptr(f["r"]), ptr(dw), ptr(routed), ptr(ws), ptr(wst), phase,
                                                  stream_of(DEV))
    for phase in (1, 2, 3):
        assert call(phase) == 0
    assert call(0) == DL_EINVAL and call(4) == DL_EINVAL
    # a column of g at or above n_tot (n_tot >= N): phase 2 reads g's columns
    bad = Graph(g.rowptr, g.col.clone(), n, n_global=n + 1)
    bad.col[nnz // 2] = n
    assert call(2, gg=bad) == DL_EINVAL
    # a column of gt at or above n_tot: phases 1 and 3
    badt = Graph(tg.rowptr, tg.col.clone(), n, n_global=n + 1)
    badt.col[tg.nnz - 1] = n + 5
    assert call(1, tt=badt) == DL_EINVAL and call(3, tt=badt) == DL_EINVAL
    # a tperm value at or above n_rec: phases 1 and 3
    tp = tperm.clone()
    tp[3] = nnz
    assert call(1, tp=tp) == DL_EINVAL and call(3, tp=tp) == DL_EINVAL
    tp[3] = -1
    assert call(1, tp=tp, n_rec=nnz + 1) == DL_EINVAL
    # n_rec below g.nnz, n_tot below N, different N, row_base != 0
    assert call(2, n_rec=nnz - 1) == DL_EINVAL and call(2, n_tot=n - 1) == DL_EINVAL
    small = Graph(tg.rowptr[:n], tg.col[:int(tg.rowptr[n - 1].item())], n - 1)
    assert call(3, tt=small) == DL_EINVAL
    g.struct.row_base = 1
    try:
        assert call(2) == DL_EINVAL
    finally:
        g.struct.row_base = 0
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------
# the record push on one GPU (local buffers stand in for the peers' blocks)
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.uint8, torch.float32])
def test_push_entries_is_bit_exact(dl, dtype):
    from disenlink_b200 import ops
    g = torch.Generator().manual_seed(3)
    n = 100003
    if dtype == torch.uint8:
        src = torch.randint(0, 256, (n,), generator=g, dtype=torch.uint8).to(DEV)
    else:
        src = torch.randn(n, generator=g).to(DEV)
        src[7] = float("nan")
        src[8] = -0.0
    sizes = [0, 1, 4097, 70001, 3]
    idx = [torch.randint(0, n, (m,), generator=g, dtype=torch.int32).to(DEV) for m in sizes]
    fill = 0xAB if dtype == torch.uint8 else SENTINEL
    dst = [torch.full((m + 9,), fill, dtype=dtype, device=DEV) for m in sizes]
    blocks = [(dst[i][5:].data_ptr(), idx[i]) for i in range(len(sizes))]
    ops.push_entries(src, blocks)
    torch.cuda.synchronize()
    for i, m in enumerate(sizes):
        want = src[idx[i].long()]
        assert np.array_equal(bits(dst[i][5:5 + m]), bits(want))
        head, tail = dst[i][:5], dst[i][5 + m:]
        assert bool((head == fill).all()) and bool((tail == fill).all())
    ops.push_entries(src, [])                                         # no peers: a no-op


# ------------------------------------------------------------------------------------------
# one rank of the step on one GPU
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world,rank", [(2, 0), (2, 1), (8, 0), (8, 3), (8, 7)])
def test_directed_rank_on_one_gpu(dl, world, rank):
    from disenlink_b200.partition import CudaBackend, NodePartition, directed_in_view
    ops, Graph = dl
    src, dst, n, rowptr, col, cases = dir_graph()
    f = full_run(ops, Graph)
    ref = f["c"]["ref"]
    K, d = K_, D_
    src_t, dst_t = t(src), t(dst)
    part = NodePartition.nnz_balanced(src_t, dst_t, n, world, rank)
    lo, hi = part.lo, part.hi
    assert hi > lo
    be = CudaBackend()
    rowptr_l, col_g = be.build_csr_directed(src_t, dst_t, part)
    assert np.array_equal(rowptr_l.cpu().numpy(), rowptr[lo:hi + 1] - rowptr[lo])
    assert np.array_equal(col_g.cpu().numpy(), col[rowptr[lo]:rowptr[hi]])
    trowptr, tsrc, tperm, tail_off = directed_in_view(src_t, dst_t, part, rowptr_l, col_g)

    def remote(x):
        x = x.to(torch.int64)
        return x[(x < lo) | (x >= hi)]
    # DirectedPartitionedLinkStep.__init__ / HaloPlan.to_local without the process group (no pairs here)
    halo = torch.unique(torch.cat([remote(col_g), remote(tsrc)]))
    n_own, n_halo = hi - lo, int(halo.numel())
    n_tot = n_own + n_halo
    assert n_halo > 0

    def to_local(ids):
        own = (ids >= lo) & (ids < hi)
        pos = torch.searchsorted(halo, ids).clamp_(max=n_halo - 1)
        return torch.where(own, ids - lo, pos + n_own)
    g = be.make_graph(rowptr_l, to_local(col_g.to(torch.int64)).to(torch.int32), n_own, n_tot)
    gt = be.make_graph(trowptr, to_local(tsrc).to(torch.int32), n_own, n_tot)
    tperm = tperm.to(torch.int32)
    nnz = g.nnz
    n_tail = tail_off[-1] - tail_off[0]
    n_rec = nnz + n_tail
    assert n_tail > 0 and gt.nnz != nnz
    gid = torch.cat([torch.arange(lo, hi, device=DEV), halo])
    # global CSR index of every record: own entries, then the tail in (i, j) order
    trow = torch.repeat_interleave(torch.arange(n_own, device=DEV), trowptr[1:] - trowptr[:-1]) + lo
    tail_glob = torch.empty(n_tail, dtype=torch.int64, device=DEV)
    remote_in = tperm.long() >= nnz
    g_rowptr = t(rowptr)
    key_glob = torch.repeat_interleave(torch.arange(n, device=DEV), g_rowptr[1:] - g_rowptr[:-1]) * n + t(col).long()
    tail_glob[tperm.long()[remote_in] - nnz] = torch.searchsorted(key_glob, tsrc[remote_in] * n + trow[remote_in])
    rec_glob = torch.cat([torch.arange(rowptr[lo], rowptr[hi], device=DEV), tail_glob])

    f32 = dict(dtype=torch.float32, device=DEV)
    Z = f["Z"][gid].contiguous()
    G = f["G"][gid].contiguous()
    kstar = torch.full((n_rec,), 0xEE, dtype=torch.uint8, device=DEV)
    w = torch.full((n_rec,), SENTINEL, **f32)
    dw = torch.full((n_rec,), SENTINEL, **f32)
    s = torch.full((n_tot, K), SENTINEL, **f32)
    # the record tails, as the pushes would deliver them
    kstar[nnz:] = f["kstar"][tail_glob]
    w[nnz:] = f["w"][tail_glob]
    dw[nnz:] = f["dw"][tail_glob]
    tails = [x[nnz:].clone() for x in (kstar, w, dw)]

    be.edge_attn_fwd(g, Z, TEMP, kstar, w, s)
    assert bool((s[n_own:] == SENTINEL).all())
    assert np.array_equal(bits(kstar), bits(f["kstar"][rec_glob])), "kstar (own + tail) differs from one GPU"
    assert np.array_equal(bits(w), bits(f["w"][rec_glob])), "w (own + tail) differs from one GPU"
    assert relerr(s[:n_own].cpu().numpy(), f["s"][lo:hi].cpu().numpy()) < ORA_TOL
    s[n_own:] = f["s"][gid][n_own:]                                   # the push of s
    dZ = torch.full((n_tot, K, d), SENTINEL, **f32)
    dZ[:n_own] = 0
    r = torch.full((n_tot, K), SENTINEL, **f32)
    routed = torch.empty(n_own, dtype=torch.int32, device=DEV)

    def backward(s_in):
        dZ[:n_own] = 0
        for phase in (1, 2, 3):
            be.factor_bwd_directed_phase(g, gt, tperm, Z, G, kstar, w, s_in, BETA, TEMP, dZ, r, dw, routed, phase)
            assert bool((dZ[n_own:] == SENTINEL).all()) and bool((r[n_own:] == SENTINEL).all())
            for x, x0 in zip((kstar, w, dw), tails):
                assert np.array_equal(bits(x[nnz:]), bits(x0)), f"record tail written in phase {phase}"
        return dZ[:n_own].clone(), r[:n_own].clone()
    dZ_own, r_own = backward(s)
    own = slice(lo, hi)
    rf = dict(r=ref["r"][own], A_r=ref["A_r"][own], dZ=ref["dZ"][own])
    check_outputs(f"directed partition world={world} rank={rank}",
                  dict(r=r_own.cpu().numpy(), dZ=dZ_own.cpu().numpy()), rf, names=("r", "dZ"))
    # hub segments depend on a row's degree only: on the single-GPU inputs (its s) the owned rows are bitwise equal
    s[:n_own] = f["s"][lo:hi]
    dZ_b, r_b = backward(s)
    assert np.array_equal(bits(dZ_b), bits(f["dZ"][lo:hi])), "owned dZ differs from the single-GPU backward"
    assert np.array_equal(bits(r_b), bits(f["r"][lo:hi]))
    assert np.array_equal(bits(dw[:nnz]), bits(f["dw"][rowptr[lo]:rowptr[hi]]))


# ------------------------------------------------------------------------------------------
# the step at world 1
# ------------------------------------------------------------------------------------------
def test_world1_in_view_equals_transpose_view(dl):
    from disenlink_b200.partition import CudaBackend, NodePartition, directed_in_view
    ops, Graph = dl
    src, dst, n, rowptr, col, cases = dir_graph()
    part = NodePartition(n, 1, 0)
    rp, cg = CudaBackend().build_csr_directed(t(src), t(dst), part)
    trowptr, tsrc, tperm, tail_off = directed_in_view(t(src), t(dst), part, rp, cg)
    tg, tp = Graph.from_edges(t(src), t(dst), n, directed=True).transpose_view()
    assert torch.equal(trowptr, tg.rowptr) and torch.equal(tsrc.to(torch.int32), tg.col)
    assert torch.equal(tperm.to(torch.int32), tp) and tail_off == [0, 0]
    assert np.array_equal(tp.cpu().numpy(), transpose_of(rowptr, col)[2])


def test_world1_step_matches_the_fused_loss(dl):
    from disenlink_b200.partition import DirectedPartitionedLinkStep
    ops, Graph = dl
    src, dst, n, rowptr, col, cases = dir_graph()
    c = dir_case(K_, D_)
    rng = np.random.default_rng(5)
    P = 20000
    u = t(np.concatenate([rng.integers(0, n, P - 500), np.full(500, int(cases["in_hubs"][0]))]))
    v = t(rng.integers(0, n, P))
    lab = t((rng.random(P) < 0.3).astype(np.float32))
    wts = torch.full((P,), 1.0 / P, device=DEV)
    step = DirectedPartitionedLinkStep(t(src), t(dst), n, u, v, lab, wts, K_, D_, BETA, TEMP)
    assert step.n_tail == 0
    step.run(t(c["Z"]))
    g = Graph.from_edges(t(src), t(dst), n, directed=True)
    Z = t(c["Z"]).requires_grad_(True)
    loss, prob, H = ops.link_bce_loss(Z, g, ops.PairBatch(u, v, n), lab, wts, BETA, TEMP)
    loss.backward()
    assert abs(float(step.loss) - float(loss)) <= ORA_TOL * abs(float(loss))
    assert relerr(step.prob[:P].cpu().numpy(), prob.detach().cpu().numpy()) < ORA_TOL
    assert relerr(step.dZ.cpu().numpy(), Z.grad.cpu().numpy()) < 5 * ORA_TOL
    step.close()
