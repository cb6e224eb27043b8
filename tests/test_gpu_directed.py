"""GPU suite of the directed backward (csrc/bwd_dir.cu, ops.factor_bwd_directed) on graphs marked directed:
integer prep bit-exact, routing bit-exact with the oracle, dZ and r within the per-element bounds of
test_gpu_kernel_paths.py against the float64 reference, determinism, the module and the fused loss."""
from functools import lru_cache

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_directed import RefDir64, csr_of, directed_cases, directed_graph, in_only_pairs, transpose_of
from test_gpu_kernel_paths import BETA, PATH_SHAPES, TEMP, case_inputs, check_outputs, hard_case, shape_case
from test_gpu_parity import ORA_TOL, dl, relerr, t  # noqa: F401  (dl is a fixture)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DIR_SHAPES = PATH_SHAPES + [(1, 16)]


@lru_cache(maxsize=None)
def dir_graph():
    n = 6000
    src, dst = directed_graph(n, 20000, 11)
    rowptr, col = csr_of(src, dst, n)
    return src, dst, n, rowptr, col, directed_cases(rowptr, col)


@lru_cache(maxsize=None)
def dir_case(K, d):
    from oracle import oracle as O
    src, dst, n, rowptr, col, cases = dir_graph()
    Z, G, _, _, _ = case_inputs(n, K, d, int(cases["in_hubs"][0]), 7000 + K * 1000 + d)
    o_k, o_w, o_s = O.edge_attn_fwd(rowptr, col, Z, TEMP)
    ref = RefDir64(rowptr, col, Z, o_k, BETA, TEMP)
    res = ref.forward_dict()
    res.update(ref.factor_bwd(G))
    return dict(Z=Z, G=G, o_k=o_k, o_w=o_w, ref=res)


def run_directed(ops, g, Z, G):
    Zt = t(Z)
    kstar, w, s = ops.edge_attn_fwd(g, Zt, TEMP)
    dZ, r = ops.factor_bwd_directed(g, Zt, t(G), kstar, w, s, BETA, TEMP)
    cpu = lambda x: x.cpu().numpy()
    return dict(kstar=cpu(kstar), w=cpu(w), s=cpu(s), dZ=cpu(dZ), r=cpu(r))


def test_graph_and_transpose_are_bit_exact(dl):
    ops, Graph = dl
    src, dst, n, rowptr, col, cases = dir_graph()
    g = Graph.from_edges(t(src), t(dst), n, directed=True)
    assert g.directed
    assert np.array_equal(g.rowptr.cpu().numpy(), rowptr) and np.array_equal(g.col.cpu().numpy(), col)
    tg, tperm = g.transpose_view()
    trowptr, tcol, tp = transpose_of(rowptr, col)
    assert np.array_equal(tg.rowptr.cpu().numpy(), trowptr)
    assert np.array_equal(tg.col.cpu().numpy(), tcol)
    assert np.array_equal(tperm.cpu().numpy(), tp)
    assert tg.n_hub == int((np.diff(trowptr) >= 512).sum()) > 0
    # edge_index / dense / csr constructors keep the pattern as given and carry the mark
    ei = torch.stack([t(src), t(dst)])
    for h in (Graph.from_edge_index(ei, n, directed=True), Graph.from_csr(t(rowptr), t(col), directed=True)):
        assert h.directed and np.array_equal(h.col.cpu().numpy(), col)
    assert not Graph.from_edge_index(ei, n).directed


@pytest.mark.parametrize("K,d", DIR_SHAPES)
def test_directed_backward_vs_ref64(dl, K, d):
    ops, Graph = dl
    src, dst, n, rowptr, col, cases = dir_graph()
    c = dir_case(K, d)
    g = Graph.from_edges(t(src), t(dst), n, directed=True)
    out = run_directed(ops, g, c["Z"], c["G"])
    assert np.array_equal(out["kstar"], c["o_k"]), f"{(out['kstar'] != c['o_k']).sum()} routing mismatches"
    assert np.array_equal(out["w"].view(np.uint32), c["o_w"].view(np.uint32)), "w not bit-identical"
    if K > 1:
        assert in_only_pairs(rowptr, col, c["o_k"], K).size      # the clamp rule is exercised
    check_outputs(f"directed K={K} d={d}", out, c["ref"], names=("s", "r", "dZ"))
    clamp = in_only_pairs(rowptr, col, c["o_k"], K)
    assert np.all(out["r"][clamp[:, 0], clamp[:, 1]] == 0.0)
    # run to run: bitwise
    again = run_directed(ops, g, c["Z"], c["G"])
    for k in ("dZ", "r"):
        assert np.array_equal(out[k].view(np.uint32), again[k].view(np.uint32)), k


@pytest.mark.parametrize("K,d", [(8, 16), (5, 32), (1, 16), (7, 20)])
def test_symmetric_graph_marked_directed(dl, K, d):
    """The same symmetric pattern through the directed backward and through the symmetric one: both within the
    bounds of the float64 reference."""
    ops, Graph = dl
    src, dst, n, rowptr, col, cases = hard_case("shift0")
    c = shape_case("shift0", K, d)
    g = Graph.from_edges(t(src), t(dst), n, symmetrize=True, directed=True)
    assert g.directed and np.array_equal(g.col.cpu().numpy(), col)
    out = run_directed(ops, g, c["Z"], c["G"])
    check_outputs(f"marked symmetric K={K} d={d}", out, c["ref"], names=("s", "r", "dZ"))
    u = Graph.from_edges(t(src), t(dst), n)
    Zt = t(c["Z"])
    kstar, w, s = ops.edge_attn_fwd(u, Zt, TEMP)
    dZ, r = ops.factor_bwd(u, Zt, t(c["G"]), kstar, w, s, BETA, TEMP)
    check_outputs(f"unmarked symmetric K={K} d={d}", dict(dZ=dZ.cpu().numpy(), r=r.cpu().numpy()), c["ref"],
                  names=("r", "dZ"))


def _module(N, seed=0):
    from disenlink_b200.model import Disentangle
    torch.manual_seed(seed)
    m = Disentangle(24, 16, 8, nfactor=4, beta=0.6, t=1)
    x = torch.randn(N, 24)
    rng = np.random.default_rng(seed)
    adj = torch.from_numpy((rng.random((N, N)) < 0.01).astype(np.float32))
    adj[torch.arange(0, N, 9), torch.arange(0, N, 9)] = 1
    assert not torch.equal(adj, adj.t())
    pu, pv = torch.from_numpy(rng.integers(0, N, 3000)), torch.from_numpy(rng.integers(0, N, 3000))
    lab = torch.from_numpy((rng.random(3000) < 0.4).astype(np.float32))
    return m, x, adj, pu, pv, lab


def _reference_grads(m, x, adj, pu, pv, lab):
    """model.py's forward (dense_forward) + autograd in float64 on the CPU."""
    import copy
    from test_oracle_live_reference import dense_forward
    m64 = copy.deepcopy(m).cpu().double()
    Z = m64.project(x.double())
    K = Z.shape[1]
    _, _, _, link_pred = dense_forward([Z[:, k, :] for k in range(K)], adj.double(), m64.beta, float(m64.temperature))
    loss = F.binary_cross_entropy(link_pred[pu, pv], lab.double())
    loss.backward()
    return loss.item(), {k: p.grad.numpy() for k, p in m64.named_parameters()}


def test_module_directed_dense_graph_and_fused_loss(dl):
    TOL = 1e-5
    ops, Graph = dl
    N = 500
    m, x, adj, pu, pv, lab = _module(N)
    ref_loss, ref_grads = _reference_grads(m, x, adj, pu, pv, lab)
    m = m.to(DEV)
    xd, adjd, pud, pvd, labd = (a.to(DEV) for a in (x, adj, pu, pv, lab))
    # an unmarked asymmetric adj still refuses the backward
    from disenlink_b200._lib import DL_EASYM, DlError
    H, link_pred = m(xd, adjd)
    with pytest.raises(DlError) as ei:
        F.binary_cross_entropy(link_pred[pud, pvd], labd).backward()
    assert ei.value.code == DL_EASYM
    m.zero_grad()
    # (a) dense adj, module marked directed
    m.adjacency = "directed"
    H, link_pred = m(xd, adjd)
    loss = F.binary_cross_entropy(link_pred[pud, pvd], labd)
    loss.backward()
    assert abs(loss.item() - ref_loss) < TOL * abs(ref_loss)
    for k, p in m.named_parameters():
        assert relerr(p.grad.cpu().numpy(), ref_grads[k]) < 5 * TOL, k
    # (b) a marked Graph handle + LinkScorer, whatever the module's setting
    m.adjacency = "symmetric"
    m.zero_grad()
    rows, cols = adjd.nonzero(as_tuple=True)
    graph = Graph.from_edges(rows, cols, N, directed=True)
    H2, scorer = m(xd, graph)
    loss2 = F.binary_cross_entropy(scorer(torch.stack([pud, pvd])), labd)
    loss2.backward()
    assert abs(loss2.item() - ref_loss) < TOL * abs(ref_loss)
    for k, p in m.named_parameters():
        assert relerr(p.grad.cpu().numpy(), ref_grads[k]) < 5 * TOL, k
    # (c) edge_index and sparse adj under adjacency = "directed" build marked graphs of the same pattern
    m.adjacency = "directed"
    for a in (torch.stack([rows, cols]), adjd.to_sparse()):
        g2 = m.disentangle_layer1._cache.get(a, N, True)
        assert g2.directed and torch.equal(g2.col, graph.col) and torch.equal(g2.rowptr, graph.rowptr)
    # (d) the fused loss on the marked graph (weights 1/P: the mean BCE): loss and every parameter gradient
    # against model.py's forward + autograd in float64
    m.zero_grad()
    batch = ops.PairBatch(pud, pvd, N)
    wts = torch.full((pud.numel(),), 1.0 / pud.numel(), device=DEV)
    loss3, prob, H3 = ops.link_bce_loss(m.project(xd), graph, batch, labd, wts, m.beta, 1.0)
    loss3.backward()
    assert abs(loss3.item() - ref_loss) < TOL * abs(ref_loss)
    for k, p in m.named_parameters():
        assert relerr(p.grad.cpu().numpy(), ref_grads[k]) < 5 * TOL, k


def test_partitioned_step_refuses_directed_training(dl):
    """The node-partitioned step always symmetrises its edge columns; asking it to train on them as given is
    refused before any work."""
    ops, Graph = dl
    from disenlink_b200.partition import PartitionedLinkStep
    src, dst = t(np.array([0, 1])), t(np.array([1, 2]))
    with pytest.raises(ValueError, match="directed"):
        PartitionedLinkStep(src, dst, 3, None, None, None, None, 2, 4, 0.5, 1.0, directed=True)


@pytest.mark.parametrize("graph_src", ["synthetic", "cora_train_columns"])
def test_train_link_directed(graph_src):
    """examples/train_link.py --directed for 20 epochs: the directed train adjacency (asymmetric: 85 % of the
    columns), finite loss falling over the run, validation AUC reported.  The Cora case uses the real Cora train
    columns of the golden fixture with random features (the datasets are not shipped)."""
    import argparse
    import os
    import sys
    from conftest import load_golden
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples"))
    import train_link
    torch.manual_seed(0)
    if graph_src == "synthetic":
        x, edge_index, _ = train_link.synthetic(n=2000, seed=0)
    else:
        g = load_golden("cora_K3_d32")
        x = torch.randn(int(g["N"]), 64)
        edge_index = torch.stack([torch.from_numpy(g["src"]), torch.from_numpy(g["dst"])])
    args = argparse.Namespace(nfactor=3, nhidden=64, nembed=32, beta=0.9, temperature=1, m=2, lr=0.01,
                              epochs=20, seed=0, log_every=1000, standardize=True, directed=True)
    out = train_link.run(args, x, edge_index, torch.device(DEV), log=lambda *_: None)
    losses = [l for l, _ in out["history"]]
    assert len(losses) == 20 and np.all(np.isfinite(losses))
    assert losses[-1] < losses[0]
    assert 0.0 < out["best_val_auc"] <= 1.0 and np.isfinite(out["test_auc"])
