"""torch.autograd bindings of the hot-path kernels (C ABI in include/disenlink_b200.h).

    factor_aggregate(Z, graph, beta, T)  -> H            model.py:56-75   (attention + aggregation; any
                                                         pattern when the graph is marked directed)
    PairBatch(u, v, N) / pair_score(Z, H, batch, T)      model.py:109-113 on explicit pairs
    allpairs_score(Z, H, T)              -> [N,N]        model.py:109-113 dense (small-N drop-in)

Everything runs on the tensors' CUDA device through libdisenlink_b200.so; nothing here has a CPU
implementation.
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib
from ._lib import check, lib, ptr, require_cuda, stream_of
from .graph import Graph


def one_minus(beta: float) -> float:
    """(1 - beta) evaluated in double like Python does at model.py:75, rounded to fp32 by ctypes."""
    return 1.0 - float(beta)


def _check_Z(Z: torch.Tensor, n_nodes: int):
    require_cuda(Z, "Z")
    if Z.dim() != 3 or Z.shape[0] != n_nodes:
        raise ValueError(f"Z must be [N={n_nodes}, K, d], got {tuple(Z.shape)}")
    if Z.dtype != torch.float32:
        raise TypeError("Z must be float32 (parity target is the reference's fp32 path)")
    K, d = int(Z.shape[1]), int(Z.shape[2])
    if not (1 <= K <= _lib.DL_MAX_K and 1 <= d <= _lib.DL_MAX_D):
        raise ValueError(f"unsupported factor shape K={K}, d={d} (K <= {_lib.DL_MAX_K}, d <= {_lib.DL_MAX_D})")
    return K, d


# --------------------------------------------------------------------------------------------
# raw kernel wrappers (no autograd)
# --------------------------------------------------------------------------------------------
def edge_attn_fwd(graph: Graph, Z: torch.Tensor, T: float = 1.0, out=None, plan: dict = None):
    """-> (kstar u8 [nnz], w f32 [nnz], s f32 [N,K]).  [ref: model.py:56-73]
    `out` = optional preallocated (kstar, w, s).  `plan` = the bwd_plan of the backward that follows with the
    same Z and T: in mode "sym" the symmetric attention leaves its softmax in plan["coef"] and sets
    plan["a_valid"], and backward pass 2 reads it instead of recomputing it (off under DL_F_NO_KEEPA)."""
    K, d = _check_Z(Z, graph.n_global)
    Z = Z.contiguous()
    dev = Z.device
    with torch.cuda.device(dev):
        if out is not None:
            kstar, w, s = out
        else:
            kstar = torch.empty(max(graph.nnz, 1), dtype=torch.uint8, device=dev)
            w = torch.empty(max(graph.nnz, 1), dtype=torch.float32, device=dev)
            s = torch.empty(graph.n_global, K, dtype=torch.float32, device=dev)
        rc = _lib.DL_EUNSUPPORTED
        sym = None
        a_out = None
        if plan is not None:
            plan["a_valid"] = False
            if plan["mode"] == "sym" and not (graph.flags & _lib.DL_F_NO_KEEPA):
                a_out = plan["coef"]
        if graph.nnz >= graph.sym_min_nnz and not (graph.flags & (_lib.DL_F_NO_SYM | _lib.DL_F_NO_STREAM |
                                                                  _lib.DL_F_NO_FL | _lib.DL_F_NO_FL_ATTN)):
            sym = graph.sym_view()              # None: not symmetric / row-partitioned
        if sym is not None:
            # every undirected edge once: rows are gathered for the upper-triangle entries only
            upper, eidx = sym
            kw = _x_scratch(graph, 2 * upper.nnz)
            rc = lib().dl_edge_attn_fwd_sym(graph.ref, upper.ref, ptr(eidx), ptr(Z), K, d, float(T), ptr(kstar),
                                            ptr(w), ptr(s), ptr(graph.hub_scratch(K)), ptr(kw), _optr(a_out),
                                            stream_of(dev))
            if rc != _lib.DL_EUNSUPPORTED:
                check(rc, "dl_edge_attn_fwd_sym")
                if a_out is not None:
                    plan["a_valid"] = True
        if rc == _lib.DL_EUNSUPPORTED:
            check(lib().dl_edge_attn_fwd(graph.ref, ptr(Z), K, d, float(T), ptr(kstar), ptr(w), ptr(s),
                                         ptr(graph.hub_scratch(K)), stream_of(dev)), "dl_edge_attn_fwd")
    return kstar[:graph.nnz], w[:graph.nnz], s


def _optr(t):
    return ptr(t) if t is not None else None


def factor_spmm_fwd(graph: Graph, Z, kstar, w, s, beta: float, out=None, sj=None, zs=None):
    """-> H [N,K,d].  [ref: model.py:75]  `sj` = optional f32 [nnz] buffer that receives s[col, kstar]
    per entry (pass it on to factor_bwd / factor_bwd_edges).  `zs` = optional [N,K,d] scratch: the
    kernel then gathers slices pre-divided by s (one DRAM transaction per entry instead of two); only
    for graphs that are not row-partitioned, and exclusive with `sj`."""
    if zs is not None and (sj is not None or graph.row_base != 0):
        raise ValueError("zs needs row_base == 0 (one GPU or a rank-local index space) and excludes sj")
    K, d = _check_Z(Z, graph.n_global)
    Z = Z.contiguous()
    dev = Z.device
    with torch.cuda.device(dev):
        H = torch.empty_like(Z) if out is None else out
        check(lib().dl_factor_spmm_fwd(graph.ref, ptr(Z), ptr(kstar), ptr(w), ptr(s), K, d,
                                       float(beta), one_minus(beta), ptr(H), _optr(sj), _optr(zs),
                                       int(Z.shape[0]) if zs is not None else 0,
                                       ptr(graph.hub_scratch(K * d)), stream_of(dev)),
              "dl_factor_spmm_fwd")
    return H


def _x_scratch(graph: Graph, n_floats: int = 0):
    """Per-entry fp32 scratch cached on the graph handle: pass 1 of the backward leaves
    <G[j,k*], Z[i,k*]> per entry there for pass 2 (nnz floats); the symmetric attention keeps its
    packed (w, kstar) records of the upper-triangle entries there during the forward (2 nnz_u floats)."""
    need = max(graph.nnz + graph.N + 8, int(n_floats), 1)       # 2 nnz_u = nnz + #self-loops <= nnz + N
    buf = getattr(graph, "_x_scratch", None)
    if buf is None or buf.numel() < need:
        buf = torch.empty(need, dtype=torch.float32, device=graph.device)
        graph._x_scratch = buf
    return buf


def bwd_plan(graph: Graph, K: int, d: int, allow_sym: bool = True) -> dict:
    """How the two backward passes of one step talk to each other.
      mode "sym"   (symmetric, not row-partitioned graphs with a factor-per-lane kernel): pass 1 leaves
                   <G[j,k*], Z[i,k*]> and kstar of the entries with col >= row in upper-view order, pass 2
                   evaluates every undirected edge once (dl_factor_bwd_edges_sym); needs nnz_u*K floats of
                   transient scratch -- when that does not fit, mode "x" is used
      mode "x"     pass 1 leaves the per-entry dots for every entry, pass 2 reads them (dl_factor_bwd_edges)
    The per-entry scratch is the graph's cached one (shared with the symmetric attention's packed records,
    which are dead by the time the backward runs).  In mode "sym", a forward given the plan (edge_attn_fwd)
    stores the softmax of the upper entries in "coef" and sets "a_valid"; pass 2 then reads it and clears
    "a_valid", since the buffer holds coefficients afterwards."""
    plan = {"mode": "x", "x": _x_scratch(graph), "x_valid": False, "a_valid": False}
    f = graph.flags
    if (allow_sym and graph.nnz >= graph.sym_min_nnz and graph.nnz > 0 and
            not (f & (_lib.DL_F_NO_SYM | _lib.DL_F_NO_STREAM | _lib.DL_F_NO_FL | _lib.DL_F_NO_XDOT)) and
            lib().dl_factor_bwd_edges_sym_supported(K, d) and graph.sym_view() is not None):
        upper, eidx = graph.sym_view()
        lower, lmirror = graph.sym_lower_view()
        nu = upper.nnz
        # 4K bytes per undirected edge of scratch (16 GB at nnz = 10^9, K = 8): only when it leaves room for
        # the rest of the step (a caller that double-buffers 25-GB inputs is better served by the two-sided pass)
        need = nu * K * 4
        free_b, _ = torch.cuda.mem_get_info(graph.device)
        cached = torch.cuda.memory_reserved(graph.device) - torch.cuda.memory_allocated(graph.device)
        if need + (8 << 30) > free_b + cached and need > (64 << 20):
            return plan
        try:
            coef = torch.empty(max(nu * K, 1), dtype=torch.float32, device=graph.device)
        except torch.cuda.OutOfMemoryError:
            return plan
        scr = _x_scratch(graph, nu + (nu + 3) // 4 + 1)
        plan.update(mode="sym", xu=scr[:nu], ku=scr[nu:nu + (nu + 3) // 4 + 1].view(torch.uint8), coef=coef,
                    upper=upper, eidx=eidx, lower=lower, lmirror=lmirror)
    return plan


def factor_bwd_gather(graph: Graph, Z, G, kstar, w, s, beta: float, dZ, r, plan: dict = None, peers=None):
    """Pass 1 of the backward: r [N,K] and dZ += beta*G + T_ (see csrc/factor_bwd.cu).
    `plan` = bwd_plan(...) (None: no per-entry dots are kept, pass 2 re-gathers the G slices); its "x_valid"
    is set when the dots were filled.  `peers` = ctypes array of the peers' copies of r (replicated layout:
    the all-gather of r rides on the kernel)."""
    K, d = _check_Z(Z, graph.n_global)
    dev = Z.device
    x_valid = ctypes.c_int(0)
    x = xi = ku = None
    if plan is not None:
        if plan["mode"] == "sym":
            x, xi, ku = plan["xu"], plan["eidx"], plan["ku"]
        else:
            x = plan["x"]
    with torch.cuda.device(dev):
        if peers is None:
            check(lib().dl_factor_bwd_gather(graph.ref, ptr(Z), ptr(G), ptr(kstar), ptr(w), ptr(s), K, d,
                                             float(beta), one_minus(beta), ptr(dZ), ptr(r), _optr(x), _optr(xi),
                                             _optr(ku), ctypes.byref(x_valid), ptr(graph.hub_scratch(K * d)),
                                             stream_of(dev)), "dl_factor_bwd_gather")
        else:
            check(lib().dl_factor_bwd_gather_push(graph.ref, ptr(Z), ptr(G), ptr(kstar), ptr(w), ptr(s), K, d,
                                                  float(beta), one_minus(beta), ptr(dZ), ptr(r),
                                                  _optr(x) if xi is None else None,
                                                  ctypes.byref(x_valid), ptr(graph.hub_scratch(K * d)),
                                                  peers, len(peers), stream_of(dev)),
                  "dl_factor_bwd_gather_push")
    if plan is not None:
        plan["x_valid"] = bool(x_valid.value)
    return bool(x_valid.value)


def _sr_scratch(graph: Graph, s):
    """[n, K, 2] scratch in which pass 2 interleaves (s, r) -- cached on the graph handle."""
    buf = getattr(graph, "_sr_scratch", None)
    if buf is None or buf.shape[0] != s.shape[0] or buf.shape[1] != s.shape[1] or buf.device != s.device:
        buf = torch.empty(s.shape[0], s.shape[1], 2, dtype=torch.float32, device=s.device)
        graph._sr_scratch = buf
    return buf


def factor_bwd_edges(graph: Graph, Z, G, kstar, w, s, r, beta: float, T: float, dZ, sj=None, plan: dict = None):
    """Pass 2 of the backward: dZ += attention-weight terms (needs r of every neighbour).
    `plan` = the bwd_plan factor_bwd_gather was given."""
    K, d = _check_Z(Z, graph.n_global)
    dev = Z.device
    valid = plan is not None and plan.get("x_valid")
    with torch.cuda.device(dev):
        if valid and plan["mode"] == "sym":
            a_valid = 1 if plan.get("a_valid") else 0
            plan["a_valid"] = False                        # from here on coef holds coefficients
            check(lib().dl_factor_bwd_edges_sym(plan["upper"].ref, plan["lower"].ref, ptr(plan["lmirror"]), ptr(Z), ptr(G),
                                                ptr(plan["ku"]), ptr(s), ptr(r), ptr(_sr_scratch(graph, s)),
                                                int(s.shape[0]), ptr(plan["xu"]), ptr(plan["coef"]), K, d,
                                                one_minus(beta), float(T), a_valid, ptr(dZ),
                                                ptr(graph.hub_scratch(K * d)), stream_of(dev)), "dl_factor_bwd_edges_sym")
            return
        if plan is not None and plan["mode"] == "sym":
            raise RuntimeError("pass 1 did not fill the upper-view dots the symmetric pass 2 was planned on")
        check(lib().dl_factor_bwd_edges(graph.ref, ptr(Z), ptr(G), ptr(kstar), ptr(w), ptr(s), ptr(r), _optr(sj),
                                        ptr(_sr_scratch(graph, s)), int(s.shape[0]),
                                        ptr(plan["x"]) if valid else None, K, d,
                                        one_minus(beta), float(T), ptr(dZ),
                                        ptr(graph.hub_scratch(K * d)), stream_of(dev)),
              "dl_factor_bwd_edges")


def factor_bwd(graph: Graph, Z, G, kstar, w, s, beta: float, T: float = 1.0, dZ=None, r=None, sj=None):
    """dL/dZ through attention + aggregation given G = dL/dH; accumulated into dZ if given.
    -> (dZ, r).  [ref: autograd of model.py:56-75]"""
    K, d = _check_Z(Z, graph.n_global)
    Z = Z.contiguous()
    G = G.contiguous()
    dev = Z.device
    with torch.cuda.device(dev):
        if dZ is None:
            dZ = torch.zeros_like(Z)
        if r is None:
            r = torch.empty(graph.n_global, K, dtype=torch.float32, device=dev)
    plan = bwd_plan(graph, K, d)
    factor_bwd_gather(graph, Z, G, kstar, w, s, beta, dZ, r, plan=plan)
    if plan["mode"] == "sym" and not plan["x_valid"]:            # pass 1 took a path without dots: plain pass 2
        plan = None
    factor_bwd_edges(graph, Z, G, kstar, w, s, r, beta, T, dZ, sj=sj, plan=plan)
    return dZ, r


def factor_bwd_directed(graph: Graph, Z, G, kstar, w, s, beta: float, T: float = 1.0, dZ=None, r=None):
    """dL/dZ through attention + aggregation for ANY 0/1 pattern (graphs marked directed), given
    G = dL/dH; accumulated into dZ if given.  Gathers over the pattern and its transpose
    (Graph.transpose_view; csrc/bwd_dir.cu).  -> (dZ, r), r = 0 where a (node, factor) has no routed
    out-entry.  [ref: autograd of model.py:56-75]"""
    K, d = _check_Z(Z, graph.n_global)
    Z = Z.contiguous()
    G = G.contiguous()
    dev = Z.device
    tg, tperm = graph.transpose_view()
    with torch.cuda.device(dev):
        if dZ is None:
            dZ = torch.zeros_like(Z)
        if r is None:
            r = torch.empty(graph.N, K, dtype=torch.float32, device=dev)
        routed = torch.empty(max(graph.N, 1), dtype=torch.int32, device=dev)
        check(lib().dl_factor_bwd_directed(graph.ref, tg.ref, ptr(tperm), ptr(Z), ptr(G), ptr(kstar), ptr(w), ptr(s),
                                           K, d, float(beta), one_minus(beta), float(T), ptr(dZ), ptr(r),
                                           ptr(_x_scratch(graph)), ptr(routed), _optr(graph.hub_scratch(K * d)),
                                           _optr(tg.hub_scratch(K * d)), stream_of(dev)), "dl_factor_bwd_directed")
    return dZ, r


def factor_bwd_directed_phase(graph: Graph, tgraph: Graph, tperm, Z, G, kstar, w, s, beta: float, T: float, dZ, r,
                              dw, routed, phase: int):
    """One phase of factor_bwd_directed (dl_factor_bwd_directed_phase) on rank-local graphs: 1 = pass 1 over the
    in-entries (r, dZ += beta G + T_), 2 = pass 2 out-side (writes dw of the own entries), 3 = pass 2 in-side
    (reads kstar, dw through tperm).  `graph` / `tgraph`: the owned rows and their in-entries (same N, row_base 0),
    columns below Z.shape[0]; kstar, w, dw: the per-entry records [own entries | records of remote in-entries],
    every tperm value below their length.  `routed`: int32 [N] scratch of phase 1."""
    K, d = int(Z.shape[1]), int(Z.shape[2])
    dev = Z.device
    n_rec = min(int(kstar.numel()), int(dw.numel()) if dw is not None else 1 << 62,
                int(w.numel()) if w is not None else 1 << 62)
    with torch.cuda.device(dev):
        check(lib().dl_factor_bwd_directed_phase(graph.ref, tgraph.ref, ptr(tperm), ptr(Z), _optr(G), ptr(kstar),
                                                 _optr(w), _optr(s), K, d, float(beta), one_minus(beta), float(T),
                                                 int(Z.shape[0]), n_rec, ptr(dZ), _optr(r), _optr(dw), _optr(routed),
                                                 _optr(graph.hub_scratch(K * d)), _optr(tgraph.hub_scratch(K * d)),
                                                 int(phase), stream_of(dev)), "dl_factor_bwd_directed_phase")


def push_entries(src: torch.Tensor, blocks):
    """dl_push_entries: for every (dst, src_idx) of `blocks`, dst[t] = src[src_idx[t]] (t < len(src_idx)); dst is
    a tensor or the device address of a peer's block (same element type as src: 1 or 4 bytes).  One launch."""
    from ._lib import DlPushDesc
    if src.element_size() not in (1, 4):
        raise ValueError("push_entries moves 1- or 4-byte elements")
    dev = src.device
    descs = (DlPushDesc * max(len(blocks), 1))()
    for i, (dst, idx) in enumerate(blocks):
        if idx.dtype != torch.int32 or idx.device != src.device:
            raise ValueError("push_entries: source indices must be int32 on the source's device")
        descs[i].dst = dst.data_ptr() if torch.is_tensor(dst) else dst
        descs[i].src_idx = idx.data_ptr() if idx.numel() else None
        descs[i].dst_idx = None
        descs[i].mask = None
        descs[i].n = int(idx.numel())
    with torch.cuda.device(dev):
        check(lib().dl_push_entries(ptr(src), src.element_size(), descs, len(blocks), stream_of(dev)),
              "dl_push_entries")


class PairBatch:
    """A batch of (u,v) node pairs resident on the GPU (int32 ids), plus -- built lazily, once --
    the node-major incidence lists the atomic-free backward walks.

    The training script's pair sets are fixed per run (main_disentangled.py:154-166), so one
    PairBatch per split is built up front and reused every epoch."""

    def __init__(self, u: torch.Tensor, v: torch.Tensor, n_nodes: int):
        require_cuda(u, "u")
        if u.shape != v.shape or u.dim() != 1:
            raise ValueError("u and v must be 1-D tensors of equal length")
        self.N = int(n_nodes)
        self.P = int(u.numel())
        if self.P:
            lo = int(torch.minimum(u.min(), v.min()).item())
            hi = int(torch.maximum(u.max(), v.max()).item())
            if lo < 0 or hi >= self.N:
                raise _lib.DlError(-3, "PairBatch")
        self.u = u.to(torch.int32).contiguous()
        self.v = v.to(torch.int32).contiguous()
        self.device = u.device
        self._inc = None

    @classmethod
    def from_pairs(cls, pairs: torch.Tensor, n_nodes: int) -> "PairBatch":
        return cls(pairs[0], pairs[1], n_nodes)

    def incidence(self):
        """-> (Graph over incidence lists, inc_pair int32 [2P])."""
        if self._inc is None:
            dev, P, N = self.device, self.P, self.N
            L = lib()
            with torch.cuda.device(dev):
                inc_ptr = torch.empty(N + 1, dtype=torch.int64, device=dev)
                inc_other = torch.empty(max(2 * P, 1), dtype=torch.int32, device=dev)
                inc_pair = torch.empty(max(2 * P, 1), dtype=torch.int32, device=dev)
                ws_bytes = L.dl_pair_incidence_workspace_bytes(P, N)
                ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
                check(L.dl_pair_incidence(ptr(self.u), ptr(self.v), P, N, ptr(inc_ptr), ptr(inc_other),
                                          ptr(inc_pair), ptr(ws), ws_bytes, stream_of(dev)),
                      "dl_pair_incidence")
                g = Graph(inc_ptr, inc_other[:2 * P], N)
            self._inc = (g, inc_pair[:2 * P])
        return self._inc


def pair_score_fwd(Z, H, batch: PairBatch, T: float = 1.0, want_logit=True, want_prob=True, out=None):
    """-> (logit [P] or None, prob [P] or None).  `out` = optional preallocated (logit, prob)."""
    K, d = _check_Z(Z, batch.N)
    Z = Z.contiguous()
    H = H.contiguous()
    dev = Z.device
    with torch.cuda.device(dev):
        if out is not None:
            logit, prob = out
            want_logit, want_prob = logit is not None, prob is not None
        else:
            logit = torch.empty(max(batch.P, 1), dtype=torch.float32, device=dev) if want_logit else None
            prob = torch.empty(max(batch.P, 1), dtype=torch.float32, device=dev) if want_prob else None
        check(lib().dl_pair_score_fwd(ptr(batch.u), ptr(batch.v), batch.P, ptr(Z), ptr(H), batch.N,
                                      K, d, float(T), ptr(logit), ptr(prob), stream_of(dev)),
              "dl_pair_score_fwd")
    return (logit[:batch.P] if want_logit else None), (prob[:batch.P] if want_prob else None)


def pair_score_bwd(Z, H, batch: PairBatch, dS, T: float = 1.0, out=None):
    """-> (dZ, dH) of the decoder given dS = dL/dlogit.  `out` = optional preallocated (dZ, dH)."""
    K, d = _check_Z(Z, batch.N)
    Z = Z.contiguous()
    H = H.contiguous()
    dS = dS.contiguous().to(torch.float32)
    dev = Z.device
    g, inc_pair = batch.incidence()
    with torch.cuda.device(dev):
        dZ, dH = out if out is not None else (torch.empty_like(Z), torch.empty_like(Z))
        check(lib().dl_pair_score_bwd(g.ref, ptr(inc_pair), ptr(Z), ptr(H), ptr(dS), K, d, float(T),
                                      ptr(dZ), ptr(dH), ptr(g.hub_scratch(2 * K * d)),
                                      stream_of(dev)), "dl_pair_score_bwd")
    return dZ, dH


# --------------------------------------------------------------------------------------------
# autograd Functions
# --------------------------------------------------------------------------------------------
def _spmm_side_buffers(graph: Graph, Z, need_grad: bool):
    """-> (sj, zs) for factor_spmm_fwd.  A graph that is not row-partitioned gets the pre-scaled path
    (zs: a transient [N,K,d] scratch; halves the DRAM transactions of the aggregation); a partitioned
    one keeps s[col,kstar] per entry for the backward instead (sj)."""
    if graph.row_base == 0 and graph.nnz > 0:
        return None, torch.empty_like(Z)
    if need_grad:
        return torch.empty(max(graph.nnz, 1), dtype=torch.float32, device=Z.device), None
    return None, None


class _FactorAggregate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, Z, graph, beta, T):
        Zc = Z.contiguous()
        kstar, w, s = edge_attn_fwd(graph, Zc, T)
        sj, zs = _spmm_side_buffers(graph, Zc, Z.requires_grad)
        H = factor_spmm_fwd(graph, Zc, kstar, w, s, beta, sj=sj, zs=zs)
        del zs
        ctx.graph, ctx.beta, ctx.T, ctx.sj = graph, float(beta), float(T), sj
        ctx.save_for_backward(Zc, kstar, w, s)
        ctx.mark_non_differentiable(kstar, w, s)
        return H, kstar, w, s

    @staticmethod
    def backward(ctx, G, _gk, _gw, _gs):
        Z, kstar, w, s = ctx.saved_tensors
        if ctx.graph.directed:
            dZ, _ = factor_bwd_directed(ctx.graph, Z, G.contiguous(), kstar, w, s, ctx.beta, ctx.T)
            return dZ, None, None, None
        # the gather-only backward collects the (j,i) terms from row i's side: it needs a symmetric
        # pattern (always true for adj_sym, main_disentangled.py:141-142).  Checked once per graph.
        # A graph marked directed takes the backward over its transpose instead (above).
        ctx.graph.assert_symmetric()
        dZ, _ = factor_bwd(ctx.graph, Z, G.contiguous(), kstar, w, s, ctx.beta, ctx.T, sj=ctx.sj)
        return dZ, None, None, None


def factor_aggregate(Z, graph: Graph, beta: float, T: float = 1.0, return_attention=False):
    """H[i,k] = beta Z[i,k] + (1-beta) sum_j att_k[i,j] Z[j,k] with the reference's hard-routed,
    source-normalised attention.  Differentiable w.r.t. Z.  [ref: model.py:55-77]"""
    H, kstar, w, s = _FactorAggregate.apply(Z, graph, beta, T)
    return (H, kstar, w, s) if return_attention else H


class _PairScore(torch.autograd.Function):
    @staticmethod
    def forward(ctx, Z, H, batch, T, as_prob):
        Zc, Hc = Z.contiguous(), H.contiguous()
        logit, prob = pair_score_fwd(Zc, Hc, batch, T, want_logit=not as_prob, want_prob=as_prob)
        out = prob if as_prob else logit
        ctx.batch, ctx.T, ctx.as_prob = batch, float(T), bool(as_prob)
        ctx.save_for_backward(Zc, Hc, out)
        return out

    @staticmethod
    def backward(ctx, gout):
        Z, H, out = ctx.saved_tensors
        if ctx.as_prob:
            dS = gout * (1.0 - out) * out   # torch's sigmoid backward: grad * (1 - y) * y
        else:
            dS = gout
        dZ, dH = pair_score_bwd(Z, H, ctx.batch, dS, ctx.T)
        return dZ, dH, None, None, None


def pair_score(Z, H, batch: PairBatch, T: float = 1.0, as_prob: bool = True):
    """sigmoid(sum_k exp(z_u^k.z_v^k/T) (h_u^k.h_v^k)) (or the logit) for every pair of the batch.
    Differentiable w.r.t. Z and H.  [ref: model.py:109-113]"""
    return _PairScore.apply(Z, H, batch, T, as_prob)


def link_bce(prob, labels, weights=None, want_grad: bool = True, dS=None):
    """sum_p weights[p] * BCE(prob[p], labels[p]) and dL/dlogit in one pass (dl_link_bce).
    -> (loss 0-dim f32 tensor, dS [P] or None).  [ref: main_disentangled.py:195]"""
    dev = prob.device
    require_cuda(prob, "prob")
    P = int(prob.numel())
    prob = prob.contiguous()
    labels = labels.to(torch.float32).contiguous()
    if weights is not None:
        weights = weights.to(torch.float32).contiguous()
    L = lib()
    with torch.cuda.device(dev):
        loss = torch.empty((), dtype=torch.float32, device=dev)
        if want_grad and dS is None:
            dS = torch.empty(P, dtype=torch.float32, device=dev)
        ws_bytes = int(L.dl_link_bce_workspace_bytes())
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        check(L.dl_link_bce(ptr(prob), ptr(labels), ptr(weights) if weights is not None else None, P,
                            ptr(dS) if want_grad else None, ptr(loss), ptr(ws), ws_bytes, stream_of(dev)),
              "dl_link_bce")
    return loss, (dS if want_grad else None)


def structured_negative_sampling(edge_index, num_nodes=None, seed: int = 0, graph: Graph = None,
                                 max_tries: int = 64):
    """torch_geometric.utils.structured_negative_sampling on the device: for every edge column
    (i, j) a node k with (i, k) not an edge column.  -> (i, j, k) int64 tensors [E].
    Seedable (counter-based Philox, see dl_structured_negative_sampling); `graph` = optional cached
    directed CSR of edge_index (Graph.from_edges(..., symmetrize=False)).
    [ref: main_disentangled.py:160]"""
    require_cuda(edge_index, "edge_index")
    dev = edge_index.device
    i = edge_index[0].to(torch.int64).contiguous()
    j = edge_index[1].to(torch.int64).contiguous()
    E = int(i.numel())
    if num_nodes is None:
        num_nodes = int(edge_index.max().item()) + 1 if E else 0
    N = int(num_nodes)
    if graph is None:
        graph = Graph.from_edges(i, j, N, symmetrize=False)
    with torch.cuda.device(dev):
        k = torch.empty(E, dtype=torch.int64, device=dev)
        failed = torch.zeros(1, dtype=torch.int32, device=dev)
        if E:
            check(lib().dl_structured_negative_sampling(graph.ref, ptr(i), E, N, int(seed) & (2**64 - 1),
                                                        int(max_tries), ptr(k), ptr(failed), stream_of(dev)),
                  "dl_structured_negative_sampling")
            if int(failed.item()):
                raise RuntimeError(f"{int(failed.item())} edges start at a node adjacent to every node: no negative exists")
    return i, j, k


def roc_auc_stats(score, labels):
    """-> float64 tensor [5] on the device: (auc, n_pos, n_neg, n_nan, 2U) -- see dl_roc_auc.  No host sync."""
    dev = score.device
    require_cuda(score, "score")
    if score.dtype != torch.float32:
        raise TypeError("score must be float32")
    P = int(score.numel())
    score = score.contiguous()
    labels = labels.to(torch.float32).contiguous()
    L = lib()
    with torch.cuda.device(dev):
        out = torch.empty(5, dtype=torch.float64, device=dev)
        ws_bytes = int(L.dl_roc_auc_workspace_bytes(P))
        ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
        check(L.dl_roc_auc(ptr(score), ptr(labels), P, ptr(out), ptr(ws), ws_bytes, stream_of(dev)), "dl_roc_auc")
    return out


def _check_seg_ptr(seg_ptr, device) -> int:
    """-> R.  seg_ptr must be an int64 [R+1] tensor on `device`; its values (0 = seg_ptr[0] <= ... <=
    seg_ptr[R] = P) are not read back here, which would synchronise with the device."""
    require_cuda(seg_ptr, "seg_ptr")
    if seg_ptr.dtype != torch.int64 or seg_ptr.dim() != 1 or seg_ptr.numel() < 2:
        raise ValueError("seg_ptr must be an int64 tensor [R+1] with R >= 1")
    if seg_ptr.device != device:
        raise ValueError(f"seg_ptr is on {seg_ptr.device}, the scores on {device}")
    return int(seg_ptr.numel()) - 1


def _check_per_pair(t, name, device, P: int):
    """A per-pair input of the segmented calls: on `device`, P elements (it is read through a raw pointer)."""
    if t.device != device:
        raise ValueError(f"{name} is on {t.device}, the scores on {device}")
    if t.numel() != P:
        raise ValueError(f"{name} has {t.numel()} elements, the scores {P}")


def roc_auc_segments(score, labels, seg_ptr):
    """roc_auc_stats of every segment [seg_ptr[r], seg_ptr[r+1]) of one score list in one launch sequence:
    -> float64 tensor [R, 5] on the device, row r = (auc, n_pos, n_neg, n_nan, 2U) of segment r alone (see
    dl_roc_auc_segments).  Equal scores in different segments never tie.  No host sync."""
    dev = score.device
    require_cuda(score, "score")
    if score.dtype != torch.float32:
        raise TypeError("score must be float32")
    P = int(score.numel())
    R = _check_seg_ptr(seg_ptr, dev)
    _check_per_pair(labels, "labels", dev, P)
    score = score.contiguous()
    labels = labels.to(torch.float32).contiguous()
    L = lib()
    with torch.cuda.device(dev):
        out = torch.empty(R, 5, dtype=torch.float64, device=dev)
        ws_bytes = int(L.dl_roc_auc_segments_workspace_bytes(P, R))
        ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
        check(L.dl_roc_auc_segments(ptr(score), ptr(labels), P, ptr(seg_ptr.contiguous()), R, ptr(out), ptr(ws),
                                    ws_bytes, stream_of(dev)), "dl_roc_auc_segments")
    return out


def link_bce_segments(prob, labels, weights, seg_ptr):
    """The loss of link_bce on every segment [seg_ptr[r], seg_ptr[r+1]) of one pair list -> float32 [R] on the
    device (an empty segment gives 0).  Loss only: the gradient of the whole list comes from link_bce /
    link_bce_loss.  `weights` may be None (all ones).  No host sync."""
    dev = prob.device
    require_cuda(prob, "prob")
    if prob.dtype != torch.float32:
        raise TypeError("prob must be float32")
    P = int(prob.numel())
    R = _check_seg_ptr(seg_ptr, dev)
    _check_per_pair(labels, "labels", dev, P)
    if weights is not None:
        _check_per_pair(weights, "weights", dev, P)
    prob = prob.contiguous()
    labels = labels.to(torch.float32).contiguous()
    if weights is not None:
        weights = weights.to(torch.float32).contiguous()
    L = lib()
    with torch.cuda.device(dev):
        loss = torch.empty(R, dtype=torch.float32, device=dev)
        ws_bytes = int(L.dl_link_bce_segments_workspace_bytes(R))
        ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
        check(L.dl_link_bce_segments(ptr(prob), ptr(labels), ptr(weights) if weights is not None else None, P,
                                     ptr(seg_ptr.contiguous()), R, ptr(loss), ptr(ws), ws_bytes, stream_of(dev)),
              "dl_link_bce_segments")
    return loss


def roc_auc(score, labels) -> float:
    """sklearn.metrics.roc_auc_score(labels, score) for binary labels, computed on the device
    (main_disentangled.py:204,219).  Raises ValueError where sklearn does (one class only, NaN)."""
    auc, n_pos, n_neg, n_nan, _ = roc_auc_stats(score, labels).tolist()
    if n_nan:
        raise ValueError("Input contains NaN.")
    if n_pos == 0 or n_neg == 0:
        raise ValueError("Only one class present in y_true. ROC AUC score is not defined in that case.")
    return auc


class _LinkBCELoss(torch.autograd.Function):
    """Whole hot path as one differentiable op with explicit buffer reuse (4 [N,K,d] buffers live):
    attention -> aggregation -> pair scores -> weighted BCE -> decoder backward -> factor backward.
    [ref: model.py:105-114 + main_disentangled.py:195 and its autograd]"""

    @staticmethod
    def forward(ctx, Z, graph, batch, labels, weights, beta, T):
        Zc = Z.detach().contiguous()
        need_grad = ctx.needs_input_grad[0]        # False under torch.no_grad(): the eager backward is skipped
        if need_grad and not graph.directed:
            graph.assert_symmetric()          # gather-only backward (see _FactorAggregate.backward)
        kstar, w, s = edge_attn_fwd(graph, Zc, T)
        sj, zs = _spmm_side_buffers(graph, Zc, need_grad)
        H = factor_spmm_fwd(graph, Zc, kstar, w, s, beta, sj=sj, zs=zs)
        del zs
        _, prob = pair_score_fwd(Zc, H, batch, T, want_logit=False)
        # torch's BCE numerics (log clamped at -100, backward clamped at 1e-12) in one fused pass;
        # weights fold the means and the 1/m of main_disentangled.py:195
        loss, dS = link_bce(prob, labels, weights, want_grad=need_grad)
        if need_grad:
            dZ, dH = pair_score_bwd(Zc, H, batch, dS, T)
            if graph.directed:
                factor_bwd_directed(graph, Zc, dH, kstar, w, s, beta, T, dZ=dZ)
            else:
                factor_bwd(graph, Zc, dH, kstar, w, s, beta, T, dZ=dZ, sj=sj)
            ctx.save_for_backward(dZ)
        ctx.mark_non_differentiable(prob, H)
        return loss, prob, H

    @staticmethod
    def backward(ctx, gloss, _gp, _gh):
        (dZ,) = ctx.saved_tensors
        # out of place: a second backward through the same graph (retain_graph, accumulation) must see
        # the unscaled dZ again, and the returned gradient must not alias a saved tensor
        return dZ * gloss, None, None, None, None, None, None


def link_bce_loss(Z, graph: Graph, batch: PairBatch, labels, weights, beta: float, T: float = 1.0):
    """sum_p weights[p] * BCE(score(u_p, v_p), labels[p]) with score as in model.py:113.
    -> (loss, prob [P], H [N,K,d]); differentiable w.r.t. Z only through `loss`."""
    return _LinkBCELoss.apply(Z, graph, batch, labels, weights, beta, T)


def pairs_exactly_once(u, v, n_nodes: int):
    """Row-major sorted pairs that occur exactly once: the `mask == 1` selection of the script's
    summed dense masks (main_disentangled.py:175-178,195).  Integer work on the device."""
    key, cnt = torch.unique(u.to(torch.int64) * n_nodes + v.to(torch.int64), return_counts=True)
    key = key[cnt == 1]
    return key // n_nodes, key % n_nodes


def pairs_at_least_once(u, v, n_nodes: int):
    """Row-major sorted unique pairs: the clamped eval masks (main_disentangled.py:188-190)."""
    key = torch.unique(u.to(torch.int64) * n_nodes + v.to(torch.int64))
    return key // n_nodes, key % n_nodes


class _AllPairsScore(torch.autograd.Function):
    @staticmethod
    def forward(ctx, Z, H, T):
        K, d = _check_Z(Z, Z.shape[0])
        Zc, Hc = Z.contiguous(), H.contiguous()
        N = int(Z.shape[0])
        dev = Z.device
        with torch.cuda.device(dev):
            prob = torch.empty(N, N, dtype=torch.float32, device=dev)
            check(lib().dl_allpairs_score_fwd(ptr(Zc), ptr(Hc), N, K, d, float(T), ptr(prob),
                                              stream_of(dev)), "dl_allpairs_score_fwd")
        ctx.T = float(T)
        ctx.save_for_backward(Zc, Hc, prob)
        return prob

    @staticmethod
    def backward(ctx, gP):
        Z, H, prob = ctx.saved_tensors
        N, K, d = (int(x) for x in Z.shape)
        dev = Z.device
        dS = gP * (1.0 - prob) * prob
        dSsym = (dS + dS.t()).contiguous()
        with torch.cuda.device(dev):
            dZ = torch.empty_like(Z)
            dH = torch.empty_like(Z)
            check(lib().dl_allpairs_score_bwd(ptr(Z), ptr(H), ptr(dSsym), N, K, d, ctx.T, ptr(dZ),
                                              ptr(dH), stream_of(dev)), "dl_allpairs_score_bwd")
        return dZ, dH, None


def allpairs_score(Z, H, T: float = 1.0):
    """Dense [N,N] link_pred of model.py:109-113 (small N: the unmodified script's contract)."""
    return _AllPairsScore.apply(Z, H, T)


def dense_alpha0(Z, T: float = 1.0):
    """alpha0 [K,N,N] = exp(Z_k Z_k^T / T), second return of Disentangle_layer (model.py:57,77)."""
    K, d = _check_Z(Z, Z.shape[0])
    Zc = Z.detach().contiguous()
    N = int(Z.shape[0])
    dev = Z.device
    with torch.cuda.device(dev):
        out = torch.empty(K, N, N, dtype=torch.float32, device=dev)
        check(lib().dl_dense_alpha0(ptr(Zc), N, K, d, float(T), ptr(out), stream_of(dev)),
              "dl_dense_alpha0")
    return out


def dense_att(graph: Graph, kstar, w, s, K: int):
    """att list of Disentangle_layer as one [K,N,N] tensor (model.py:70-74,77)."""
    dev = graph.device
    with torch.cuda.device(dev):
        out = torch.zeros(K, graph.N, graph.N, dtype=torch.float32, device=dev)
        check(lib().dl_dense_att(graph.ref, ptr(kstar), ptr(w), ptr(s), K, ptr(out), stream_of(dev)),
              "dl_dense_att")
    return out
