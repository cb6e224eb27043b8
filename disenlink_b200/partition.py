"""Node-partitioned execution of the hot path across the GPUs of one node.

The reference is single-process (SURVEY.md section 2.1).  For graphs that do not fit one device the
nodes are cut into `world` contiguous ranges with about equal numbers of CSR entries (split points
on the degree prefix sum), and every rank keeps RANK-LOCAL storage only:

    per-node arrays   rows [0, n_own)            the nodes the rank owns          (global lo + row)
                      rows [n_own, n_own+n_halo) the remote nodes it reads: the columns of its CSR
                                                 rows and the endpoints of the pairs it scores or
                                                 differentiates, sorted by global id (= grouped by owner)
    CSR               rowptr [n_own+1], columns as LOCAL indices, in global column order
    pairs             an equal contiguous share of every pair batch (local indices), plus the incidence
                      lists of the owned nodes over all pairs

so memory per rank is O(N / world + halo) and the kernels of csrc/ run unchanged on the local graph
(dl_graph.N = n_own, row_base = 0).  Before a kernel reads halo rows their OWNERS push them -- exactly
what is read, straight into the reader's array over NVLink peer memory (dl_push_rows, csrc/peer_copy.cu):

    Z      every halo row (attention reads whole rows of every neighbour)
    s, r   every halo row (K floats per node)
    H      only the endpoints of the reader's pairs
    dH     only the ROUTED factor slices G[j, k*] the reader's backward pass 1 gathers: by the symmetry
           of adjacency and routing the owner of j knows them from its own entries (dl_need_masks)
    prob   the P scores (flat all-gather, dl_push_slice)

No reduction, no atomics, owner computes; a barrier orders the ranks after each push.  Each row's result
comes from the same kernel code walking the same column-sorted row as on one GPU, so integers and routing
are bit-identical to the single-GPU run and floats differ only where a row crosses a range cut of the streaming
kernels (up to 2048 entries per range; the cuts depend on the local entry count).

Per step:  push Z -> attention -> need-masks, push s -> aggregation -> push H -> pair scores -> gather prob
           -> loss -> decoder backward -> push dH slices -> backward pass 1 -> push r -> backward pass 2

DirectedPartitionedLinkStep trains on the edge columns as given (no symmetrisation): each rank also holds the
in-entries of its nodes, the owners of entries push their per-entry records (kstar, w, dw) to the owners of the
columns (dl_push_entries), and the directed backward runs phase by phase (DESIGN.md section 6a).

The orchestration is backend-agnostic: the product backend (`CudaBackend`) calls the CUDA kernels and the
exchange goes over peer memory; tests inject a CPU backend and the exchange falls back to torch.distributed
point-to-point (gloo, world_size 2), which is also the path when the ranks cannot map each other's memory.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass, field

import torch
import torch.distributed as dist


# --------------------------------------------------------------------------------------------
# partition of the node range
# --------------------------------------------------------------------------------------------
@dataclass
class NodePartition:
    n_global: int
    world: int
    rank: int
    bounds: list = field(default=None)          # world + 1 split points; None = equal ranges

    def __post_init__(self):
        if self.bounds is None:
            per = (self.n_global + self.world - 1) // self.world
            self.bounds = [min(r * per, self.n_global) for r in range(self.world)] + [self.n_global]
        assert len(self.bounds) == self.world + 1 and self.bounds[0] == 0 and self.bounds[-1] == self.n_global

    @classmethod
    def nnz_balanced(cls, src: torch.Tensor, dst: torch.Tensor, n_global: int, world: int, rank: int):
        """Split points on the prefix sum of the (directed-column) degrees, so every rank gets about the
        same number of CSR entries.  Every rank computes the same bounds from the same edge list."""
        if world == 1:
            return cls(int(n_global), 1, 0)
        deg = torch.bincount(src, minlength=n_global) + torch.bincount(dst, minlength=n_global)
        cum = torch.cumsum(deg, 0)
        total = int(cum[-1].item())
        targets = torch.tensor([total * r // world for r in range(1, world)], device=cum.device, dtype=cum.dtype)
        cuts = torch.searchsorted(cum, targets, right=False).tolist()
        bounds = [0] + [int(min(max(c + 1, 0), n_global)) for c in cuts] + [int(n_global)]
        for i in range(1, len(bounds)):
            bounds[i] = max(bounds[i], bounds[i - 1])
        return cls(int(n_global), int(world), int(rank), bounds)

    @property
    def lo(self) -> int:
        return self.bounds[self.rank]

    @property
    def hi(self) -> int:
        return self.bounds[self.rank + 1]

    @property
    def n_local(self) -> int:
        return self.hi - self.lo


def owned_entries(src: torch.Tensor, dst: torch.Tensor, part: NodePartition):
    """Directed (local_row, global_col) entries of the symmetrised adjacency whose row this rank
    owns: (s,t) if s is owned, (t,s) if t is owned (duplicates are collapsed by the CSR build).
    [ref: main_disentangled.py:141  adj_sym = adj + adj.t()]"""
    ms = (src >= part.lo) & (src < part.hi)
    mt = (dst >= part.lo) & (dst < part.hi)
    rows = torch.cat([src[ms], dst[mt]]) - part.lo
    cols = torch.cat([dst[ms], src[mt]])
    return rows, cols


def owned_out_entries(src: torch.Tensor, dst: torch.Tensor, part: NodePartition):
    """Directed (local_row, global_col) entries whose row this rank owns: the edge columns as given."""
    m = (src >= part.lo) & (src < part.hi)
    return src[m] - part.lo, dst[m]


def pair_shard(P: int, world: int, rank: int):
    """Contiguous equal share of a pair batch (padded length per rank, [p_lo, p_hi))."""
    per = (P + world - 1) // world
    lo = min(rank * per, P)
    return per, lo, min(lo + per, P)


# --------------------------------------------------------------------------------------------
# optional locality reorder (SURVEY 8(e)): fewer remote columns per rank = a smaller halo to push
# --------------------------------------------------------------------------------------------
class NodeOrder:
    """A renumbering of the nodes.  new_of_old[i] = new id of node i.  Per-node arrays of the caller
    (features, embeddings, gradients) are taken to the new order with rows_to_new and back with rows_to_old."""

    def __init__(self, new_of_old: torch.Tensor):
        self.new_of_old = new_of_old.to(torch.int64)
        self.old_of_new = torch.empty_like(self.new_of_old)
        self.old_of_new[self.new_of_old] = torch.arange(self.new_of_old.numel(), dtype=torch.int64,
                                                        device=self.new_of_old.device)

    def relabel(self, ids: torch.Tensor) -> torch.Tensor:
        return self.new_of_old.to(ids.device)[ids.to(torch.int64)]

    def rows_to_new(self, x_old: torch.Tensor) -> torch.Tensor:
        return x_old[self.old_of_new.to(x_old.device)]

    def rows_to_old(self, y_new: torch.Tensor) -> torch.Tensor:
        return y_new[self.new_of_old.to(y_new.device)]


def locality_partition(src: torch.Tensor, dst: torch.Tensor, n_global: int, world: int, sweeps: int = 12,
                       slack: float = 1.05):
    """-> (NodeOrder, bounds): a renumbering of the nodes and `world + 1` split points such that the contiguous
    ranges hold about equal numbers of CSR entries (within `slack`) AND most neighbours of a node live in its
    own range.  Host-side integer work, once per graph, deterministic (every rank computes the same result from
    the same edge list): reverse Cuthill-McKee order cut into equal-entry blocks, then balanced label
    propagation -- a node moves to the part holding most of its neighbours while that part stays under its
    entry cap -- and finally parts are made contiguous, RCM order inside a part.
    What it buys is graph-dependent: on the real Pubmed citation graph the halo rows of an 8-way partition drop
    from 44 288 to 18 793 and the share of remote CSR entries from 0.88 to 0.37 (tests/test_partition_gloo.py);
    a random power-law graph without locality (bench.py's generator) keeps 0.76 of 0.875.
    Use:  order, bounds = locality_partition(src, dst, N, world)
          step = PartitionedLinkStep(order.relabel(src), order.relabel(dst), N, order.relabel(u), order.relabel(v),
                                     ..., bounds=bounds);   x_own = order.rows_to_new(x)[step.part.lo:step.part.hi]"""
    import numpy as np
    import scipy.sparse as sp
    from scipy.sparse.csgraph import reverse_cuthill_mckee
    n, world = int(n_global), int(world)
    s_, d_ = src.detach().cpu().numpy().astype(np.int64), dst.detach().cpu().numpy().astype(np.int64)
    ar = np.arange(n)
    if world <= 1 or n == 0 or s_.size == 0:
        return NodeOrder(torch.arange(n, dtype=torch.int64)), NodePartition(n, max(world, 1), 0).bounds
    rows, cols = np.concatenate([s_, d_]), np.concatenate([d_, s_])
    A = sp.csr_matrix((np.ones(rows.size, np.float32), (rows, cols)), shape=(n, n))
    A.data[:] = 1.0                                             # duplicate columns collapse, like the CSR build
    deg = np.diff(A.indptr).astype(np.float64)
    rcm = np.asarray(reverse_cuthill_mckee(A, symmetric_mode=True), dtype=np.int64)
    pos = np.empty(n, np.int64)
    pos[rcm] = ar
    cum = np.cumsum(deg[rcm])
    tot = float(cum[-1])
    cuts = np.array([np.searchsorted(cum, tot * r / world) + 1 for r in range(1, world)], dtype=np.int64)
    part = np.searchsorted(cuts, pos, side="right")
    cap = tot / world * float(slack)
    for _ in range(int(sweeps)):
        onehot = sp.csr_matrix((np.ones(n, np.float32), (ar, part)), shape=(n, world))
        votes = np.asarray((A @ onehot).todense())              # neighbours of every node per part
        best = votes.argmax(1)
        gain = votes[ar, best] - votes[ar, part]
        cand = np.nonzero(gain > 0)[0]
        if cand.size == 0:
            break
        load = np.bincount(part, weights=deg, minlength=world)
        # per destination part: candidates by decreasing gain, accepted while the part stays under its cap
        # (entries that LEAVE a part are only credited in the next sweep, so the cap is never exceeded)
        o = np.lexsort((-gain[cand], best[cand]))
        cand = cand[o]
        b = best[cand]
        csum = np.cumsum(deg[cand])
        start = np.concatenate([[0.0], csum[:-1]])
        first = np.r_[True, b[1:] != b[:-1]]
        within = csum - np.maximum.accumulate(np.where(first, start, 0.0))
        ok = load[b] + within <= cap
        if not ok.any():
            break
        part[cand[ok]] = b[ok]
    old_of_new = np.argsort(part.astype(np.int64) * n + pos, kind="stable")
    new_of_old = np.empty(n, np.int64)
    new_of_old[old_of_new] = ar
    bounds = [0] + np.cumsum(np.bincount(part, minlength=world)).tolist()
    return NodeOrder(torch.from_numpy(new_of_old)), [int(b) for b in bounds]


# --------------------------------------------------------------------------------------------
# halo plan: who reads which remote rows (integer work, once per graph + pair batch)
# --------------------------------------------------------------------------------------------
def _exchange_lists(lists, world, rank, group, device):
    """lists[p] = 1-D int64 tensor for peer p -> received[p] = what peer p addressed to this rank.
    Point-to-point (works over gloo and NCCL)."""
    sizes = torch.tensor([int(t.numel()) for t in lists], dtype=torch.int64, device=device)
    all_sizes = [torch.empty_like(sizes) for _ in range(world)]
    dist.all_gather(all_sizes, sizes, group=group)
    recv = [torch.empty(int(all_sizes[p][rank].item()), dtype=torch.int64, device=device) for p in range(world)]
    ops = []
    for p in range(world):
        if p == rank:
            recv[p] = lists[p].clone()
            continue
        if lists[p].numel():
            ops.append(dist.P2POp(dist.isend, lists[p].contiguous(), p, group=group))
        if recv[p].numel():
            ops.append(dist.P2POp(dist.irecv, recv[p], p, group=group))
    if ops:
        for w in dist.batch_isend_irecv(ops):
            w.wait()
    return recv


class HaloPlan:
    """Local index space of one rank and the send lists of the exchange.

    local(id) = id - lo for owned nodes, n_own + position in the sorted halo list otherwise.
    For every peer q:  send_all[q]   own-local rows q reads (its whole block of my nodes, in q's halo
                                     order; destination = contiguous block starting at dst_base[q]);
                       send_pair[q], dst_pair[q]   the subset q needs for its pairs (H), with q's local index
                       recv_all[q] = (first row, count), recv_pair[q] = local rows: what arrives from q."""

    def __init__(self, part: NodePartition, halo_all: torch.Tensor, halo_pair: torch.Tensor, group=None):
        self.part, self.group = part, group
        world, rank = part.world, part.rank
        dev = halo_all.device
        self.n_own = part.n_local
        self.halo = halo_all                       # sorted unique global ids of the remote nodes read here
        self.n_halo = int(halo_all.numel())
        self.n_tot = self.n_own + self.n_halo
        bounds = torch.tensor(part.bounds, dtype=torch.int64, device=dev)
        # block of owner p inside the halo: [hoff[p], hoff[p+1]) (empty for this rank itself)
        self.hoff = torch.searchsorted(halo_all, bounds).tolist()
        self.send_all = [None] * world
        self.dst_base = [0] * world
        self.send_pair = [None] * world
        self.dst_pair = [None] * world
        self.recv_all = {q: (self.n_own + self.hoff[q], self.hoff[q + 1] - self.hoff[q]) for q in range(world)}
        self.recv_pair = {}
        if world == 1:
            return
        need = [halo_all[self.hoff[p]:self.hoff[p + 1]] for p in range(world)]
        got = _exchange_lists(need, world, rank, group, dev)
        # where my rows land at peer q: q's n_own + q's hoff[rank]
        mine = torch.tensor([self.n_own] + self.hoff, dtype=torch.int64, device=dev)
        allm = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allm, mine, group=group)
        for q in range(world):
            if q == rank:
                continue
            self.send_all[q] = (got[q] - part.lo).to(torch.int32)
            self.dst_base[q] = int(allm[q][0].item()) + int(allm[q][1 + rank].item())
        # pair subset: (global id, local index at the reader) pairs
        pos = torch.searchsorted(halo_all, halo_pair) + self.n_own
        hp_off = torch.searchsorted(halo_pair, bounds).tolist()
        need_id = [halo_pair[hp_off[p]:hp_off[p + 1]] for p in range(world)]
        need_loc = [pos[hp_off[p]:hp_off[p + 1]] for p in range(world)]
        self.recv_pair = {q: need_loc[q] for q in range(world)}
        got_id = _exchange_lists(need_id, world, rank, group, dev)
        got_loc = _exchange_lists(need_loc, world, rank, group, dev)
        for q in range(world):
            if q == rank:
                continue
            self.send_pair[q] = (got_id[q] - part.lo).to(torch.int32)
            self.dst_pair[q] = got_loc[q].to(torch.int32)

    def to_local(self, ids: torch.Tensor) -> torch.Tensor:
        """global node ids (owned or in the halo) -> local indices (int64)."""
        lo, hi = self.part.lo, self.part.hi
        if self.n_halo == 0:
            return ids - lo
        own = (ids >= lo) & (ids < hi)
        pos = torch.searchsorted(self.halo, ids).clamp_(max=self.n_halo - 1)
        return torch.where(own, ids - lo, pos + self.n_own)


# --------------------------------------------------------------------------------------------
# exchange: pushes over NVLink peer memory, or torch.distributed point-to-point
# --------------------------------------------------------------------------------------------
class PeerExchange:
    """Owner-pushes-what-the-reader-reads over CUDA IPC peer mappings (dl_push_rows / dl_push_slice).

    Every exchanged array is registered once: its CUDA IPC handle goes round the process group and each
    rank maps the peers' copies.  The ranks must be processes on one node with P2P access between all
    GPUs; otherwise (or on CPU tensors) `available` is False and the exchange goes through
    torch.distributed send / recv.

    Ordering contract: a push writes into buffers the peers read.  Every push is FOLLOWED by a barrier
    (the peers may read once it returns) and the caller puts a barrier BEFORE the first push of a step
    into a buffer whose last reader is not separated from it by another barrier (Z: see
    PartitionedLinkStep.forward)."""

    def __init__(self, world: int, rank: int, device, group=None, enable: bool = True):
        self.world, self.rank, self.group, self.device = world, rank, group, device
        self.peers = {}          # id(array) -> {peer rank: address of its copy in this process}
        self._keep = {}          # id(array) -> the array (a registration must not outlive its tensor)
        self._opened = {}        # IPC handle bytes -> base address of the peer's block in this process
        self.is_cuda = torch.device(device).type == "cuda"
        self.available = bool(enable) and world > 1 and self.is_cuda
        if world > 1 and self.is_cuda:
            self._flag = torch.zeros(1, dtype=torch.float32, device=device)

    def register(self, t: torch.Tensor) -> bool:
        """Collective: every rank registers its copy of the same logical array.  -> False when the mapping
        is not possible (the exchange then stays on torch.distributed for every array)."""
        if not self.available:
            return False
        from ._lib import lib
        mine = None
        try:
            h = t.untyped_storage()._share_cuda_()
            hb = bytes(h[1])
            # torch: [version byte][type byte: b'c' = a cudaMalloc block][64-byte cudaIpcMemHandle_t]
            if len(hb) == 66 and hb[1:2] == b"c":
                hb = hb[2:]
            if len(hb) == 64:
                mine = (hb, int(h[3]) + t.storage_offset() * t.element_size())
        except Exception:                                   # pragma: no cover - allocator without IPC
            mine = None
        objs = [None] * self.world
        dist.all_gather_object(objs, mine, group=self.group)
        bases, ok = {}, all(o is not None for o in objs)
        if ok:
            with torch.cuda.device(self.device):
                for r, (hb, off) in enumerate(objs):
                    if r == self.rank:
                        continue
                    base = self._opened.get(hb)             # one cudaMalloc block may hold several arrays
                    if base is None:
                        out = ctypes.c_void_p()
                        # opened with THIS device current: a peer mapping kernels of this device can use
                        if lib().dl_ipc_open(hb, ctypes.byref(out)) != 0 or not out.value:
                            ok = False
                            break
                        base = self._opened[hb] = out.value
                    bases[r] = base + off
        flag = torch.tensor([1.0 if ok else 0.0], device=self.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
        if flag.item() < 1.0:
            self.available = False
            self.peers.clear()
            return False
        self.peers[id(t)] = bases
        self._keep[id(t)] = t
        return True

    def close(self) -> None:
        """Unmap every peer allocation (call on every rank, after a barrier)."""
        if self._opened:
            from ._lib import lib
            with torch.cuda.device(self.device):
                for base in self._opened.values():
                    lib().dl_ipc_close(ctypes.c_void_p(base))
        self._opened.clear()
        self.peers.clear()
        self._keep.clear()
        self.available = False

    def barrier(self) -> None:
        if self.world == 1:
            return
        if self.is_cuda:
            dist.all_reduce(self._flag, group=self.group)   # stream-ordered after this rank's pushes
        else:
            dist.barrier(group=self.group)

    def push_rows(self, arr, send, recv, dst_base=None, dst_idx=None, masks=None, vec_per_factor=0):
        """For every peer q: rows send[q] (own-local) of `arr` -> the peer's copy of `arr`, at rows
        dst_base[q] + t (contiguous) or dst_idx[q][t].  masks[q] = uint32 [n_own] (+ vec_per_factor): only
        the flagged factor slices.  recv = what arrives here (used by the torch.distributed path only):
        {q: (first row, count)} or {q: local rows}.  Followed by a barrier."""
        if self.world == 1:
            return
        bases = self.peers.get(id(arr)) if self.available else None
        row_elems = 1
        for n in arr.shape[1:]:
            row_elems *= int(n)
        row_bytes = row_elems * arr.element_size()          # (a rank that owns no nodes and reads none has zero rows)
        if bases is not None and row_bytes % 16 == 0:
            from ._lib import DlPushDesc, check, lib, stream_of
            peers = [q for q in range(self.world) if q != self.rank]
            descs = (DlPushDesc * len(peers))()
            for i, q in enumerate(peers):
                off = 0 if dst_idx is not None else dst_base[q] * row_bytes
                descs[i].dst = bases[q] + off
                descs[i].src_idx = send[q].data_ptr()
                descs[i].dst_idx = dst_idx[q].data_ptr() if dst_idx is not None else None
                descs[i].mask = masks[q].data_ptr() if masks is not None else None
                descs[i].n = int(send[q].numel())
            with torch.cuda.device(self.device):
                check(lib().dl_push_rows(arr.data_ptr(), row_bytes, int(vec_per_factor) if masks is not None else 0,
                                         descs, len(peers), stream_of(self.device)), "dl_push_rows")
        else:
            # torch.distributed point-to-point: whole rows (the slice masks are a traffic optimisation only)
            ops, bufs = [], {}
            for q in range(self.world):
                if q == self.rank:
                    continue
                if send[q].numel():
                    ops.append(dist.P2POp(dist.isend, arr[send[q].long()].contiguous(), q, group=self.group))
                n_in = int(recv[q].numel()) if torch.is_tensor(recv[q]) else int(recv[q][1])
                if n_in:
                    bufs[q] = torch.empty((n_in,) + tuple(arr.shape[1:]), dtype=arr.dtype, device=arr.device)
                    ops.append(dist.P2POp(dist.irecv, bufs[q], q, group=self.group))
            if ops:
                for w in dist.batch_isend_irecv(ops):
                    w.wait()
            for q, b in bufs.items():
                if torch.is_tensor(recv[q]):
                    arr[recv[q]] = b
                else:
                    arr[recv[q][0]:recv[q][0] + recv[q][1]] = b
        self.barrier()

    def push_entries(self, arr, send, dst_off, recv):
        """Per-entry records: for every peer q, arr[send[q]] -> the peer's copy of `arr` at dst_off[q] + t
        (dl_push_entries, one launch).  recv = {q: (first, count)}: what arrives here (torch.distributed path
        only).  Followed by a barrier."""
        if self.world == 1:
            return
        bases = self.peers.get(id(arr)) if self.available else None
        if bases is not None:
            from ._lib import DlPushDesc, check, lib, stream_of
            peers = [q for q in range(self.world) if q != self.rank]
            descs = (DlPushDesc * len(peers))()
            for i, q in enumerate(peers):
                descs[i].dst = bases[q] + dst_off[q] * arr.element_size()
                descs[i].src_idx = send[q].data_ptr() if send[q].numel() else None
                descs[i].dst_idx = None
                descs[i].mask = None
                descs[i].n = int(send[q].numel())
            with torch.cuda.device(self.device):
                check(lib().dl_push_entries(arr.data_ptr(), arr.element_size(), descs, len(peers),
                                            stream_of(self.device)), "dl_push_entries")
        else:
            ops, bufs = [], {}
            for q in range(self.world):
                if q == self.rank:
                    continue
                if send[q].numel():
                    ops.append(dist.P2POp(dist.isend, arr[send[q].long()].contiguous(), q, group=self.group))
                first, n_in = recv[q]
                if n_in:
                    bufs[q] = torch.empty(n_in, dtype=arr.dtype, device=arr.device)
                    ops.append(dist.P2POp(dist.irecv, bufs[q], q, group=self.group))
            if ops:
                for w in dist.batch_isend_irecv(ops):
                    w.wait()
            for q, b in bufs.items():
                arr[recv[q][0]:recv[q][0] + recv[q][1]] = b
        self.barrier()

    def gather_flat(self, full: torch.Tensor, per: int) -> None:
        """All-gather of a flat array split into `world` slices of `per` elements (the P scores)."""
        if self.world == 1:
            return
        bases = self.peers.get(id(full)) if self.available else None
        n_bytes = per * full.element_size()
        if bases is not None and n_bytes % 16 == 0 and full.data_ptr() % 16 == 0:
            from ._lib import check, lib, stream_of
            off = self.rank * n_bytes
            peers = [q for q in range(self.world) if q != self.rank]
            dst = (ctypes.c_void_p * len(peers))(*[bases[q] + off for q in peers])
            with torch.cuda.device(self.device):
                check(lib().dl_push_slice(full.data_ptr() + off, dst, len(peers), n_bytes, stream_of(self.device)),
                      "dl_push_slice")
            self.barrier()
        else:
            dist.all_gather_into_tensor(full, full[self.rank * per:(self.rank + 1) * per].clone(), group=self.group)


# --------------------------------------------------------------------------------------------
# product backend
# --------------------------------------------------------------------------------------------
class CudaBackend:
    """The product backend: every call goes to libdisenlink_b200.so."""

    def __init__(self):
        from . import ops
        from .graph import Graph
        self.ops, self.Graph = ops, Graph

    def build_csr(self, src, dst, part: NodePartition):
        """-> (rowptr int64 [n_own+1], col int32 [nnz] GLOBAL ids, ascending inside a row)."""
        return self._csr_of(*owned_entries(src, dst, part), part)

    def build_csr_directed(self, src, dst, part: NodePartition):
        """build_csr of the edge columns as given (owned out-entries, de-duplicated)."""
        return self._csr_of(*owned_out_entries(src, dst, part), part)

    def _csr_of(self, rows, cols, part: NodePartition):
        from ._lib import check, lib, ptr, stream_of
        dev = rows.device
        E = int(rows.numel())
        L = lib()
        with torch.cuda.device(dev):
            rowptr = torch.empty(part.n_local + 1, dtype=torch.int64, device=dev)
            col = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
            meta = torch.zeros(2, dtype=torch.int64, device=dev)
            ws_bytes = L.dl_csr_build_workspace_bytes(E, part.n_local)
            ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
            check(L.dl_csr_build_rect(ptr(rows.contiguous()), ptr(cols.contiguous()), E, part.n_local,
                                      part.n_global, 0, ptr(rowptr), ptr(col), ptr(meta),
                                      meta[1:].data_ptr(), ptr(ws), ws_bytes, stream_of(dev)),
                  "dl_csr_build_rect")
            nnz = int(meta[0].item())
            del ws
            col = col[:nnz].clone()
        return rowptr, col

    def make_graph(self, rowptr, col_local, n_own, n_tot):
        return self.Graph(rowptr, col_local, n_own, row_base=0, n_global=n_tot)

    def build_incidence(self, u, v, part: NodePartition):
        """Incidence lists of the owned nodes over ALL pairs -> (inc_ptr, inc_other GLOBAL ids, inc_pair)."""
        from ._lib import check, lib, ptr, stream_of
        P = int(u.numel())
        dev = u.device
        u32, v32 = u.to(torch.int32).contiguous(), v.to(torch.int32).contiguous()
        L = lib()
        with torch.cuda.device(dev):
            inc_ptr = torch.empty(part.n_local + 1, dtype=torch.int64, device=dev)
            inc_other = torch.empty(max(2 * P, 1), dtype=torch.int32, device=dev)
            inc_pair = torch.empty(max(2 * P, 1), dtype=torch.int32, device=dev)
            ws_bytes = L.dl_pair_incidence_workspace_bytes(P, part.n_local + 1)
            ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
            check(L.dl_pair_incidence_range(ptr(u32), ptr(v32), P, part.lo, part.hi, ptr(inc_ptr),
                                            ptr(inc_other), ptr(inc_pair), ptr(ws), ws_bytes,
                                            stream_of(dev)), "dl_pair_incidence_range")
            m = int(inc_ptr[-1].item())
            del ws
        return inc_ptr, inc_other[:m].clone(), inc_pair[:m].clone()

    def make_pairs(self, u_loc, v_loc, n_tot):
        return self.ops.PairBatch(u_loc, v_loc, n_tot)

    def bwd_plan(self, g, K, d):
        return self.ops.bwd_plan(g, K, d)

    def need_masks(self, g, kstar, halo_off, world, masks):
        from ._lib import check, lib, ptr, stream_of
        with torch.cuda.device(masks.device):
            check(lib().dl_need_masks(g.ref, ptr(kstar), ptr(halo_off), world, ptr(masks), stream_of(masks.device)),
                  "dl_need_masks")

    # -- kernels (all write only the owned rows [0, n_own) of the local arrays) --
    def edge_attn_fwd(self, g, Z, T, kstar, w, s, plan=None):
        self.ops.edge_attn_fwd(g, Z, T, out=(kstar, w, s), plan=plan)

    def factor_spmm_fwd(self, g, Z, kstar, w, s, beta, H, sj=None, zs=None):
        self.ops.factor_spmm_fwd(g, Z, kstar, w, s, beta, out=H, sj=sj, zs=zs)

    def pair_score_fwd(self, Z, H, shard, T, prob_slice):
        self.ops.pair_score_fwd(Z, H, shard, T, out=(None, prob_slice))

    def pair_score_bwd(self, inc, inc_pair, Z, H, dS, T, dZ, dH):
        from ._lib import check, lib, ptr, stream_of
        K, d = int(Z.shape[1]), int(Z.shape[2])
        dev = Z.device
        with torch.cuda.device(dev):
            check(lib().dl_pair_score_bwd(inc.ref, ptr(inc_pair), ptr(Z), ptr(H), ptr(dS), K, d, float(T),
                                          ptr(dZ), ptr(dH), ptr(inc.hub_scratch(2 * K * d)),
                                          stream_of(dev)), "dl_pair_score_bwd")

    def link_bce(self, prob, labels, weights, dS):
        """-> loss (0-dim tensor); dS [P] written in place."""
        loss, _ = self.ops.link_bce(prob, labels, weights, want_grad=True, dS=dS)
        return loss

    def factor_bwd_gather(self, g, Z, G, kstar, w, s, beta, dZ, r, plan=None):
        self.ops.factor_bwd_gather(g, Z, G, kstar, w, s, beta, dZ, r, plan=plan)

    def factor_bwd_edges(self, g, Z, G, kstar, w, s, r, beta, T, dZ, sj=None, plan=None):
        if plan is not None and plan["mode"] == "sym" and not plan["x_valid"]:
            plan = None
        self.ops.factor_bwd_edges(g, Z, G, kstar, w, s, r, beta, T, dZ, sj=sj, plan=plan)

    def factor_bwd_directed_phase(self, g, gt, tperm, Z, G, kstar, w, s, beta, T, dZ, r, dw, routed, phase):
        self.ops.factor_bwd_directed_phase(g, gt, tperm, Z, G, kstar, w, s, beta, T, dZ, r, dw, routed, phase)


# --------------------------------------------------------------------------------------------
# the step
# --------------------------------------------------------------------------------------------
class PartitionedLinkStep:
    """One forward+backward pass of the hot path on a node-partitioned graph.

    Buffers are allocated once, rank-local.  The caller writes the factor embeddings of the nodes this
    rank owns into `self.Z_own` (a view of the first n_own rows of the local array) or passes them to
    `run()`; `run()` leaves dL/dZ of the owned rows in `self.dZ` ([n_own, K, d]), H of the owned rows in
    `self.H[:n_own]` and all P scores in `self.prob`.

    (src, dst) are the edge columns of an undirected graph: the step always trains on their symmetrisation
    (adj_sym, see owned_entries).  ``directed=True`` -- training on the columns as given -- is refused here;
    DirectedPartitionedLinkStep does that."""

    DIRECTED = False

    def __init__(self, src, dst, n_global, u, v, labels, weights, K, d, beta, T,
                 world=1, rank=0, group=None, backend=None, device=None, mark=None, balance=True,
                 peer_push=True, bounds=None, directed=False):
        if not self.DIRECTED and (directed or getattr(src, "directed", False)):
            raise ValueError("PartitionedLinkStep trains on the symmetrised edge columns only: use "
                             "DirectedPartitionedLinkStep to train on directed edge columns as given")
        self.mark = mark if mark is not None else (lambda name: None)  # phase boundary hook (bench)
        self.group = group
        self.be = backend if backend is not None else CudaBackend()
        self.K, self.d, self.beta, self.T = int(K), int(d), float(beta), float(T)
        dev = device if device is not None else src.device
        self.device = dev
        world, rank = int(world), int(rank)
        # split points: given (e.g. by locality_partition), on the degree prefix sum, or equal node counts
        if bounds is not None:
            self.part = part = NodePartition(int(n_global), world, rank, [int(b) for b in bounds])
        else:
            self.part = part = (NodePartition.nnz_balanced(src, dst, int(n_global), world, rank) if balance
                                else NodePartition(int(n_global), world, rank))
        be = self.be
        # ---- integer setup: CSR of the owned rows, pair shard, incidence lists, halo, local indices ----
        rowptr, col_g = self._build_csr(src, dst, part)
        self.P = int(u.numel())
        self.p_per, self.p_lo, self.p_hi = pair_shard(self.P, world, rank)
        su, sv = u[self.p_lo:self.p_hi].to(torch.int64), v[self.p_lo:self.p_hi].to(torch.int64)
        inc_ptr, inc_other_g, self.inc_pair = be.build_incidence(u, v, part)
        lo, hi = part.lo, part.hi

        def remote(t):
            t = t.to(torch.int64)
            return t[(t < lo) | (t >= hi)]
        if world > 1:
            halo_pair = torch.unique(torch.cat([remote(su), remote(sv), remote(inc_other_g)]))
            halo_all = torch.unique(torch.cat([remote(self._read_columns(src, dst, col_g)), halo_pair]))
        else:
            halo_pair = halo_all = torch.empty(0, dtype=torch.int64, device=dev)
        self.plan = plan = HaloPlan(part, halo_all, halo_pair, group)
        n_own, n_tot = plan.n_own, plan.n_tot
        self.n_own, self.n_tot = n_own, n_tot
        col_l = plan.to_local(col_g.to(torch.int64)).to(torch.int32) if world > 1 else col_g
        self.graph = be.make_graph(rowptr, col_l, n_own, n_tot)
        self.shard = be.make_pairs(plan.to_local(su), plan.to_local(sv), n_tot)
        inc_other_l = plan.to_local(inc_other_g.to(torch.int64)).to(torch.int32) if world > 1 else inc_other_g
        self.inc = be.make_graph(inc_ptr, inc_other_l, n_own, n_tot)
        n_rec = self._build_records(src, dst, rowptr, col_g)     # per-entry arrays: own entries (+ peers' records)
        del col_g, inc_other_g, su, sv
        # ---- buffers ----
        P_pad = self.p_per * world
        f32 = dict(dtype=torch.float32, device=dev)
        self.labels = torch.zeros(P_pad, **f32)
        self.labels[:self.P] = labels
        self.weights = torch.zeros(P_pad, **f32)
        self.weights[:self.P] = weights
        nnz = self.graph.nnz
        self.kstar = torch.empty(max(n_rec, 1), dtype=torch.uint8, device=dev)
        self.w = torch.empty(max(n_rec, 1), **f32)
        # the aggregation gathers slices pre-divided by s (scratch = the dH buffer, idle during the forward;
        # own and halo rows alike: s of the halo has been pushed by then); with DL_F_NO_PRESCALE it gathers
        # s[col, kstar] per entry and hands the per-entry copy to pass 2
        # -- as long as rescaling every local row (own + halo: 8 D bytes each) costs less than the per-entry gathers
        # it saves (a rank of an 8-way partition holds ~N halo rows for nnz / 8 entries: there it does not)
        self.prescale = (hasattr(be, "bwd_plan") and not (getattr(self.graph, "flags", 0) & 8)
                         and n_tot * 8 <= max(nnz, 1))
        self.sj = None if self.prescale else torch.empty(max(nnz, 1), **f32)
        # how pass 1 hands its per-entry dots to pass 2 (and, on one GPU, the symmetric pass 2 with its
        # coefficient scratch); None: pass 2 gathers everything itself (test backend)
        self.plan_bwd = self._bwd_plan()
        self.Z = torch.zeros(n_tot, K, d, **f32)
        self.Z_own = self.Z[:n_own]
        self.s = torch.ones(n_tot, K, **f32)
        self.r = torch.zeros(n_tot, K, **f32)
        self.H = torch.zeros(n_tot, K, d, **f32)
        self.dH = torch.zeros(n_tot, K, d, **f32)
        self.dZ = torch.zeros(n_own, K, d, **f32)
        self.prob = torch.zeros(P_pad, **f32)
        self.dS = torch.zeros(P_pad, **f32)
        self.loss = None
        self.masks = None
        if world > 1:
            self.masks = torch.zeros(world, max(n_own, 1), dtype=torch.int32, device=dev)
            self.halo_off = torch.tensor([n_own + o for o in plan.hoff], dtype=torch.int32, device=dev)
        # ---- exchange ----
        self.px = PeerExchange(world, rank, dev, group, enable=peer_push and isinstance(be, CudaBackend))
        self.pushed = False
        if self.px.available:
            self.pushed = all([self.px.register(t) for t in self._exchanged()])

    # -- what the directed step overrides (DirectedPartitionedLinkStep) --
    def _build_csr(self, src, dst, part):
        """-> (rowptr, global columns) of the owned rows: the symmetrised edge columns."""
        return self.be.build_csr(src, dst, part)

    def _read_columns(self, src, dst, col_g):
        """Global ids whose Z / s rows the kernels read, besides the pair endpoints."""
        return col_g

    def _build_records(self, src, dst, rowptr, col_g) -> int:
        """-> length of the per-entry arrays (kstar, w)."""
        return self.graph.nnz

    def _bwd_plan(self):
        return self.be.bwd_plan(self.graph, self.K, self.d) if hasattr(self.be, "bwd_plan") else None

    def _exchanged(self):
        """The arrays peers write into (registered for peer pushes)."""
        return (self.Z, self.s, self.r, self.H, self.dH, self.prob)

    def close(self):
        """Collective: unmap the peers' buffers (a step object that is rebuilt must not leak mappings)."""
        self.px.barrier()
        if self.px.is_cuda:
            torch.cuda.synchronize(self.device)
        self.px.close()

    def exchange_volume(self):
        """Rows this rank sends per step, by kind (for the bench's exchange accounting)."""
        plan = self.plan
        n_all = sum(int(t.numel()) for t in plan.send_all if t is not None)
        n_pair = sum(int(t.numel()) for t in plan.send_pair if t is not None)
        return {"n_own": self.n_own, "n_halo": plan.n_halo, "rows_out_all": n_all, "rows_out_pair": n_pair}

    def forward(self):
        part, be, g, mark, px, plan = self.part, self.be, self.graph, self.mark, self.px, self.plan
        Z = self.Z
        mark("begin")
        # Write-after-read guard: a peer may still be reading last step's halo rows of Z (backward pass 2
        # is the last reader and no barrier follows it), so nobody overwrites them before everyone is here.
        px.barrier()
        mark("wait")                 # what the slowest rank of the previous step costs everybody (load imbalance)
        px.push_rows(Z, plan.send_all, plan.recv_all, dst_base=plan.dst_base)
        mark("ag_Z")
        if self.plan_bwd is not None:
            # the symmetric attention leaves its softmax in the plan's coefficient buffer for backward pass 2
            be.edge_attn_fwd(g, Z, self.T, self.kstar, self.w, self.s, plan=self.plan_bwd)
        else:
            be.edge_attn_fwd(g, Z, self.T, self.kstar, self.w, self.s)
        mark("attn_fwd")
        if part.world > 1:
            if hasattr(be, "need_masks"):
                be.need_masks(g, self.kstar, self.halo_off, part.world, self.masks)
            px.push_rows(self.s, plan.send_all, plan.recv_all, dst_base=plan.dst_base)
        mark("ag_s")
        be.factor_spmm_fwd(g, Z, self.kstar, self.w, self.s, self.beta, self.H, self.sj,
                           self.dH if self.prescale else None)
        mark("spmm_fwd")
        px.push_rows(self.H, plan.send_pair, plan.recv_pair, dst_idx=plan.dst_pair)
        mark("ag_H")
        lo = part.rank * self.p_per
        if self.p_hi > self.p_lo:
            be.pair_score_fwd(Z, self.H, self.shard, self.T, self.prob[lo:lo + (self.p_hi - self.p_lo)])
        mark("pair_fwd")
        px.gather_flat(self.prob, self.p_per)
        mark("ag_prob")
        return self.H, self.prob

    def loss_and_grad_logit(self):
        """weighted BCE over all pairs and dL/dlogit (every rank evaluates the full P-vector; it
        is P floats), with F.binary_cross_entropy's clamps (see dl_link_bce)."""
        self.loss = self.be.link_bce(self.prob, self.labels, self.weights, self.dS)
        self.mark("loss")
        return self.loss

    def backward(self):
        part, be, g, mark, px, plan = self.part, self.be, self.graph, self.mark, self.px, self.plan
        Z = self.Z
        be.pair_score_bwd(self.inc, self.inc_pair, Z, self.H, self.dS, self.T, self.dZ, self.dH)
        mark("pair_bwd")
        if part.world > 1:
            # only the routed slices G[j, k*] the reader's pass 1 gathers
            d4 = self.d // 4 if (self.d % 4 == 0 and (self.d // 4) & (self.d // 4 - 1) == 0) else 0
            masks = [self.masks[q] for q in range(part.world)] if (d4 and hasattr(be, "need_masks")) else None
            px.push_rows(self.dH, plan.send_all, plan.recv_all, dst_base=plan.dst_base, masks=masks, vec_per_factor=d4)
        mark("ag_dH")
        be.factor_bwd_gather(g, Z, self.dH, self.kstar, self.w, self.s, self.beta, self.dZ, self.r, plan=self.plan_bwd)
        mark("bwd_gather")
        px.push_rows(self.r, plan.send_all, plan.recv_all, dst_base=plan.dst_base)
        mark("ag_r")
        be.factor_bwd_edges(g, Z, self.dH, self.kstar, self.w, self.s, self.r, self.beta, self.T, self.dZ, self.sj,
                            plan=self.plan_bwd)
        mark("bwd_edges")
        return self.dZ

    def run(self, Z_own=None):
        """Z_own (optional): [n_own, K, d] embeddings of the owned nodes, copied into the local array; by
        default the caller has written `self.Z_own` itself."""
        if Z_own is not None and Z_own.data_ptr() != self.Z_own.data_ptr():
            self.Z_own.copy_(Z_own)
        self.forward()
        self.loss_and_grad_logit()
        return self.backward()


# --------------------------------------------------------------------------------------------
# the step on directed edge columns
# --------------------------------------------------------------------------------------------
def directed_in_view(src, dst, part: NodePartition, rowptr, col_g):
    """The in-entries of the owned nodes, from the global edge columns every rank holds.

    rowptr / col_g: this rank's directed CSR (owned rows, GLOBAL columns, ascending in a row).  ->
      trowptr int64 [n_own+1]   row j - lo lists the in-entries (i, j) of owned node j, by ascending source i
                                (the order of Graph.transpose_view on one GPU)
      tsrc    int64 [m]         global source i of every in-entry
      tperm   int64 [m]         index into the per-entry record space [own CSR entries | tail]: the CSR index of
                                (i - lo, j) for an owned source, nnz_own + position in the tail otherwise
      tail_off list [world+1]   the tail = every remote in-entry sorted by (i, j); sender q's block is
                                [tail_off[q], tail_off[q+1]), in q's own CSR order"""
    n, lo, hi = part.n_global, part.lo, part.hi
    dev = col_g.device
    s64, d64 = src.to(torch.int64), dst.to(torch.int64)
    m = (d64 >= lo) & (d64 < hi)
    key = torch.unique((d64[m] - lo) * n + s64[m])                      # sorted: by owned node, then source
    tj, tsrc = key // n, key % n
    trowptr = torch.zeros(part.n_local + 1, dtype=torch.int64, device=dev)
    trowptr[1:] = torch.cumsum(torch.bincount(tj, minlength=part.n_local), 0)
    entry_key = tsrc * n + tj + lo                                      # (i, j) in global ids
    own = (tsrc >= lo) & (tsrc < hi)
    nnz_own = int(col_g.numel())
    rows = torch.repeat_interleave(torch.arange(part.n_local, device=dev), rowptr[1:] - rowptr[:-1])
    out_key = (rows + lo) * n + col_g.to(torch.int64)                   # the CSR entries, ascending
    tail_key = torch.sort(entry_key[~own]).values
    tperm = torch.empty_like(tsrc)
    tperm[own] = torch.searchsorted(out_key, entry_key[own])
    tperm[~own] = nnz_own + torch.searchsorted(tail_key, entry_key[~own])
    bounds = torch.tensor(part.bounds, dtype=torch.int64, device=dev)
    tail_off = torch.searchsorted(tail_key // max(n, 1), bounds).tolist()
    return trowptr, tsrc, tperm, tail_off


def entry_send_lists(col_g, part: NodePartition):
    """-> [world] int64 tensors: the CSR indices of this rank's entries whose column rank q owns, in CSR order (the
    records q's in-view reads from its tail block for this rank; empty for this rank itself)."""
    bounds = torch.tensor(part.bounds, dtype=torch.int64, device=col_g.device)
    owner = torch.searchsorted(bounds[1:], col_g.to(torch.int64), right=True)
    owner[owner == part.rank] = -1
    return [torch.nonzero(owner == q).flatten() for q in range(part.world)]


class DirectedPartitionedLinkStep(PartitionedLinkStep):
    """PartitionedLinkStep on the edge columns AS GIVEN: a de-duplicated directed CSR of the owned rows, the
    directed backward (csrc/bwd_dir.cu) run phase by phase on rank-local graphs.  Same arguments and the same
    run / forward / loss_and_grad_logit / backward / close contract.

    Entry e = (i, j) lives on the owner of i.  Besides the owned rows each rank holds the IN-VIEW of its nodes
    (directed_in_view: row j lists the in-entries (i, j), a Graph of its own so in-hubs get hub items) and
    per-entry records kstar, w, dw of length nnz_own + n_tail: the attention / pass 2 out-side write the own
    prefix, the owners of remote in-entries push the tail (dl_push_entries).  The halo is the out-neighbours, the
    in-neighbours and the pair endpoints: the symmetrised graph's halo.

    Per step:  push Z -> attention -> need-masks, push s, push kstar and w records -> aggregation -> push H
               -> pair scores -> gather prob -> loss -> decoder backward -> push dH slices -> pass 1 (in-view)
               -> pass 2 out-side -> push dw records -> pass 2 in-side
    r is read only for the entry's own row, so it is not exchanged."""

    DIRECTED = True

    def _build_csr(self, src, dst, part):
        return self.be.build_csr_directed(src, dst, part)

    def _read_columns(self, src, dst, col_g):
        # pass 2's in-side reads Z of the sources of the owned nodes' in-entries
        d64 = dst.to(torch.int64)
        m = (d64 >= self.part.lo) & (d64 < self.part.hi)
        return torch.cat([col_g.to(torch.int64), src.to(torch.int64)[m]])

    def _build_records(self, src, dst, rowptr, col_g) -> int:
        part, plan, dev = self.part, self.plan, self.device
        world, rank = part.world, part.rank
        nnz = self.graph.nnz
        trowptr, tsrc, tperm, tail_off = directed_in_view(src, dst, part, rowptr, col_g)
        tcol_l = plan.to_local(tsrc).to(torch.int32) if world > 1 else tsrc.to(torch.int32)
        self.tgraph = self.be.make_graph(trowptr, tcol_l, self.n_own, self.n_tot)
        self.tperm = tperm.to(torch.int32)
        self.n_tail = tail_off[-1] - tail_off[0]
        if hasattr(self.graph, "_sym"):                         # directed patterns: no symmetric view to try
            self.graph._sym = False
            self.tgraph._sym = False
        sends = entry_send_lists(col_g, part)
        self.rec_send = [None] * world
        self.rec_dst = [0] * world
        self.rec_recv = {q: (nnz + tail_off[q], tail_off[q + 1] - tail_off[q]) for q in range(world)}
        if world > 1:
            mine = torch.tensor([nnz] + tail_off, dtype=torch.int64, device=dev)
            allm = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(allm, mine, group=self.group)
            for q in range(world):
                if q == rank:
                    continue
                send = sends[q]
                want = int(allm[q][2 + rank].item()) - int(allm[q][1 + rank].item())
                if int(send.numel()) != want:
                    raise RuntimeError(f"rank {rank}: {int(send.numel())} entry records for rank {q}, which expects "
                                       f"{want} (the ranks disagree on the edge columns)")
                self.rec_send[q] = send.to(torch.int32)
                self.rec_dst[q] = int(allm[q][0].item()) + int(allm[q][1 + rank].item())
        n_rec = nnz + self.n_tail
        self.dw = torch.empty(max(n_rec, 1), dtype=torch.float32, device=dev)
        self.routed = torch.empty(max(self.n_own, 1), dtype=torch.int32, device=dev)
        return n_rec

    def _bwd_plan(self):
        return None                                             # the directed passes keep no per-entry dots

    def _exchanged(self):
        return (self.Z, self.s, self.H, self.dH, self.prob, self.kstar, self.w, self.dw)

    def exchange_volume(self):
        v = super().exchange_volume()
        n_rec = sum(int(t.numel()) for t in self.rec_send if t is not None)
        v.update(n_tail=self.n_tail, records_out=n_rec, record_bytes_out_fwd=5 * n_rec, record_bytes_out_bwd=4 * n_rec)
        return v

    def forward(self):
        part, be, g, mark, px, plan = self.part, self.be, self.graph, self.mark, self.px, self.plan
        Z = self.Z
        mark("begin")
        # Z halo rows and the record tails: their last readers are the previous step's pass 2 in-side
        px.barrier()
        mark("wait")
        px.push_rows(Z, plan.send_all, plan.recv_all, dst_base=plan.dst_base)
        mark("ag_Z")
        be.edge_attn_fwd(g, Z, self.T, self.kstar, self.w, self.s)
        mark("attn_fwd")
        if part.world > 1:
            if hasattr(be, "need_masks"):
                be.need_masks(g, self.kstar, self.halo_off, part.world, self.masks)
            px.push_rows(self.s, plan.send_all, plan.recv_all, dst_base=plan.dst_base)
        mark("ag_s")
        px.push_entries(self.kstar, self.rec_send, self.rec_dst, self.rec_recv)
        px.push_entries(self.w, self.rec_send, self.rec_dst, self.rec_recv)
        mark("ag_rec")
        be.factor_spmm_fwd(g, Z, self.kstar, self.w, self.s, self.beta, self.H, None,
                           self.dH if self.prescale else None)
        mark("spmm_fwd")
        px.push_rows(self.H, plan.send_pair, plan.recv_pair, dst_idx=plan.dst_pair)
        mark("ag_H")
        lo = part.rank * self.p_per
        if self.p_hi > self.p_lo:
            be.pair_score_fwd(Z, self.H, self.shard, self.T, self.prob[lo:lo + (self.p_hi - self.p_lo)])
        mark("pair_fwd")
        px.gather_flat(self.prob, self.p_per)
        mark("ag_prob")
        return self.H, self.prob

    def backward(self):
        part, be, g, mark, px, plan = self.part, self.be, self.graph, self.mark, self.px, self.plan
        Z = self.Z
        be.pair_score_bwd(self.inc, self.inc_pair, Z, self.H, self.dS, self.T, self.dZ, self.dH)
        mark("pair_bwd")
        if part.world > 1:
            # the routed slices G[i, k*] of the peers' in-entries: dl_need_masks on the owned out-entries
            d4 = self.d // 4 if (self.d % 4 == 0 and (self.d // 4) & (self.d // 4 - 1) == 0) else 0
            masks = [self.masks[q] for q in range(part.world)] if (d4 and hasattr(be, "need_masks")) else None
            px.push_rows(self.dH, plan.send_all, plan.recv_all, dst_base=plan.dst_base, masks=masks, vec_per_factor=d4)
        mark("ag_dH")
        args = (g, self.tgraph, self.tperm, Z, self.dH, self.kstar, self.w, self.s, self.beta, self.T, self.dZ,
                self.r, self.dw, self.routed)
        be.factor_bwd_directed_phase(*args, 1)
        mark("bwd_gather")
        be.factor_bwd_directed_phase(*args, 2)
        mark("bwd_out")
        px.push_entries(self.dw, self.rec_send, self.rec_dst, self.rec_recv)
        mark("ag_dw")
        be.factor_bwd_directed_phase(*args, 3)
        mark("bwd_in")
        return self.dZ
