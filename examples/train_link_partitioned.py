"""The training loop of main_disentangled.py (reference lines 131-221) on a NODE-PARTITIONED graph: one
process per GPU, every rank keeps the features, embeddings and gradients of the nodes it owns plus a halo
(disenlink_b200.partition.PartitionedLinkStep), the factor MLPs are replicated and their gradients summed
across the ranks.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 4 --master-addr 127.0.0.1 --master-port 29533 \\
        examples/train_link_partitioned.py --dataset synthetic --epochs 50

    ... --directed: train on the directed train adjacency (the script's ``adj``, main_disentangled.py:137-140) with
        disenlink_b200.partition.DirectedPartitionedLinkStep, as examples/train_link.py --directed does on one GPU

Same protocol as the script (85/10/5 split of the edge columns, adjacency = symmetrised train edges, m rounds
of structured negative sampling on the full edge set, loss = BCE(pos) + BCE(neg)/m over pairs occurring exactly
once, model selection on validation AUC, test AUC with the best weights).  The validation and test pairs ride in
the same pair batch with weight 0: they are scored by the same step and contribute nothing to the gradient.

Per epoch and rank:   Z_own = MLPs(x_own)                               (library GEMMs, autograd)
                      step.run(Z_own)  -> loss, all P scores, dL/dZ_own  (the hot path, csrc/ kernels + halo pushes)
                      Z_own.backward(dL/dZ_own); all-reduce(parameter gradients); Adam
Every rank starts from the same weights and applies the same summed gradient, so the replicas stay identical.
"""
from __future__ import annotations

import argparse
import copy
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from disenlink_b200.partition import DirectedPartitionedLinkStep, PartitionedLinkStep  # noqa: E402


class PartitionedLinkTrainer:
    """model: disenlink_b200.model.Disentangle (replicated); x_own: features of the nodes this rank owns
    ([n_own, F], rows step.part.lo .. step.part.hi of the global matrix); step: the rank's PartitionedLinkStep."""

    def __init__(self, model, x_own, step: PartitionedLinkStep, optimizer, group=None):
        self.model, self.x_own, self.step, self.opt, self.group = model, x_own, step, optimizer, group
        self.world = step.part.world
        if self.world > 1:                                   # one set of initial weights: rank 0's
            for p in model.parameters():
                dist.broadcast(p.data, 0, group=group)

    def train_step(self):
        """-> loss (0-dim tensor, identical on every rank)."""
        step = self.step
        Z_own = self.model.project(self.x_own)               # [n_own, K, d]
        step.run(Z_own.detach())
        self.opt.zero_grad(set_to_none=False)
        if Z_own.numel():
            Z_own.backward(step.dZ)                          # dL/dZ of the owned rows -> the replicated MLPs
        if self.world > 1:
            for p in self.model.parameters():
                if p.grad is None:                           # a rank that owns no node still joins the reduction
                    p.grad = torch.zeros_like(p)
                dist.all_reduce(p.grad, op=dist.ReduceOp.SUM, group=self.group)
        self.opt.step()
        return step.loss

    @torch.no_grad()
    def scores(self):
        """All P scores of the last step (every rank holds all of them)."""
        return self.step.prob[:self.step.P]


# ------------------------------------------------------------------------------------------------
# the script's protocol on the device (CUDA only: negative sampling, mask semantics and AUC are kernels)
# ------------------------------------------------------------------------------------------------
def build_pairs(edge_index, n, m, seed, device):
    """-> (train_edges [2,E_tr], u, v, labels, weights, slices) with slices = {"train" | "val" | "test": (lo, hi)}
    into the one pair batch; val / test pairs carry weight 0."""
    from disenlink_b200 import data as dl_data
    from disenlink_b200 import ops
    from disenlink_b200.graph import Graph
    from train_link import edge_labels
    E = edge_index.shape[1]
    tr, te, va = dl_data.split_edges(E, seed, device)
    train_edges = edge_index[:, tr]
    full = Graph.from_edges(edge_index[0], edge_index[1], n, symmetrize=False)
    edge_keys = torch.unique(edge_index[0] * n + edge_index[1])
    neg = {"tr": [], "va": [], "te": []}
    for m_index in range(m):                                               # main_disentangled.py:159-163
        i, _, k = ops.structured_negative_sampling(edge_index, n, seed=seed * 1000 + m_index, graph=full)
        for name, idx in (("tr", tr), ("va", va), ("te", te)):
            neg[name].append(torch.stack([i[idx], k[idx]]))
    neg = {k_: torch.cat(v_, dim=1) for k_, v_ in neg.items()}
    pu, pv = ops.pairs_exactly_once(train_edges[0], train_edges[1], n)     # :175-178,195
    nu, nv = ops.pairs_exactly_once(neg["tr"][0], neg["tr"][1], n)
    us, vs, ws, slices, at = [pu, nu], [pv, nv], [], {}, 0
    ws.append(torch.full((pu.numel(),), 1.0 / max(pu.numel(), 1), device=device))
    ws.append(torch.full((nu.numel(),), 1.0 / (m * max(nu.numel(), 1)), device=device))
    at = pu.numel() + nu.numel()
    slices["train"] = (0, at)
    for name, idx, ng in (("val", va, neg["va"]), ("test", te, neg["te"])):   # clamped eval masks (:188-190)
        u, v = ops.pairs_at_least_once(torch.cat([edge_index[0][idx], ng[0]]), torch.cat([edge_index[1][idx], ng[1]]), n)
        us.append(u), vs.append(v), ws.append(torch.zeros(u.numel(), device=device))
        slices[name] = (at, at + u.numel())
        at += u.numel()
    u, v = torch.cat(us), torch.cat(vs)
    return train_edges, u, v, edge_labels(u, v, edge_keys, n), torch.cat(ws), slices


def main():
    from disenlink_b200 import data as dl_data
    from disenlink_b200 import ops
    from disenlink_b200.model import Disentangle
    from train_link import synthetic
    ap = argparse.ArgumentParser()
    ap.add_argument("--dataset", default="synthetic")
    ap.add_argument("--root", default="data")
    ap.add_argument("--nfactor", type=int, default=3)
    ap.add_argument("--nhidden", type=int, default=512)
    ap.add_argument("--nembed", type=int, default=32)
    ap.add_argument("--beta", type=float, default=0.9)
    ap.add_argument("--temperature", type=int, default=1)
    ap.add_argument("--m", type=int, default=5)
    ap.add_argument("--lr", type=float, default=0.01)
    ap.add_argument("--epochs", type=int, default=100)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--log-every", type=int, default=10)
    ap.add_argument("--locality", action="store_true",
                    help="renumber the nodes with partition.locality_partition first (graphs with locality: smaller halo)")
    ap.add_argument("--directed", action="store_true", help="train on the directed train adjacency, not adj_sym")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    torch.manual_seed(args.seed)                               # every rank builds the same inputs
    if args.dataset in ("cora", "citeseer", "pubmed"):
        x, edge_index, _ = dl_data.read_planetoid(os.path.join(args.root, args.dataset, "raw"), args.dataset)
    elif args.dataset in ("chameleon", "squirrel", "crocodile"):
        x, edge_index, _ = dl_data.read_wikipedia_npz(os.path.join(args.root, args.dataset, "raw", f"{args.dataset}.npz"))
        x = dl_data.row_standardize(x)
    else:
        x, edge_index, _ = synthetic(seed=args.seed)
        x = dl_data.row_standardize(x)
    n = x.shape[0]
    bounds = None
    if args.locality and world > 1:
        # on the FULL edge set (every rank computes the same renumbering); node ids only name rows, so the
        # protocol below is unchanged -- features and edges simply move to the new numbering
        from disenlink_b200.partition import locality_partition
        order, bounds = locality_partition(edge_index[0], edge_index[1], n, world)
        x, edge_index = order.rows_to_new(x), order.relabel(edge_index)
    edge_index = edge_index.to(device)
    train_edges, u, v, labels, weights, slices = build_pairs(edge_index, n, args.m, args.seed, device)
    step_cls = DirectedPartitionedLinkStep if args.directed else PartitionedLinkStep
    step = step_cls(train_edges[0], train_edges[1], n, u, v, labels, weights, args.nfactor, args.nembed,
                    args.beta, float(args.temperature), world=world, rank=rank, bounds=bounds)
    x_own = x[step.part.lo:step.part.hi].to(device)
    model = Disentangle(x.shape[1], args.nhidden, args.nembed, nfactor=args.nfactor, beta=args.beta,
                        t=args.temperature).to(device)
    opt = torch.optim.Adam(model.parameters(), lr=args.lr, weight_decay=5e-4)
    trainer = PartitionedLinkTrainer(model, x_own, step, opt)
    best_auc, best_test, best_state = 0.0, 0.0, None
    for epoch in range(args.epochs):
        loss = trainer.train_step()
        prob = trainer.scores()
        (a, b), (c, e) = slices["val"], slices["test"]
        auc = ops.roc_auc(prob[a:b].contiguous(), labels[a:b].contiguous())       # from the training forward, like :202
        if auc > best_auc:
            best_auc, best_state = auc, copy.deepcopy(model.state_dict())
            best_test = ops.roc_auc(prob[c:e].contiguous(), labels[c:e].contiguous())
        if rank == 0 and epoch % args.log_every == 0:
            print(f"epoch: {epoch} loss: {float(loss):.5f} val_auc: {best_auc:.4f}", flush=True)
    if rank == 0:
        print(f"best val auc: {best_auc:.4f}", flush=True)
        print(f"test auc (at the best validation epoch): {best_test:.4f}", flush=True)
    model.load_state_dict(best_state)
    step.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
