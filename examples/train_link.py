"""The training loop of main_disentangled.py (reference lines 131-221) on the scalable path: CSR graph
handle instead of dense [N,N] adjacency / masks, pair lists instead of boolean-mask indexing, and
every per-epoch step on the device (negative sampling, fused BCE, AUC).

    python examples/train_link.py --dataset cora --root /path/to/reference/data --nfactor 3 --beta 0.9
    python examples/train_link.py --dataset chameleon --root /path/to/reference/data_pre_false --nfactor 5 --beta 0.7
    python examples/train_link.py --dataset synthetic
    python examples/train_link.py --dataset chameleon --root /path/to/reference/data_pre_false --nfactor 5 --directed

Same protocol as the script: 85/10/5 split of the directed edge columns, adjacency = symmetrised
train edges, m rounds of structured negative sampling on the FULL edge set, loss = BCE(pos) +
BCE(neg)/m over pairs that occur exactly once, early stopping on validation AUC computed from the
training forward, test AUC with the best weights.

--directed trains on the directed train adjacency (the script's ``adj``, main_disentangled.py:137-140) instead
of ``adj_sym``: the train columns are used as given, in a graph marked directed, whose backward runs over the
pattern and its transpose.  Split, negatives and AUC are unchanged.
"""
from __future__ import annotations

import argparse
import copy
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from disenlink_b200 import data as dl_data  # noqa: E402
from disenlink_b200 import ops  # noqa: E402
from disenlink_b200.graph import Graph  # noqa: E402
from disenlink_b200.model import Disentangle  # noqa: E402


def synthetic(n=3000, communities=8, deg=12, feat=64, seed=0):
    """Planted-partition graph whose features carry the community (a stand-in when no dataset is on disk)."""
    g = torch.Generator().manual_seed(seed)
    comm = torch.randint(0, communities, (n,), generator=g)
    src = torch.randint(0, n, (n * deg,), generator=g)
    same = torch.rand(n * deg, generator=g) < 0.85
    order = torch.argsort(comm)
    bounds = torch.searchsorted(comm[order], torch.arange(communities + 1))
    lo, hi = bounds[comm[src]], bounds[comm[src] + 1]
    pick = lo + (torch.rand(n * deg, generator=g) * (hi - lo)).long().clamp_(max=n - 1)
    dst = torch.where(same, order[pick.clamp(max=n - 1)], torch.randint(0, n, (n * deg,), generator=g))
    keep = src != dst
    key = torch.unique(torch.cat([src[keep] * n + dst[keep], dst[keep] * n + src[keep]]))
    x = torch.nn.functional.one_hot(comm, communities).float() @ torch.randn(communities, feat, generator=g)
    x = x + 0.5 * torch.randn(n, feat, generator=g)
    return x, torch.stack([key // n, key % n]), comm


def edge_labels(u, v, edge_keys, n):
    """ori_adj[u, v] of the script: 1 where (u, v) is a column of the full edge set."""
    k = u.long() * n + v.long()
    pos = torch.searchsorted(edge_keys, k).clamp_(max=edge_keys.numel() - 1)
    return (edge_keys[pos] == k).float()


def run(args, x, edge_index, device, log=print):
    n = x.shape[0]
    x = dl_data.row_standardize(x).to(device) if args.standardize else x.to(device)
    edge_index = edge_index.to(device)
    E = edge_index.shape[1]
    tr, te, va = dl_data.split_edges(E, args.seed, device)
    train_edges = edge_index[:, tr]
    if getattr(args, "directed", False):                                   # adj as a CSR (:137-140)
        graph = Graph.from_edges(train_edges[0], train_edges[1], n, directed=True)
    else:
        graph = Graph.from_edges(train_edges[0], train_edges[1], n)        # adj_sym as a CSR
    full = Graph.from_edges(edge_index[0], edge_index[1], n, symmetrize=False)
    edge_keys = torch.unique(edge_index[0] * n + edge_index[1])
    neg = {"tr": [], "va": [], "te": []}
    for m_index in range(args.m):                                          # main_disentangled.py:159-163
        i, _, k = ops.structured_negative_sampling(edge_index, n, seed=args.seed * 1000 + m_index, graph=full)
        for name, idx in (("tr", tr), ("va", va), ("te", te)):
            neg[name].append(torch.stack([i[idx], k[idx]]))
    neg = {k_: torch.cat(v_, dim=1) for k_, v_ in neg.items()}
    # loss masks: pairs that occur exactly once (summed dense masks compared == 1, :175-178,195)
    pu, pv = ops.pairs_exactly_once(train_edges[0], train_edges[1], n)
    nu, nv = ops.pairs_exactly_once(neg["tr"][0], neg["tr"][1], n)
    train_batch = ops.PairBatch(torch.cat([pu, nu]), torch.cat([pv, nv]), n)
    labels = torch.cat([edge_labels(pu, pv, edge_keys, n), edge_labels(nu, nv, edge_keys, n)])
    weights = torch.cat([torch.full((pu.numel(),), 1.0 / max(pu.numel(), 1), device=device),
                         torch.full((nu.numel(),), 1.0 / (args.m * max(nu.numel(), 1)), device=device)])

    def eval_set(pos_idx, negs):                                           # clamped masks (:188-190)
        u, v = ops.pairs_at_least_once(torch.cat([edge_index[0][pos_idx], negs[0]]),
                                       torch.cat([edge_index[1][pos_idx], negs[1]]), n)
        return ops.PairBatch(u, v, n), edge_labels(u, v, edge_keys, n)

    val_batch, val_lab = eval_set(va, neg["va"])
    test_batch, test_lab = eval_set(te, neg["te"])

    model = Disentangle(x.shape[1], args.nhidden, args.nembed, nfactor=args.nfactor, beta=args.beta,
                        t=args.temperature).to(device)
    opt = torch.optim.Adam(model.parameters(), lr=args.lr, weight_decay=5e-4)
    best_auc, stale, best_state, history = 0.0, 0, None, []
    for epoch in range(args.epochs):
        Z = model.project(x)
        loss, _, H = ops.link_bce_loss(Z, graph, train_batch, labels, weights, args.beta, args.temperature)
        opt.zero_grad()
        loss.backward()
        opt.step()
        _, val_prob = ops.pair_score_fwd(Z.detach(), H, val_batch, args.temperature, want_logit=False)
        auc = ops.roc_auc(val_prob, val_lab)
        history.append((loss.item(), auc))
        if auc > best_auc:
            best_auc, stale, best_state = auc, 0, copy.deepcopy(model.state_dict())
        else:
            stale += 1
        if stale > 200:
            break
        if epoch % args.log_every == 0:
            log(f"epoch: {epoch} loss: {loss.item():.5f} val_auc: {best_auc:.4f}")
    model.load_state_dict(best_state)
    with torch.no_grad():
        Z = model.project(x)
        H = ops.factor_aggregate(Z, graph, args.beta, args.temperature)
        _, test_prob = ops.pair_score_fwd(Z, H, test_batch, args.temperature, want_logit=False)
    test_auc = ops.roc_auc(test_prob, test_lab)
    log(f"test auc: {test_auc:.4f}")
    return {"history": history, "best_val_auc": best_auc, "test_auc": test_auc}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dataset", default="synthetic")
    ap.add_argument("--root", default="data")
    ap.add_argument("--sub_dataset", default="Amherst41", help="fb100 school / twitch-e language")
    ap.add_argument("--nfactor", type=int, default=3)
    ap.add_argument("--nhidden", type=int, default=512)
    ap.add_argument("--nembed", type=int, default=32)
    ap.add_argument("--beta", type=float, default=0.9)
    ap.add_argument("--temperature", type=int, default=1)
    ap.add_argument("--m", type=int, default=5)
    ap.add_argument("--lr", type=float, default=0.01)
    ap.add_argument("--epochs", type=int, default=300)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--gpu", type=int, default=0)
    ap.add_argument("--log-every", type=int, default=10)
    ap.add_argument("--directed", action="store_true", help="train on the directed train adjacency, not adj_sym")
    args = ap.parse_args()
    torch.manual_seed(args.seed)
    device = torch.device(f"cuda:{args.gpu}")
    if args.dataset in ("cora", "citeseer", "pubmed"):
        x, edge_index, _ = dl_data.read_planetoid(os.path.join(args.root, args.dataset, "raw"), args.dataset)
        args.standardize = False
    elif args.dataset in ("chameleon", "squirrel", "crocodile"):
        x, edge_index, _ = dl_data.read_wikipedia_npz(os.path.join(args.root, args.dataset, "raw", f"{args.dataset}.npz"))
        args.standardize = True
    elif args.dataset in ("texas", "wisconsin", "cornell"):                       # main_disentangled.py:69-71,89-94
        x, edge_index, _ = dl_data.read_webkb(os.path.join(args.root, args.dataset, "raw"))
        args.standardize = True
    elif args.dataset == "fb100":                                                   # :61-63,104-108
        x, edge_index, _ = dl_data.read_fb100(os.path.join(args.root, "facebook100", args.sub_dataset + ".mat"))
        args.standardize = True
    elif args.dataset == "twitch-e":                                                # :61-63,104-114 (reversed columns appended)
        x, edge_index, _ = dl_data.read_twitch(os.path.join(args.root, "twitch", args.sub_dataset), args.sub_dataset)
        edge_index = torch.cat([edge_index, edge_index.flip(0)], dim=1)
        args.standardize = True
    else:
        x, edge_index, _ = synthetic(seed=args.seed)
        args.standardize = True
    run(args, x, edge_index, device)


if __name__ == "__main__":
    main()
