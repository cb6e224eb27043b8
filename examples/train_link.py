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

--run R (main_disentangled.py:131,224) trains R independent runs with seeds --seed, --seed + 1, ... together:
one union graph, one stacked model, one optimizer step per epoch (disenlink_b200/runs.py), per-run early
stopping, then the per-run test AUCs and their mean +- std.  Run r gives what a single run with
--seed (seed + r) gives, up to the summation order of the batched GEMMs.

--capture E captures the epoch once as a CUDA graph and replays it (disenlink_b200/capture.py): stopping rule and
model selection on the device, one device-to-host copy per chunk of E epochs, Adam with capturable=True (bias
correction on the device).  Works with --run R and --directed; the loop ends at the first chunk boundary after
every run has stopped.
"""
from __future__ import annotations

import argparse
import copy
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from disenlink_b200 import data as dl_data  # noqa: E402
from disenlink_b200 import ops  # noqa: E402
from disenlink_b200.capture import CapturedEpoch  # noqa: E402
from disenlink_b200.graph import Graph  # noqa: E402
from disenlink_b200.model import Disentangle  # noqa: E402
from disenlink_b200.runs import DisentangleRuns, EarlyStopping, RunSet, edge_labels  # noqa: E402


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
    if getattr(args, "capture", None):
        opt = torch.optim.Adam(model.parameters(), lr=args.lr, weight_decay=5e-4, capturable=True)
        ce = CapturedEpoch(model, opt, x, graph, train_batch, labels, weights, val_batch, val_lab, test_batch,
                           test_lab, args.beta, args.temperature, patience=200, chunk=args.capture)
        out = ce.run(args.epochs, log=log, log_every=args.log_every)
        log(f"test auc: {out['test_auc'][0]:.4f}")
        return {"history": out["history"][0], "best_val_auc": out["best_val_auc"][0], "test_auc": out["test_auc"][0]}
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


def batched_model(args, nfeat, seeds):
    """DisentangleRuns whose run r is the model run() builds after torch.manual_seed(seeds[r])."""
    models = []
    for seed in seeds:
        torch.manual_seed(seed)
        models.append(Disentangle(nfeat, args.nhidden, args.nembed, nfactor=args.nfactor, beta=args.beta,
                                  t=args.temperature))
    return DisentangleRuns.from_models(models)


def batched_epoch(args, x, runs, model, opt, stop):
    """One epoch of every run: projection, fused loss forward + backward over the union, one Adam step, the
    per-run losses and validation AUCs, the stopping update.  -> host list [R losses, R AUCs, R best AUCs,
    R stopped flags], the epoch's one device-to-host copy."""
    Z = model.project(x)
    loss, prob, H = ops.link_bce_loss(Z, runs.graph, runs.train, runs.train_labels, runs.train_weights,
                                      args.beta, args.temperature)
    opt.zero_grad()
    loss.backward()
    opt.step()
    run_loss = ops.link_bce_segments(prob, runs.train_labels, runs.train_weights, runs.train_ptr)
    _, val_prob = ops.pair_score_fwd(Z.detach(), H, runs.val, args.temperature, want_logit=False)
    auc = ops.roc_auc_segments(val_prob, runs.val_labels, runs.val_ptr)[:, 0]
    stop.update(auc)
    return torch.cat([run_loss.double(), auc, stop.best_auc, stop.stopped.double()]).cpu().tolist()


def run_batched(args, x, edge_index, device, log=print):
    """run() for seeds args.seed + r, r < args.run, trained together (main_disentangled.py:131-224).
    -> {"runs": [{"seed", "history", "best_val_auc", "test_auc"} per run], "test_auc_mean", "test_auc_std"}"""
    n = x.shape[0]
    x = dl_data.row_standardize(x).to(device) if args.standardize else x.to(device)
    seeds = [args.seed + r for r in range(args.run)]
    runs = RunSet(edge_index.to(device), n, seeds, args.m, directed=getattr(args, "directed", False))
    model = batched_model(args, x.shape[1], seeds).to(device)
    R = len(seeds)
    if getattr(args, "capture", None):
        opt = torch.optim.Adam(model.parameters(), lr=args.lr, weight_decay=5e-4, capturable=True)
        ce = CapturedEpoch(model, opt, x, runs.graph, runs.train, runs.train_labels, runs.train_weights, runs.val,
                           runs.val_labels, runs.test, runs.test_labels, args.beta, args.temperature, patience=200,
                           chunk=args.capture, train_ptr=runs.train_ptr, val_ptr=runs.val_ptr, test_ptr=runs.test_ptr)
        res = ce.run(args.epochs, log=log, log_every=args.log_every)
        history, best_val, test_auc = res["history"], res["best_val_auc"], res["test_auc"]
    else:
        opt = torch.optim.Adam(model.parameters(), lr=args.lr, weight_decay=5e-4)
        stop = EarlyStopping(list(model.parameters()), patience=200)
        history = [[] for _ in range(R)]
        active = [True] * R
        for epoch in range(args.epochs):
            host = batched_epoch(args, x, runs, model, opt, stop)
            for r in range(R):
                if active[r]:
                    history[r].append((host[r], host[R + r]))
            active = [not bool(f) for f in host[3 * R:]]
            if epoch % args.log_every == 0:
                log(f"epoch: {epoch} active runs: {sum(active)}/{R} loss: {np.mean(host[:R]):.5f} (mean) "
                    f"val_auc: " + " ".join(f"{b:.4f}" for b in host[2 * R:3 * R]))
            if not any(active):
                break
        stop.restore()
        with torch.no_grad():
            Z = model.project(x)
            H = ops.factor_aggregate(Z, runs.graph, args.beta, args.temperature)
            _, test_prob = ops.pair_score_fwd(Z, H, runs.test, args.temperature, want_logit=False)
        test_auc = ops.roc_auc_segments(test_prob, runs.test_labels, runs.test_ptr)[:, 0].tolist()
        best_val = stop.best_auc.tolist()
    out = []
    for r, seed in enumerate(seeds):
        log(f"run {r} (seed {seed}): epochs {len(history[r])} best val auc {best_val[r]:.4f} test auc {test_auc[r]:.4f}")
        out.append({"seed": seed, "history": history[r], "best_val_auc": best_val[r], "test_auc": test_auc[r]})
    mean, std = float(np.mean(test_auc)), float(np.std(test_auc))
    log(f"test auc over {R} runs: {mean:.4f} ± {std:.4f}")
    return {"runs": out, "test_auc_mean": mean, "test_auc_std": std}


def parse_args(argv=None):
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
    ap.add_argument("--run", type=int, default=1, help="independent runs (seeds --seed + r), trained together")
    ap.add_argument("--capture", type=int, default=None, metavar="E",
                    help="replay the epoch as a CUDA graph, reading the records back every E epochs")
    args = ap.parse_args(argv)
    if args.run < 1:
        ap.error(f"--run must be >= 1, got {args.run}")
    if args.capture is not None and args.capture < 1:
        ap.error(f"--capture must be >= 1 epochs per chunk, got {args.capture}")
    return args


def main():
    args = parse_args()
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
    if args.run > 1:
        run_batched(args, x, edge_index, device)
    else:
        run(args, x, edge_index, device)


if __name__ == "__main__":
    main()
