"""CLI driver with the reference's flags (MC-GRA/main.py:78-139) on the native attack.

    python -m mcgra_b200.main --dataset cora --w1=0.01 --w6=10 --w7=10 --w9=10 --w10=1000 --lr=-2 \
           --useH_A --useY_A --useY --measure=MSELoss            (MC-GRA/README.md:29)

Data: `./dataset/<name>.npz` in the reference's npz layout (adj_data/indices/indptr/shape, attr_*, labels), or
`--dataset synthetic:<n>:<f>:<c>`.  `--arch gcn` with `--mode evaluate` (the MC-GRA attack, topology_attack.py) or
`--mode baseline` (the GraphMI attack it is compared against, baseline.py; no adjacency noise) run natively.

Several GPUs: `torchrun --nproc-per-node N -m mcgra_b200.main ...` (WORLD_SIZE > 1) joins a process group and runs the
tile-row sharded attack; every rank forms only the row bands of feature_adj it touches and of the result it owns."""
import argparse
import os
import random
from copy import deepcopy

import numpy as np
import scipy.sparse as sp
import torch

from . import synth
from .baseline import PGDAttack as GraphMI
from .engine import TILE, HostBands, output_band, shard_tile_rows
from .metrics import metric_pool, metric_pool_sharded, precision_recall_at_k
from .models.gcn import GCN, embedding_GCN
from .topology_attack import PGDAttack


DEFENSE_MI_TYPES = ("linear_HSIC", "linear_CKA", "DP")
DEFENSE_BETA_KEYS = ("layer-0", "layer-1", "layer-2", "layer_inter-0", "layer_inter-1")
# test accuracy of the plain GCN per dataset, the defended training's model-selection reference (MC-GPB/main.py:290-299)
PLAIN_ACC = {"cora": 0.757, "citeseer": 0.6303, "polblogs": 0.8386, "usair": 0.4703, "brazil": 0.7308, "AIDS": 0.6682,
             "enzyme": 0.6461, "ogb_arxiv": 0.376}


def parse_beta(text):
    """--beta "b0,b1,b2,i0,i1" -> the beta dict of mcgpb_gcn.GCN.fit (keys DEFENSE_BETA_KEYS)."""
    parts = [] if text is None else text.split(",")
    if len(parts) != len(DEFENSE_BETA_KEYS):
        raise ValueError(f"--beta {text!r}: --defense needs {len(DEFENSE_BETA_KEYS)} comma-separated values for "
                         + ", ".join(DEFENSE_BETA_KEYS))
    try:
        vals = [float(v) for v in parts]
    except ValueError:
        raise ValueError(f"--beta {text!r}: the values must be numbers") from None
    if not all(np.isfinite(vals)):
        raise ValueError(f"--beta {text!r}: the values must be finite")
    return dict(zip(DEFENSE_BETA_KEYS, vals))


def build_parser():
    p = argparse.ArgumentParser()
    p.add_argument('--seed', type=int, default=15)
    p.add_argument('--epochs', type=int, default=100)
    p.add_argument('--lr', type=float, default=0.01)
    p.add_argument('--weight_decay', type=float, default=5e-4)
    p.add_argument('--hidden', type=int, default=16)
    p.add_argument('--dropout', type=float, default=0.5)
    p.add_argument('--nlayers', type=int, default=2)
    p.add_argument('--arch', type=str, choices=["gcn", "gat", "sage"], default='gcn')
    p.add_argument('--dataset', type=str, default='cora')
    p.add_argument('--density', type=float, default=10000000.0)
    p.add_argument('--model', type=str, default='PGD', choices=['PGD', 'min-max'])
    p.add_argument('--nlabel', type=float, default=1.0)
    p.add_argument('--iter', type=int, default=1)
    p.add_argument('--max_eval', type=int, default=100)
    p.add_argument('--log_name', type=str, default="result.txt")
    p.add_argument("--mode", type=str, default="evaluate")
    p.add_argument("--measure", type=str, default="HSIC", choices=["HSIC", "MSELoss", "KL", "KDE", "CKA", "DP"])
    p.add_argument("--measure2", type=str, default="HSIC")
    p.add_argument("--nofeature", action='store_true')
    p.add_argument('--weight_aux', type=float, default=0)
    p.add_argument('--weight_sup', type=float, default=1)
    for k in range(1, 11):
        p.add_argument(f'--w{k}', type=float, default=0)
    p.add_argument('--eps', type=float, default=0)
    p.add_argument('--useH_A', action='store_true')
    p.add_argument('--useY_A', action='store_true')
    p.add_argument('--useY', action='store_true')
    p.add_argument('--ensemble', action='store_true')
    p.add_argument('--add_noise', action='store_true')
    p.add_argument('--defense', action='store_true',
                   help="attack a victim trained with MC-GPB's defence (mcgpb_gcn.GCN.fit with --beta and --MI_type)")
    p.add_argument('--MI_type', type=str, default='linear_HSIC', choices=DEFENSE_MI_TYPES,
                   help="--defense: the information-bottleneck penalty of the defended training")
    p.add_argument('--beta', type=str, default=None,
                   help="--defense: five comma-separated penalty weights for " + ", ".join(DEFENSE_BETA_KEYS))
    p.add_argument('--topk', type=int, default=0,
                   help="K > 0: write the K highest-scoring pairs to results/<log_name>.topk.npz and log precision / "
                        "recall against the true edges")
    p.add_argument("--dist_backend", type=str, default="nccl", choices=["nccl", "gloo"],
                   help="process-group backend under torchrun (WORLD_SIZE > 1): nccl, one GPU per rank (LOCAL_RANK); "
                        "gloo, every rank on cuda:0")
    return p


def load_graph(name, root='./dataset'):
    """(adj csr, features dense float32, labels int64).  npz layout of the reference's datasets (dataset.py:340-361)."""
    if name.startswith("synthetic"):
        _, n, f, c = name.split(":")
        g = synth.make_graph(int(n), int(f), int(c))
        e = g["edges"]
        adj = sp.coo_matrix((np.ones(len(e), np.float32), (e[:, 0], e[:, 1])), shape=(int(n), int(n)))
        adj = (adj + adj.T).tocsr()
        return adj, g["features"], g["labels"]
    with np.load(os.path.join(root, name + '.npz'), allow_pickle=True) as z:
        adj = sp.csr_matrix((z['adj_data'], z['adj_indices'], z['adj_indptr']), shape=z['adj_shape'])
        if 'attr_data' in z:
            feats = sp.csr_matrix((z['attr_data'], z['attr_indices'], z['attr_indptr']), shape=z['attr_shape'])
            feats = np.asarray(feats.todense(), dtype=np.float32)
        else:
            feats = np.eye(adj.shape[0], dtype=np.float32)
        labels = np.asarray(z['labels'] if 'labels' in z else z['node_labels']).astype(np.int64)
    adj = adj + adj.T
    adj = adj.tolil()
    adj.setdiag(0)
    adj = adj.tocsr()
    adj.eliminate_zeros()
    adj.data[:] = 1
    return adj.astype(np.float32), feats, labels


def eye_rows(n, r0, r1, device=None):
    """Rows [r0, r1) of the n x n identity."""
    e = torch.zeros(r1 - r0, n, device=device)
    i = torch.arange(r1 - r0, device=device)
    e[i, r0 + i] = 1.0
    return e


def dot_product_decode(Z, dataset, rows=None):
    """main.dot_product_decode (main.py:44-55) -> feature_adj, or only its rows [r0, r1) (`rows`), formed from Z alone."""
    n = Z.shape[0]
    r0, r1 = rows if rows is not None else (0, n)
    eye = eye_rows(n, r0, r1, Z.device)
    if dataset in ('cora', 'citeseer', 'AIDS') or dataset.startswith("synthetic"):
        return torch.sigmoid(torch.relu(Z[r0:r1] @ Z.t() - eye))
    Zn = torch.nn.functional.normalize(Z, p=2, dim=1)
    return torch.relu(Zn[r0:r1] @ Zn.t() - eye)


def feature_adj_bands(Z, dataset, rank, world, nofeature=False):
    """feature_adj as the row bands one rank of `world` touches -- its tile-row shard (engine.shard_tile_rows) for the
    loop and its band of the result (engine.output_band) for the ensemble -- each formed on Z's device from Z alone
    (identity rows with --nofeature): no rank holds the n x n matrix."""
    n = Z.shape[0]
    tr0, tr1 = shard_tile_rows((n + TILE - 1) // TILE, world)[rank]
    bands = {}
    for r0, r1 in {(tr0 * TILE, min(n, tr1 * TILE)), output_band(n, rank, world)}:
        if r1 > r0:
            bands[(r0, r1)] = eye_rows(n, r0, r1, Z.device) if nofeature else dot_product_decode(Z, dataset, (r0, r1))
    return HostBands(n, bands)


def _share_victim(victim, device):
    """Rank 0's trained victim and random-number state on every rank, so that all ranks attack the same victim and
    continue the same random streams (the draws of --eps) whatever the run-to-run variation of training."""
    import torch.distributed as dist
    with torch.no_grad():
        for t in victim.state_dict().values():
            dist.broadcast(t, 0)
    for get, put in ((torch.get_rng_state, torch.set_rng_state), (torch.cuda.get_rng_state, torch.cuda.set_rng_state)):
        state = get().to(device)
        dist.broadcast(state, 0)
        put(state.cpu())


def _defend(victim, args, dataset, features, adj, labels, idx_train, idx_val, idx_test, device):
    """Train MC-GPB's defended GCN (mcgpb_gcn.GCN.fit with args.beta / args.MI_type) on the sparse adjacency and copy its
    weights (gc1.*, gc2.*, linear1.*) into `victim`.  The model selection compares against the reference's plain
    accuracy of the dataset, or else the test accuracy of the plain `victim` as trained."""
    from . import mcgpb_gcn, utils
    if dataset in PLAIN_ACC:
        plain_acc = PLAIN_ACC[dataset]
    else:
        with torch.no_grad():
            plain_acc = float(utils.accuracy(victim.predict()[idx_test], victim.labels[idx_test]))
    model = mcgpb_gcn.GCN(nfeat=features.shape[1], nhid=16, nclass=int(labels.max()) + 1, nlayer=args.nlayers,
                          dropout=0.5, weight_decay=5e-4, device=device).to(device)
    for layer in model.gc:
        layer.to(device)
    model.fit(features, adj, labels, idx_train, idx_val, idx_test, beta=args.beta, MI_type=args.MI_type,
              plain_acc=plain_acc)
    # the link AUROC of every layer of the weights fit selected, in eval mode (fit's own final_layer_aucs are of a
    # training-mode forward, and None when no epoch passed its selection test)
    model.eval()
    with torch.no_grad():
        layer_aucs = [mcgpb_gcn.link_auc(e, model.origin_csr) for e in model(model.features, model.adj_norm)[1]]
    victim.load_state_dict(model.state_dict())
    with torch.no_grad():
        acc = float(utils.accuracy(victim.predict()[idx_test], victim.labels[idx_test]))
    return {"acc_test": acc, "plain_acc": plain_acc, "final_layer_aucs": layer_aucs}


def main(argv=None):
    args = build_parser().parse_args(argv)
    topk = vars(args).pop("topk")         # not part of the reference's parameter line in the log
    backend = vars(args).pop("dist_backend")
    if topk < 0:
        raise ValueError(f"--topk {topk}: K must be >= 0 (0 = off)")
    if args.arch != "gcn" or args.mode not in ("evaluate", "baseline"):
        raise NotImplementedError("only --arch gcn with --mode evaluate or --mode baseline are on the B200 path "
                                  "(SURVEY.md 2)")
    if args.mode == "baseline" and args.eps != 0:
        raise NotImplementedError("--mode baseline with --eps != 0: the GraphMI baseline attack has no adjacency noise")
    if args.defense:
        args.beta = parse_beta(args.beta)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world == 1:
        return _run(args, topk, torch.device("cuda:0"), 0, 1)
    import torch.distributed as dist
    device = torch.device("cuda", 0 if backend == "gloo" else int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(device)
    dist.init_process_group(backend, **({"device_id": device} if backend == "nccl" else {}))
    try:
        return _run(args, topk, device, dist.get_rank(), dist.get_world_size())
    finally:
        dist.destroy_process_group()


def _run(args, topk, device, rank, world):
    np.random.seed(args.seed); random.seed(args.seed); torch.manual_seed(args.seed); torch.cuda.manual_seed(args.seed)
    adj_sp, feats, labels = load_graph(args.dataset)
    dataset = args.dataset
    if args.dataset.startswith("synthetic"):
        # the reference's dataset-keyed tables (feature similarity main.py:44-55, dot_product_decode2
        # topology_attack.py:421-467) have no synthetic entry: synthetic graphs use the Cora branches
        args.dataset = "cora"
    n = adj_sp.shape[0]
    rng = np.random.RandomState(args.seed)
    perm = rng.permutation(n)
    idx_train, idx_val, idx_test = perm[:max(n // 10, 1)], perm[n // 10:n // 5], perm[n // 5:]
    idx_attack = np.array(random.sample(range(n), int(n * args.nlabel)))
    num_edges = int(0.5 * args.density * adj_sp.sum() / n ** 2 * len(idx_attack) ** 2)
    # the true adjacency stays sparse (COO on the device): no dense n x n on the host (main.py:162 densifies it there)
    coo = adj_sp.tocoo()
    adj = torch.sparse_coo_tensor(torch.from_numpy(np.vstack([coo.row, coo.col]).astype(np.int64)),
                                  torch.from_numpy(coo.data.astype(np.float32)), (n, n)).coalesce().to(device)
    features = torch.from_numpy(feats)
    labels_t = torch.from_numpy(labels)
    if args.mode == "baseline":
        feature_adj = None      # GraphMI never reads it
    elif world > 1 and args.eps == 0:
        feature_adj = feature_adj_bands(features.to(device), args.dataset, rank, world, args.nofeature)
    else:       # (--eps != 0 needs feature_adj as a full tensor, also on several GPUs)
        feature_adj = dot_product_decode(features.to(device), args.dataset)
        if args.nofeature:
            feature_adj = torch.eye(n, device=device)
    victim = GCN(nfeat=features.shape[1], nclass=int(labels.max()) + 1, nhid=16, nlayer=args.nlayers, dropout=0.5,
                 weight_decay=5e-4, device=device).to(device)
    for layer in victim.gc:
        layer.to(device)
    defended = None
    if rank == 0:
        victim.fit(features, adj, labels_t, idx_train, idx_val)
        if args.defense:
            defended = _defend(victim, args, dataset, features, adj, labels_t, idx_train, idx_val, idx_test, device)
    if world > 1:
        _share_victim(victim, device)
    embedding = embedding_GCN(nfeat=features.shape[1], nhid=16, nlayer=args.nlayers, device=device)
    embedding.gc = deepcopy(victim.gc)
    victim.eval(); embedding.eval()
    weight_param = tuple(getattr(args, f"w{k}") for k in range(1, 11))
    if args.mode == "baseline":
        model = GraphMI(model=victim, embedding=embedding, nnodes=n, loss_type='CE', device=device)
        model.attack(None, 10 ** args.lr, 0, args.weight_sup, weight_param, feature_adj, 0, 0, 0, idx_train, idx_val,
                     idx_test, adj, features, torch.zeros(1), labels_t, idx_attack, num_edges, 0, epochs=args.epochs)
    else:
        with torch.no_grad():
            H_A2 = embedding(features.to(device), adj.to(device))
            Y_A = victim(features.to(device), adj.to(device))
        model = PGDAttack(model=victim, embedding=embedding, H_A=H_A2, Y_A=Y_A, nnodes=n, loss_type='CE', device=device)
        model.attack(args, None, 10 ** args.lr, 0, args.weight_sup, weight_param, feature_adj, 0, 0, 0, idx_train,
                     idx_val, idx_test, adj, features, torch.zeros(1), labels_t, idx_attack, num_edges, 0,
                     epochs=args.epochs)
    inference_adj = model.modified_adj
    if world == 1:
        auc = metric_pool(adj, inference_adj, idx_attack, None)
        auc_train = metric_pool(adj, inference_adj, idx_train, None)
        auc_all = metric_pool(adj, inference_adj, np.arange(n), None, True)
        density = float(inference_adj.mean())
    else:       # every rank holds its row band of the result (model.modified_adj_rows)
        import torch.distributed as dist
        row0 = model.modified_adj_rows[0]
        auc, auc_train, auc_all = (metric_pool_sharded(adj, inference_adj, row0, n, ix)
                                   for ix in (idx_attack, idx_train, np.arange(n)))
        total = inference_adj.double().sum().reshape(1)
        dist.all_reduce(total)
        density = float(total.item()) / float(n) ** 2
        if rank == 0:
            print(f"current auc={auc_all}")
    if rank == 0:
        os.makedirs("./results/", exist_ok=True)
        with open(os.path.join("./results", args.log_name), "a") as f:
            f.write(f"current parameter: {args}\n")
            if defended is not None:
                f.write(f"Defended victim: test accuracy={defended['acc_test']}\tplain accuracy={defended['plain_acc']}\n")
                f.write(f"Defended victim: final layer AUROCs={defended['final_layer_aucs']}\n")
            f.write(f"In attack graph: AUC={auc}\tIn train graph: AUC={auc_train}\tIn Whole Graph: AUC={auc_all}\n")
            f.write(f"current density: {density}\n")
    if topk > 0:
        rows, cols, scores = model.recovered_edges(topk)      # (world > 1: the same pairs on every rank)
        if rank != 0:
            return auc_all
        precision, recall = precision_recall_at_k(rows, cols, adj, n)
        np.savez(os.path.join("./results", args.log_name + ".topk.npz"), rows=rows.cpu().numpy(),
                 cols=cols.cpu().numpy(), scores=scores.cpu().numpy())
        with open(os.path.join("./results", args.log_name), "a") as f:
            f.write(f"Top-K: precision={precision} recall={recall} k={topk}\n")
    return auc_all


if __name__ == "__main__":
    main()
