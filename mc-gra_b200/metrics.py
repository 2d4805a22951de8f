"""AUC / AP / ranking on the GPU (reference: main.metric_pool, MC-GRA/main.py:66-75; AP of
gcn_parameterized.metric, gcn_parameterized.py:55-65) through mcgra_auc_ap / mcgra_argsort_desc, and the top-k recovered
edges of a score matrix (mcgra_topk_stage) with their precision / recall against the true edges."""
import numpy as np
import torch

from . import _native as N
from ._native import call, ptr


def roc_auc_ap(scores, labels, npos_max=None):
    """scores: float32 device tensor (any shape); labels: same numel, non-zero = positive.
    Returns (auc, ap) as Python floats (sklearn roc_curve+auc / average_precision_score semantics)."""
    s = scores.detach().reshape(-1).to(torch.float32).contiguous()
    lab = labels.reshape(-1)
    if lab.dtype != torch.uint8:
        lab = (lab != 0).to(torch.uint8)
    lab = lab.contiguous()
    assert s.is_cuda and lab.is_cuda and s.numel() == lab.numel()
    total = s.numel()
    if npos_max is None:
        npos_max = int(lab.sum().item())
    npos_max = max(int(npos_max), 1)
    ws = torch.empty(N.lib().mcgra_auc_workspace_bytes(total, npos_max), dtype=torch.uint8, device=s.device)
    out = torch.zeros(4, dtype=torch.float64, device=s.device)
    call("mcgra_auc_ap", ptr(s), ptr(lab), total, npos_max, ptr(ws), ptr(out), N.stream_ptr())
    o = out.cpu().numpy()
    if int(o[2]) > npos_max:
        raise N.NativeError(f"positives {int(o[2])} exceed npos_max {npos_max}")
    return float(o[0]), float(o[1])


def auc_ap_from_edges(scores_dense, edges):
    """All n^2 ordered pairs incl. the diagonal (metric_pool semantics); positives = both orientations of `edges`."""
    n = scores_dense.shape[0]
    dev = scores_dense.device
    e = torch.as_tensor(edges, device=dev).long()
    lab = torch.zeros(n, n, dtype=torch.uint8, device=dev)
    lab[e[:, 0], e[:, 1]] = 1
    lab[e[:, 1], e[:, 0]] = 1
    return roc_auc_ap(scores_dense, lab, npos_max=2 * int(e.shape[0]))


def metric_pool(ori_adj, inference_adj, idx, index_delete=None, print_cfg=False):
    """Same signature / value as main.metric_pool: ROC-AUC over adj[idx][:,idx] (index_delete has no effect on
    the AUC in the reference either, main.py:70-72)."""
    dev = inference_adj.device
    idx_t = torch.as_tensor(np.asarray(idx), device=dev).long()
    if torch.is_tensor(ori_adj) and ori_adj.is_sparse:      # label matrix as uint8 on the device, never a dense host n x n
        a = ori_adj.to(dev).coalesce()
        lab = torch.zeros(a.shape, dtype=torch.uint8, device=dev)
        ij = a.indices()
        lab[ij[0], ij[1]] = (a.values() != 0).to(torch.uint8)
        real = lab[idx_t][:, idx_t]
    else:
        real = ori_adj.to(dev)[idx_t][:, idx_t]
    pred = inference_adj[idx_t][:, idx_t]
    auc, _ = roc_auc_ap(pred, real)
    if print_cfg:
        print(f"current auc={auc}")
    return auc


def argsort_desc(scores):
    """Stable descending arg-sort of a float32 device tensor (recovered-edge ranking)."""
    s = scores.detach().reshape(-1).to(torch.float32).contiguous()
    total = s.numel()
    ws = torch.empty(N.lib().mcgra_sort_workspace_bytes(total), dtype=torch.uint8, device=s.device)
    order = torch.empty(total, dtype=torch.int64, device=s.device)
    call("mcgra_argsort_desc", ptr(s), total, ptr(order), ptr(ws), N.stream_ptr())
    return order


def auc_ap_from_edges_sharded(scores_band, row0, n, edges, group=None):
    """metric_pool semantics (all n^2 ordered pairs) when every rank holds a ROW BAND of the scores (rows row0 ...): the
    positives' keys are all-gathered, every rank ranks its own negatives against the global positives (mcgra_auc_stage),
    the integer counts are all-reduced and every rank finishes with the same AUC / AP."""
    dev = scores_band.device
    rows = scores_band.shape[0]
    e = torch.as_tensor(edges, device=dev).long()
    lab = torch.zeros(rows, n, dtype=torch.uint8, device=dev)
    for a, b in ((e[:, 0], e[:, 1]), (e[:, 1], e[:, 0])):
        m = (a >= row0) & (a < row0 + rows)
        lab[a[m] - row0, b[m]] = 1
    return _auc_ap_sharded(scores_band, lab, max(2 * int(e.shape[0]), 1), group)


def metric_pool_sharded(ori_adj, scores_band, row0, n, idx, group=None):
    """metric_pool(ori_adj, gathered scores, idx) when every rank holds a ROW BAND of the n x n scores (rows row0 ...):
    ROC-AUC over adj[idx][:, idx], the same value on every rank.  Each rank scores the rows of idx that fall in its band
    (all columns idx) and reads their labels from ori_adj (sparse COO or dense) by index, never as an n x n matrix.
    Bands may be empty; together they must cover each row once."""
    import torch.distributed as dist
    dev = scores_band.device
    rows, row0 = int(scores_band.shape[0]), int(row0)
    if scores_band.dim() != 2 or scores_band.shape[1] != n or row0 < 0 or row0 + rows > n:
        raise ValueError(f"rows [{row0}, {row0 + rows}) of an n = {n} score matrix expected, got shape "
                         f"{tuple(scores_band.shape)}")
    idx_t = torch.as_tensor(np.asarray(idx), device=dev).long()
    mine = idx_t[(idx_t >= row0) & (idx_t < row0 + rows)]
    pred = scores_band[mine - row0][:, idx_t]
    a = ori_adj.to(dev)
    real = (a.coalesce() if a.is_sparse else a).index_select(0, mine).index_select(1, idx_t)
    lab = ((real.to_dense() if real.is_sparse else real) != 0).to(torch.uint8)
    npos = lab.sum(dtype=torch.int64).reshape(1)
    dist.all_reduce(npos, group=group)
    return _auc_ap_sharded(pred, lab, max(int(npos.item()), 1), group)[0]


def _auc_ap_sharded(scores, lab, npos_max, group):
    """AUC / AP of the union of every rank's (scores, labels): the positives' keys are all-gathered, every rank ranks its
    own negatives against the global positives (mcgra_auc_stage), the integer counts are all-reduced and every rank
    finishes with the same values.  `npos_max`: a bound on the positives of all ranks together, the same on every rank."""
    import torch.distributed as dist
    dev = scores.device
    world = dist.get_world_size(group)
    s = scores.detach().reshape(-1).to(torch.float32).contiguous()
    lab = lab.reshape(-1).contiguous()
    total = s.numel()
    ws = torch.zeros(N.lib().mcgra_auc_workspace_bytes(max(total, 1), npos_max), dtype=torch.uint8, device=dev)
    out = torch.zeros(4, dtype=torch.float64, device=dev)
    st = N.stream_ptr()
    call("mcgra_auc_stage", 0, ptr(s), ptr(lab), total, npos_max, ptr(ws), ptr(out), st)
    counter = ws[:8].view(torch.int64)
    keys = ws[256:256 + 4 * npos_max].view(torch.int32)
    cnt = counter.clone()
    counts = [torch.zeros_like(cnt) for _ in range(world)]
    dist.all_gather(counts, cnt, group=group)
    allk = [torch.empty(npos_max, dtype=torch.int32, device=dev) for _ in range(world)]
    dist.all_gather(allk, keys.clone(), group=group)
    counts = [int(c.item()) for c in counts]
    if sum(counts) > npos_max:
        raise N.NativeError(f"positives {sum(counts)} exceed npos_max {npos_max}")
    keys.fill_(-1)                       # 0xffffffff: unused slots sort to the top
    o = 0
    for c, k in zip(counts, allk):
        keys[o:o + c] = k[:c]
        o += c
    counter.fill_(o)
    call("mcgra_auc_stage", 1, ptr(s), ptr(lab), total, npos_max, ptr(ws), ptr(out), st)
    ho = int(N.lib().mcgra_auc_hist_offset(npos_max))
    hist = ws[ho:ho + 8 * (npos_max + 2)].view(torch.int64)
    sums = ws[8:24].view(torch.int64)
    dist.all_reduce(hist, group=group)
    dist.all_reduce(sums, group=group)
    call("mcgra_auc_stage", 2, ptr(s), ptr(lab), total, npos_max, ptr(ws), ptr(out), st)
    r = out.cpu().numpy()
    return float(r[0]), float(r[1])


# ---- top-k recovered edges -------------------------------------------------------------------------------------------
# Candidates are the pairs (i, j), i < j, scored by S[i, j] (the lower triangle and the diagonal are never read).  Order:
# score descending, then the row-major index i * n + j ascending, i.e. the first k entries of a stable descending
# arg-sort of the upper-triangle values listed row-major.  -0.0 == +0.0; a NaN candidate raises.


def _check_k(n, k):
    P = n * (n - 1) // 2
    k = int(k)
    if k < 0 or k > P:
        raise ValueError(f"k = {k} is outside [0, n (n - 1) / 2 = {P}]")
    return k


def _empty_pairs(dev):
    return (torch.empty(0, dtype=torch.int64, device=dev), torch.empty(0, dtype=torch.int64, device=dev),
            torch.empty(0, dtype=torch.float32, device=dev))


def _topk_threshold(s, row0, rows, n, k, reduce_hist=None):
    """Stages 0-6 of mcgra_topk_stage on the band `s` (rows row0 ...): the histogram levels (summed over ranks by
    `reduce_hist` between them), the selects and the count.  Returns (ws, control words [tau, t, > tau, == tau])."""
    ws = torch.empty(N.lib().mcgra_topk_workspace_bytes(rows, n, k), dtype=torch.uint8, device=s.device)
    hist = ws[N.TOPK_HIST_OFFSET:N.TOPK_HIST_OFFSET + 8 * (N.TOPK_BINS + 1)].view(torch.int64)
    sp_ = ptr(s) if rows > 0 else None
    st = N.stream_ptr()
    for level in range(3):
        call("mcgra_topk_stage", 2 * level, sp_, row0, rows, n, k, ptr(ws), 0, 0, None, None, st)
        if reduce_hist is not None:
            reduce_hist(hist)
        if level == 0:
            nan = int(hist[N.TOPK_BINS].item())
            if nan:
                raise ValueError(f"{nan} NaN score(s) among the candidate pairs (i < j)")
        call("mcgra_topk_stage", 2 * level + 1, sp_, row0, rows, n, k, ptr(ws), 0, 0, None, None, st)
    call("mcgra_topk_stage", 6, sp_, row0, rows, n, k, ptr(ws), 0, 0, None, None, st)
    ctrl = ws[:40].view(torch.int64).tolist()
    if ctrl[4]:
        raise N.NativeError("top-k: the histogram holds fewer than k candidates")
    return ws, ctrl[:4]


def _order_pairs(idx, val, n):
    """Slots in index order -> (rows, cols, scores) by the stable descending sort of the values."""
    order = argsort_desc(val)
    idx = idx[order]
    return idx // n, idx % n, val[order]


def topk_pairs(scores, k):
    """The k highest-scoring node pairs of an n x n float32 device tensor: (rows, cols, scores) as int64, int64 and
    float32 device tensors of length k, rows < cols, in (score desc, row-major index asc) order."""
    if scores.dim() != 2 or scores.shape[0] != scores.shape[1]:
        raise ValueError(f"topk_pairs needs a square score matrix, got shape {tuple(scores.shape)}")
    n = int(scores.shape[0])
    k = _check_k(n, k)
    if k == 0:
        return _empty_pairs(scores.device)
    s = scores.detach().to(torch.float32).contiguous()
    ws, (tau, t, gt, eq) = _topk_threshold(s, 0, n, n, k)
    if gt + t != k or t > eq:
        raise N.NativeError(f"top-k: inconsistent counts (> tau {gt}, ties {t} of {eq}, k {k})")
    idx = torch.empty(k, dtype=torch.int64, device=s.device)
    val = torch.empty(k, dtype=torch.float32, device=s.device)
    call("mcgra_topk_stage", 7, ptr(s), 0, n, n, k, ptr(ws), 0, t, ptr(idx), ptr(val), N.stream_ptr())
    return _order_pairs(idx, val, n)


def topk_pairs_sharded(scores_band, row0, n, k, group=None):
    """topk_pairs when every rank holds a ROW BAND of the scores (rows row0 .. row0 + rows - 1, all n columns): the
    histograms are all-reduced between the levels, the per-band counts all-gathered; rank r writes its candidates above
    the threshold and clamp(t - ties of the bands above it, 0, its ties) of the ties, and the padded results are
    all-gathered, so every rank returns the same k triples.  Bands may be empty; together they must cover each row once."""
    import torch.distributed as dist
    if scores_band.dim() != 2 or scores_band.shape[1] != n:
        raise ValueError(f"row band of an n = {n} score matrix expected, got shape {tuple(scores_band.shape)}")
    rows, row0, n = int(scores_band.shape[0]), int(row0), int(n)
    if row0 < 0 or row0 + rows > n:
        raise ValueError(f"rows [{row0}, {row0 + rows}) outside [0, {n})")
    k = _check_k(n, k)
    dev = scores_band.device
    if k == 0:
        return _empty_pairs(dev)
    s = scores_band.detach().to(torch.float32).contiguous()
    ws, (tau, t, gt, eq) = _topk_threshold(s, row0, rows, n, k, lambda h: dist.all_reduce(h, group=group))
    world, me = dist.get_world_size(group), dist.get_rank(group)
    mine = torch.tensor([row0, gt, eq], dtype=torch.int64, device=dev)
    counts = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(counts, mine, group=group)
    counts = [c.tolist() for c in counts]
    segs, off, ties_before = [], 0, 0           # bands in row order = global index order
    for q in sorted(range(world), key=lambda q: (counts[q][0], q)):
        _, gt_q, eq_q = counts[q]
        quota = min(max(t - ties_before, 0), eq_q)
        segs.append((q, off, gt_q + quota))
        if q == me:
            my_off, my_quota = off, quota
        off += gt_q + quota
        ties_before += eq_q
    if off != k:
        raise N.NativeError(f"top-k: the bands hold {off} of the k = {k} pairs (overlapping or missing rows?)")
    idx = torch.zeros(k, dtype=torch.int64, device=dev)
    val = torch.zeros(k, dtype=torch.float32, device=dev)
    call("mcgra_topk_stage", 7, ptr(s) if rows > 0 else None, row0, rows, n, k, ptr(ws), my_off, my_quota, ptr(idx),
         ptr(val), N.stream_ptr())
    all_idx = [torch.empty_like(idx) for _ in range(world)]
    all_val = [torch.empty_like(val) for _ in range(world)]
    dist.all_gather(all_idx, idx, group=group)
    dist.all_gather(all_val, val, group=group)
    for q, o, m in segs:
        idx[o:o + m] = all_idx[q][o:o + m]
        val[o:o + m] = all_val[q][o:o + m]
    return _order_pairs(idx, val, n)


def _edge_keys(edges, n, device):
    """Sorted distinct undirected keys min(a, b) * n + max(a, b) of the true edges, self-loops dropped.  `edges`: an E x 2
    array / tensor of node pairs, or a sparse COO (torch) or scipy sparse adjacency (non-zero entries are edges)."""
    import scipy.sparse as sp
    if torch.is_tensor(edges) and edges.is_sparse:
        a = edges.coalesce()
        e = a.indices()[:, a.values() != 0].t()
    elif sp.issparse(edges):
        c = edges.tocoo()
        nz = c.data != 0
        e = torch.from_numpy(np.stack([c.row[nz], c.col[nz]], 1).astype(np.int64))
    else:
        e = torch.as_tensor(np.asarray(edges) if not torch.is_tensor(edges) else edges).reshape(-1, 2)
    e = e.to(device=device, dtype=torch.int64)
    if e.numel() and (int(e.min()) < 0 or int(e.max()) >= n):
        raise ValueError(f"edge endpoints outside [0, {n})")
    e = e[e[:, 0] != e[:, 1]]
    lo, hi = torch.minimum(e[:, 0], e[:, 1]), torch.maximum(e[:, 0], e[:, 1])
    return torch.unique(lo * n + hi)


def precision_recall_at_k(rows, cols, edges, n):
    """Precision hits / k and recall hits / |E| of the k pairs (rows[q], cols[q]) against the undirected true edges
    (self-loops dropped, duplicates and both orientations counted once).  Returns (precision, recall) as floats."""
    rows = torch.as_tensor(rows).reshape(-1).to(torch.int64)
    cols = torch.as_tensor(cols).reshape(-1).to(device=rows.device, dtype=torch.int64)
    keys = _edge_keys(edges, int(n), rows.device)
    k, ne = rows.numel(), keys.numel()
    if k == 0 or ne == 0:
        return 0.0, 0.0
    q = torch.minimum(rows, cols) * n + torch.maximum(rows, cols)
    pos = torch.searchsorted(keys, q).clamp_(max=ne - 1)
    hits = int((keys[pos] == q).sum())
    return hits / k, hits / ne
