"""NumPy reference of the catalogue top-k calls (mr_topk_scores / mr_catalogue_topk): test and benchmark
infrastructure only, built on the oracle's RankLayer key (oracle.movierec_oracle.rank_groups) and metric sums
(metrics_from_positions)."""

import numpy as np

from oracle import movierec_oracle as o


def catalogue_topk(p, k, excl_rowptr, excl_items, excl_ids=None, targets=None):
    """Top-k of each row of p (U, N) over the items not in the row's exclusion list, in the RankLayer order of
    rank_groups (descending, NaN as -inf, the lower item id first among ties).  Row u uses the list
    excl_items[excl_rowptr[r]:excl_rowptr[r+1]], r = excl_ids[u] (default u); rows outside the table, ids outside
    [0, N) and excl_rowptr None exclude nothing.  targets: never excluded; pos[u] = the target's place among the
    candidates (N when the target lies outside [0, N)).  Returns (items (U, k) int32 with -1 padding, scores (U, k)
    float32 with NaN padding, pos or None, (hit_sum, dcg_sum) or None)."""
    p = np.asarray(p, dtype=np.float32)
    U, N = p.shape
    items = np.full((U, k), -1, np.int32)
    scores = np.full((U, k), np.nan, np.float32)
    pos = np.zeros(U, np.int32) if targets is not None else None
    for u in range(U):
        keep = np.ones(N, bool)
        r = int(excl_ids[u]) if excl_ids is not None else u
        if excl_rowptr is not None and 0 <= r < len(excl_rowptr) - 1:
            ex = np.asarray(excl_items[int(excl_rowptr[r]):int(excl_rowptr[r + 1])], np.int64)
            keep[ex[(ex >= 0) & (ex < N)]] = False
        t = int(targets[u]) if targets is not None else -1
        if 0 <= t < N:
            keep[t] = True
        cand = np.flatnonzero(keep)
        key = np.where(np.isnan(p[u, cand]), -np.inf, p[u, cand])
        order = cand[np.argsort(-key, kind="stable")]
        m = min(k, order.size)
        items[u, :m] = order[:m]
        scores[u, :m] = p[u, order[:m]]
        if pos is not None:
            pos[u] = int(np.flatnonzero(order == t)[0]) if 0 <= t < N else N
    sums = o.metrics_from_positions(pos, k) if pos is not None else None
    return items, scores, pos, sums


def csr(lists):
    """[[items of row 0], [items of row 1], ...] -> (rowptr int64, items int32), each list sorted ascending."""
    rowptr = np.zeros(len(lists) + 1, np.int64)
    rowptr[1:] = np.cumsum([len(x) for x in lists])
    items = np.concatenate([np.sort(np.asarray(x, np.int32)) for x in lists]) if lists else np.zeros(0, np.int32)
    return rowptr, items.astype(np.int32)
