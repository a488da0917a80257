"""NumPy reference of the ragged-list top-k calls (mr_topk_lists / mr_rank_lists): test and benchmark infrastructure
only, built on the oracle's RankLayer key (oracle.movierec_oracle.rank_groups: descending, NaN as -inf, a stable sort
so the earlier position wins ties) and metric sums (metrics_from_positions)."""

import numpy as np

from oracle import movierec_oracle as o


def topk_lists(scores, rowptr, k, targets=None, bad_lists=None):
    """Top-k positions of each list scores[rowptr[u]:rowptr[u+1]].  targets: a position per list; pos[u] = the number
    of candidates ordered before it (the list length when it lies outside [0, len)).  bad_lists: a boolean per list
    (an out-of-range user): -1 / NaN slots and pos = len.  Returns (top_pos (U, k) int32 with -1 padding, top_scores
    (U, k) float32 with NaN padding, pos or None, (hit_sum, dcg_sum) or None)."""
    s = np.asarray(scores, dtype=np.float32).reshape(-1)
    rowptr = np.asarray(rowptr, dtype=np.int64)
    U = rowptr.size - 1
    lens = np.diff(rowptr)
    seg = np.repeat(np.arange(U), lens)
    at = np.arange(s.size) - rowptr[seg]  # position in the list
    key = np.where(np.isnan(s), -np.inf, s)
    order = np.lexsort((at, -key, seg))  # per list: rank_groups' key, descending, the earlier position first
    rank = np.empty(s.size, np.int64)
    rank[order] = np.arange(s.size) - rowptr[seg[order]]
    bad = np.zeros(U, bool) if bad_lists is None else np.asarray(bad_lists, bool)
    top_pos = np.full((U, k), -1, np.int32)
    top_scores = np.full((U, k), np.nan, np.float32)
    sel = (rank < k) & ~bad[seg]
    top_pos[seg[sel], rank[sel]] = at[sel]
    top_scores[seg[sel], rank[sel]] = s[sel]
    pos = None
    if targets is not None:
        t = np.asarray(targets, np.int64).reshape(-1)
        ok = (t >= 0) & (t < lens) & ~bad
        pos = lens.astype(np.int32)
        pos[ok] = rank[rowptr[:-1][ok] + t[ok]]
    sums = o.metrics_from_positions(pos, k) if pos is not None else None
    return top_pos, top_scores, pos, sums


def csr(lists):
    """[[items of list 0], [items of list 1], ...] -> (rowptr int64, items int32), order kept."""
    rowptr = np.zeros(len(lists) + 1, np.int64)
    rowptr[1:] = np.cumsum([len(x) for x in lists])
    items = np.concatenate([np.asarray(x, np.int32).reshape(-1) for x in lists]) if lists else np.zeros(0, np.int32)
    return rowptr, items.astype(np.int32)
