"""NumPy reference of the audience calls (mr_audience_scores / mr_catalogue_audience): test and benchmark infrastructure
only.  It is catalogue_oracle.catalogue_topk on the transposed score matrix restricted to the pool's valid users, with
the exclusion lists and targets mapped to pool positions and pos clipped at k."""

import numpy as np

from catalogue_oracle import catalogue_topk, csr
from oracle import movierec_oracle as o

INT32_MAX = np.iinfo(np.int32).max


def audience(p, k, users=None, num_users=INT32_MAX, excl_rowptr=None, excl_users=None, excl_ids=None, targets=None):
    """p (U, M): row u is user users[u] (default u; strictly ascending), column j an item.  For each column, the k best
    users with an id in [0, num_users) not on the column's exclusion list (row r = excl_ids[j], default j, of
    (excl_rowptr, excl_users); rows outside the table exclude nothing), in descending score (NaN as -inf, the lower user
    id first among ties).  targets (M,): never excluded; pos[j] = the target's place among the candidates when < k,
    else k (also for a target outside the pool).  Returns (users (M, k) int32 with -1 padding, scores (M, k) float32
    with NaN padding, pos or None, (hit_sum, dcg_sum) or None)."""
    p = np.asarray(p, np.float32)
    U, M = p.shape
    ids = np.arange(U, dtype=np.int64) if users is None else np.asarray(users, np.int64).reshape(-1)
    valid = np.flatnonzero((ids >= 0) & (ids < num_users))
    vids = ids[valid]

    def at_pool(x):  # pool positions of the ids x, -1 where absent
        x = np.asarray(x, np.int64).reshape(-1)
        at = np.searchsorted(vids, x)
        ok = at < vids.size
        ok[ok] = vids[at[ok]] == x[ok]
        return np.where(ok, at, -1)

    lists = []
    for j in range(M):
        r = int(excl_ids[j]) if excl_ids is not None else j
        ex = []
        if excl_rowptr is not None and 0 <= r < len(excl_rowptr) - 1:
            a = at_pool(excl_users[int(excl_rowptr[r]):int(excl_rowptr[r + 1])])
            ex = a[a >= 0]
        lists.append(ex)
    rp, it = csr(lists)
    tpos = at_pool(targets) if targets is not None else None
    top, scores, pos, _ = catalogue_topk(p[valid].T, k, rp, it, targets=tpos)
    top_users = np.where(top >= 0, vids[np.maximum(top, 0)] if vids.size else -1, -1).astype(np.int32)
    sums = None
    if pos is not None:
        pos = np.where(tpos < 0, k, np.minimum(pos, k)).astype(np.int32)
        sums = o.metrics_from_positions(pos, k)
    return top_users, scores, pos, sums
