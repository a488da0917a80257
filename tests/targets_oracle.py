"""NumPy reference of the many-targets catalogue calls (mr_targets_scores / mr_catalogue_targets): test and benchmark
infrastructure only, built on catalogue_oracle's order (descending score, NaN as -inf, -0 == +0, the lower item id first
among ties) and the same exclusion rules."""

import math

import numpy as np

N_METRICS = 5  # hit, precision, recall, ndcg, map per cutoff (MR_TGT_HIT .. MR_TGT_MAP)


def target_positions(p, tgt_rowptr, tgt_items, excl_rowptr=None, excl_items=None, excl_ids=None, bad_rows=()):
    """tpos (nnz,) int32 in list order: for row u with targets tgt_items[tgt_rowptr[u]:tgt_rowptr[u+1]], the number of
    candidates ordered before each target, where the candidates are the items not on the row's exclusion list (list
    excl_ids[u], default u; rows outside the table and ids outside [0, N) exclude nothing) plus every target of the
    row.  N for a target outside [0, N) and for every target of a row in bad_rows (an out-of-range user)."""
    p = np.asarray(p, dtype=np.float32)
    U, N = p.shape
    tgt_rowptr = np.asarray(tgt_rowptr, np.int64)
    tgt_items = np.asarray(tgt_items, np.int64)
    tpos = np.full(tgt_items.size, N, np.int32)
    for u in range(U):
        b, e = int(tgt_rowptr[u]), int(tgt_rowptr[u + 1])
        if b == e or u in bad_rows:
            continue
        keep = np.ones(N, bool)
        r = int(excl_ids[u]) if excl_ids is not None else u
        if excl_rowptr is not None and 0 <= r < len(excl_rowptr) - 1:
            ex = np.asarray(excl_items[int(excl_rowptr[r]):int(excl_rowptr[r + 1])], np.int64)
            keep[ex[(ex >= 0) & (ex < N)]] = False
        t = tgt_items[b:e]
        inside = (t >= 0) & (t < N)
        keep[t[inside]] = True
        cand = np.flatnonzero(keep)
        key = np.where(np.isnan(p[u, cand]), -np.inf, p[u, cand])
        order = cand[np.argsort(-key, kind="stable")]  # -0 and +0 compare equal: stable keeps the lower id first
        place = np.full(N, N, np.int64)
        place[order] = np.arange(order.size)
        tpos[b:e] = np.where(inside, place[np.clip(t, 0, N - 1)], N)
    return tpos


def gain(p):
    return math.log(2.0) / math.log(p + 2.0)


def target_metrics(tpos, tgt_rowptr, ks):
    """float64 sums [users with a target, mrr, then per cutoff k: hit, precision, recall, ndcg, map] of the
    positions, the rules of movierec_b200.h (rows with an empty list are skipped)."""
    tgt_rowptr = np.asarray(tgt_rowptr, np.int64)
    out = np.zeros(2 + N_METRICS * len(ks), np.float64)
    for u in range(tgt_rowptr.size - 1):
        b, e = int(tgt_rowptr[u]), int(tgt_rowptr[u + 1])
        if b == e:
            continue
        ps = np.sort(np.asarray(tpos[b:e], np.int64))
        n = ps.size
        out[0] += 1.0
        out[1] += 1.0 / (ps[0] + 1.0)
        for c, k in enumerate(ks):
            h = int(np.sum(ps < k))
            m = min(k, n)
            idcg = sum(gain(i) for i in range(m))
            base = 2 + N_METRICS * c
            out[base + 0] += 1.0 if ps[0] < k else 0.0
            out[base + 1] += h / k
            out[base + 2] += h / n
            out[base + 3] += sum(gain(int(x)) for x in ps[:h]) / idcg
            out[base + 4] += sum((j + 1) / (int(x) + 1.0) for j, x in enumerate(ps[:h])) / m
    return out
