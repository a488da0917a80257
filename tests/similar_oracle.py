"""NumPy reference of similar items / users (mr_similar): the representation and the similarity in float64 and float32,
and the selection through catalogue_oracle.catalogue_topk with each query's own id merged into its exclusion list.  Test
and benchmark infrastructure only."""

import numpy as np

from catalogue_oracle import catalogue_topk, csr

K_USER, K_ITEM = "user_embedding/embeddings", "item_embedding/embeddings"
K_GMF_USER, K_GMF_ITEM = "gmf_user_embedding/embeddings", "gmf_item_embedding/embeddings"


def side_parts(w, side, mf):
    """Keras weights -> (E (N, d), W1_s (d, L1) or None, G (N, f) or None, w_gmf (f,) or None) of side "items" / "users":
    W1_s is the side's row block of hidden_1 (user rows first), w_gmf the GMF block of the output kernel."""
    E = np.asarray(w[K_ITEM if side == "items" else K_USER])
    W1 = w.get("hidden_1/kernel")
    W1s = None
    if W1 is not None:
        d_u = np.asarray(w[K_USER]).shape[1]
        W1s = np.asarray(W1)[d_u:] if side == "items" else np.asarray(W1)[:d_u]
    G = np.asarray(w[K_GMF_ITEM if side == "items" else K_GMF_USER]) if mf else None
    wg = np.asarray(w["output/kernel"]).reshape(-1)[:mf] if mf else None
    return E, W1s, G, wg


def representation(E, W1s, G, w_gmf, dtype=np.float64):
    """r_x = concat(p_x / |p_x|, g_x / |g_x|) / sqrt(n_parts) for every row: p = E . W1s (no bias), g = w_gmf * G; a
    part with zero norm stays zero; n_parts counts the parts the model has."""
    parts = []
    if W1s is not None:
        parts.append(np.asarray(E, dtype) @ np.asarray(W1s, dtype))
    if G is not None:
        parts.append(np.asarray(w_gmf, dtype)[None, :] * np.asarray(G, dtype))
    scale = dtype(1.0) / np.sqrt(dtype(len(parts)))
    out = []
    for p in parts:
        nrm = np.sqrt((p * p).sum(axis=1, keepdims=True))
        out.append(np.where(nrm > 0, p / np.where(nrm > 0, nrm, 1), 0).astype(dtype) * scale)
    return np.concatenate(out, axis=1)


def similarity(R, ids):
    """(M, N) similarities of the queries ids against every row; an out-of-range query's row is 0."""
    ids = np.asarray(ids, np.int64)
    ok = (ids >= 0) & (ids < R.shape[0])
    Q = np.zeros((ids.size, R.shape[1]), R.dtype)
    Q[ok] = R[ids[ok]]
    return Q @ R.T


def truth(w, side, mf, ids):
    """(float32, float64) similarities of ids against every row of the side."""
    parts = side_parts(w, side, mf)
    return similarity(representation(*parts, dtype=np.float32), ids), similarity(representation(*parts), ids)


def similar_select(scores, ids, k, excl_rowptr=None, excl_items=None, excl_ids=None):
    """The selection of mr_similar on its own scores (M, N): catalogue_topk over the candidates [0, N) minus the query
    and its exclusion list (row excl_ids[j], default j); an out-of-range query gets -1 / NaN everywhere."""
    scores = np.asarray(scores, np.float32)
    M, N = scores.shape
    ids = np.asarray(ids, np.int64)
    lists = []
    for j in range(M):
        r = int(excl_ids[j]) if excl_ids is not None else j
        ex = set()
        if excl_rowptr is not None and 0 <= r < len(excl_rowptr) - 1:
            ex = set(int(x) for x in excl_items[int(excl_rowptr[r]):int(excl_rowptr[r + 1])])
        if 0 <= ids[j] < N:
            ex.add(int(ids[j]))
        lists.append(sorted(ex))
    rp, ex = csr(lists)
    top, sc, _, _ = catalogue_topk(scores, k, rp, ex)
    bad = (ids < 0) | (ids >= N)
    top[bad] = -1
    sc[bad] = np.nan
    return top, sc
