"""NumPy restatement of mr_fold_in_users (include/movierec_b200.h), built from the oracle's own pieces: for each step,
the negatives of every positive from `device_sample_group` on the history as a one-user CSR (index = position in the
list, epoch = step), `forward` / `backward` of a one-user model whose user tables are the rows being folded in (the
gradient of those rows only, with the l2[0] term), then `adam_step` (per-user state, iterations = step + 1) or
`sgd_step`.  Runs in the dtype of the weights it is given (float32 or float64)."""

import numpy as np

from oracle import movierec_oracle as o

USER_KEYS = (o.K_USER, o.K_GMF_USER)


def fold_in_user(w, hist, steps, negs, seed, l2_0=0.0, optimizer="adam", lr=0.05, beta_1=0.9, beta_2=0.999,
                 init=None):
    """One user.  w: the model's weights (dict of the oracle's layout, any dtype); hist: ascending item ids; init: None
    (zero rows) or {K_USER: row, K_GMF_USER: row}.  Returns ({K_USER: row, K_GMF_USER: row (if GMF)}, last loss)."""
    dt = w[o.K_ITEM].dtype
    num_items = w[o.K_ITEM].shape[0]
    hist = np.asarray(hist, np.int64)
    n = hist.size
    sub = {k: v for k, v in w.items() if k not in USER_KEYS}
    rows = {}
    for k in USER_KEYS:
        if k in w:
            rows[k] = (np.zeros((1, w[k].shape[1]), dt) if init is None else
                       np.asarray(init[k], dt).reshape(1, -1).copy())
    state = {"iterations": 0, "m": {k: np.zeros_like(v) for k, v in rows.items()},
             "v": {k: np.zeros_like(v) for k, v in rows.items()}}
    rowptr = np.array([0, n], np.int64)
    loss = float("nan")
    L = [0] * o._num_layers(w)
    L[0] = l2_0
    for t in range(steps):
        model = dict(sub, **rows)
        if n:
            groups = [np.append(o.device_sample_group(rowptr, hist, num_items, 0, j, negs, seed, t), hist[j])
                      for j in range(n)]
            items = np.concatenate(groups).astype(np.int64)
            y = np.tile([0] * negs + [1], n).astype(dt)
        else:
            items = np.zeros(0, np.int64)
            y = np.zeros(0, dt)
        users = np.zeros(items.size, np.int64)
        if n:
            c = o.forward(model, users, items)
            loss = float(np.mean(o.bce_from_logits(c["z"], y), dtype=np.float64))
            g = o.backward(model, c, y, None, L)
            grads = {k: g[k] for k in rows}
        else:
            loss = float("nan")
            grads = {k: dt.type(2.0 * l2_0) * v for k, v in rows.items()}
        if optimizer == "adam":
            o.adam_step(rows, state, grads, lr, beta_1, beta_2)
        else:
            o.sgd_step(rows, grads, lr)
    return {k: v[0] for k, v in rows.items()}, loss


def fold_in(w, rowptr, items, steps, negs, seed, init_users=None, **kw):
    """Every user of a CSR: (user_mlp (U, d_u), user_gmf (U, f) or None, loss (U,))."""
    U = len(rowptr) - 1
    mlp, gmf, loss = [], [], []
    for u in range(U):
        init = None
        if init_users is not None and init_users[u] >= 0:
            init = {k: w[k][init_users[u]] for k in USER_KEYS if k in w}
        r, lo = fold_in_user(w, items[rowptr[u]:rowptr[u + 1]], steps, negs, seed, init=init, **kw)
        mlp.append(r[o.K_USER])
        gmf.append(r.get(o.K_GMF_USER))
        loss.append(lo)
    dt = w[o.K_ITEM].dtype
    d_u = w[o.K_USER].shape[1]
    out_mlp = np.array(mlp, dt).reshape(U, d_u)
    out_gmf = np.array(gmf, dt).reshape(U, -1) if o.K_GMF_USER in w else None
    return out_mlp, out_gmf, np.array(loss, np.float64)
