"""NumPy restatement of mr_fold_in_items (include/movierec_b200.h): fold_in_oracle's procedure with the sides swapped,
built from the same oracle pieces, and the role-swapped model under which item fold-in equals user fold-in.  Runs in
the dtype of the weights it is given (float32 or float64)."""

import numpy as np

from oracle import movierec_oracle as o

ITEM_KEYS = (o.K_ITEM, o.K_GMF_ITEM)


def fold_in_item(w, raters, steps, negs, seed, l2_0=0.0, optimizer="adam", lr=0.05, beta_1=0.9, beta_2=0.999,
                 init=None):
    """mr_fold_in_items for one item: fold_in_user with the sides swapped, for any L[0] (odd ones give the item rows one
    more column than the user rows).  raters: ascending user ids; the negatives are users drawn by
    `device_sample_group` over num_users candidates.  init: None (zero rows) or {K_ITEM: row, K_GMF_ITEM: row}.
    Returns ({K_ITEM: row, K_GMF_ITEM: row (if GMF)}, last loss)."""
    dt = w[o.K_USER].dtype
    num_users = w[o.K_USER].shape[0]
    raters = np.asarray(raters, np.int64)
    n = raters.size
    sub = {k: v for k, v in w.items() if k not in ITEM_KEYS}
    rows = {}
    for k in ITEM_KEYS:
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
            groups = [np.append(o.device_sample_group(rowptr, raters, num_users, 0, p, negs, seed, t), raters[p])
                      for p in range(n)]
            users = np.concatenate(groups).astype(np.int64)
            y = np.tile([0] * negs + [1], n).astype(dt)
            c = o.forward(model, users, np.zeros(users.size, np.int64))
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


def swap_sides(w):
    """The role-swapped model: user and item tables exchanged, the row blocks of W[1] exchanged ([W1i; W1u]) and,
    without a hidden layer, the two MLP halves of the output kernel exchanged.  It scores (i, u) as w scores (u, i),
    so fold_in_item on w equals fold_in_user on swap_sides(w).  For an odd L[0] the swapped user rows are the wider
    ones: the oracle, which reads widths from the tables, takes that; the library's layout (d_u = L[0] // 2) does not."""
    d_u = w[o.K_USER].shape[1]
    s = dict(w)
    s[o.K_USER], s[o.K_ITEM] = w[o.K_ITEM], w[o.K_USER]
    if o.K_GMF_USER in w:
        s[o.K_GMF_USER], s[o.K_GMF_ITEM] = w[o.K_GMF_ITEM], w[o.K_GMF_USER]
    if o._num_layers(w) > 1:
        k1 = o.hidden_names(1)[0]
        s[k1] = np.concatenate([w[k1][d_u:], w[k1][:d_u]])
    else:
        f = w[o.K_GMF_USER].shape[1] if o.K_GMF_USER in w else 0
        wo = w[o.K_OUT_W]
        s[o.K_OUT_W] = np.concatenate([wo[:f], wo[f + d_u:], wo[f:f + d_u]])
    return s
