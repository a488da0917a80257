"""Item fold-in's host-side surface, CPU only: the workspace query, the C ABI's refusals before any device work, the
parsing and checking of rater lists, and the NumPy reference against user fold-in on the role-swapped model and on a
hand-checkable case."""

import ctypes

import numpy as np
import pytest

from fold_in_items_oracle import fold_in_item, swap_sides
from fold_in_oracle import fold_in_user
from movierec import _engine
from movierec import _native as nat
from oracle import movierec_oracle as o
from test_catalogue_targets_host import _model_desc
from test_fold_in_host import _cfg

MR_ERR_INVALID, MR_ERR_WORKSPACE = -1, -2


def test_workspace_query_needs_no_device():
    q = nat.lib.mr_fold_in_items_workspace_bytes
    for layers, mf in (([256, 128, 64], 64), ([64, 32, 16, 8], 8), ([6, 4], 0), ([7], 3)):
        m = _model_desc(layers, mf, 138493, 26744, fake_params=True)
        a = q(ctypes.byref(m), 2000, 140000)
        assert a > 0
        if len(layers) > 1:
            assert a >= 138493 * layers[1] * 4  # the user half of the first layer
            more = _model_desc(layers, mf, 2 * 138493, 26744, fake_params=True)
            assert q(ctypes.byref(more), 2000, 140000) - a >= 138493 * layers[1] * 4 - 256  # grows with num_users x L[1]
        assert q(ctypes.byref(m), 4000, 140000) > a  # grows with the items (their sort)
        assert q(ctypes.byref(m), 2000, 0) == a  # not with the ratings
        assert q(ctypes.byref(m), 0, 0) > 0
        for bad in ((-1, 0), (10, -1), (1 << 31, 0), (10, 1 << 31)):
            assert q(ctypes.byref(m), *bad) == 0, bad
    assert q(None, 10, 10) == 0
    assert q(ctypes.byref(_model_desc([256, 128, 64], 64, 10, 10)), 10, 10) == 0  # no parameters
    bad = _model_desc([256, 128, 64], 64, 10, 10, fake_params=True)
    bad.n_layers = nat.MR_MAX_LAYERS + 1
    assert q(ctypes.byref(bad), 10, 10) == 0


def test_argument_validation_needs_no_device():
    fake = ctypes.c_void_p(16)  # never dereferenced: validation fails first
    m = _model_desc([256, 128, 64], 64, 100, 50, fake_params=True)
    ws = (ctypes.c_char * 256)()
    good = dict(rowptr=fake, users=fake, M=4, nnz=8, init=None, cfg=_cfg(), mlp=fake, gmf=fake, ws_bytes=256)

    def call(rowptr, users, M, nnz, init, cfg, mlp, gmf, ws_bytes):
        return nat.lib.mr_fold_in_items(ctypes.byref(m), rowptr, users, M, nnz, init,
                                        ctypes.byref(cfg) if cfg is not None else None, mlp, gmf, None, ws, ws_bytes,
                                        None)

    bad = [dict(cfg=None), dict(cfg=_cfg(steps=-1)), dict(cfg=_cfg(negs=0)), dict(cfg=_cfg(negs=nat.MR_MAX_NEGS + 1)),
           dict(cfg=_cfg(optimizer=2)), dict(cfg=_cfg(lr=float("nan"))), dict(cfg=_cfg(beta_1=1.0)),
           dict(cfg=_cfg(beta_2=-0.1)), dict(cfg=_cfg(epsilon=0.0)), dict(M=-1), dict(nnz=-1), dict(M=1 << 31),
           dict(nnz=1 << 31), dict(rowptr=None), dict(users=None), dict(mlp=None), dict(gmf=None)]
    for change in bad:
        assert call(**dict(good, **change)) == MR_ERR_INVALID, change
        assert "fold_in_items" in nat.last_error(), change
    assert nat.lib.mr_fold_in_items(None, fake, fake, 4, 8, None, ctypes.byref(_cfg()), fake, fake, None, ws, 256,
                                    None) == MR_ERR_INVALID
    # SGD takes no betas; an empty rater set needs no users; nothing to fold needs no outputs
    assert call(**dict(good, cfg=_cfg(optimizer=nat.OPT_SGD, beta_1=1.0))) == MR_ERR_WORKSPACE
    assert call(**dict(good, users=None, nnz=0)) == MR_ERR_WORKSPACE
    assert call(**dict(good, M=0, nnz=0, mlp=None, gmf=None)) == MR_ERR_WORKSPACE
    assert call(**good) == MR_ERR_WORKSPACE
    assert "workspace" in nat.last_error() and "fold_in_items" in nat.last_error()
    m0 = _model_desc([6, 4], 0, 100, 50, fake_params=True)  # no GMF branch: out_item_gmf may be NULL
    assert nat.lib.mr_fold_in_items(ctypes.byref(m0), fake, fake, 4, 8, None, ctypes.byref(_cfg()), fake, None, None,
                                    ws, 256, None) == MR_ERR_WORKSPACE


def test_rater_lists_are_parsed_and_checked():
    rowptr, users = _engine.fold_in_histories([[5, 2, 2, 9], [], np.int64([3])], 10, "items")
    assert rowptr.tolist() == [0, 3, 3, 4] and users.tolist() == [2, 5, 9, 3] and users.dtype == np.int32
    rp, us = _engine.fold_in_histories((np.int64([0, 2, 2]), np.int32([1, 4])), 10, "items")
    assert rp.tolist() == [0, 2, 2] and us.tolist() == [1, 4]
    with pytest.raises(IndexError, match="raters: a user lies outside"):
        _engine.fold_in_histories([[1, 10]], 10, "items")
    with pytest.raises(IndexError, match="user"):
        _engine.fold_in_histories([[-1]], 10, "items")
    for bad in ((np.int64([1, 2]), np.int32([1, 4])), (np.int64([0, 3]), np.int32([1, 4])),
                (np.int64([0, 2, 1, 2]), np.int32([1, 4])), (np.int64([0, 2]), np.int32([4, 1])),
                (np.int64([0, 2]), np.int32([4, 4]))):
        with pytest.raises(ValueError, match="raters"):
            _engine.fold_in_histories(bad, 10, "items")
    with pytest.raises(ValueError, match="covers every user"):
        _engine.fold_in_histories([list(range(10))], 10, "items")
    assert _engine.fold_in_histories([list(range(9))], 10, "items")[0].tolist() == [0, 9]
    # the user direction keeps its words
    with pytest.raises(ValueError, match="a history covers every item"):
        _engine.fold_in_histories([list(range(10))], 10)
    with pytest.raises(IndexError, match="histories: an item lies outside"):
        _engine.fold_in_histories([[10]], 10)


def _model(layers, mf, nu=40, ni=6, seed=3, dtype=np.float64):
    return o.init_weights(nu, ni, layers, mf, np.random.default_rng(seed), dtype)


@pytest.mark.parametrize("layers,mf", [([8, 4], 2), ([10, 6, 3], 3), ([6], 0), ([4], 2), ([7], 3), ([9, 5, 3], 2)])
@pytest.mark.parametrize("optimizer,l2_0", [("adam", 0.0), ("sgd", 0.01), ("adam", 0.01)])
def test_reference_is_user_fold_in_on_the_swapped_model(layers, mf, optimizer, l2_0):
    w = _model(layers, mf)
    s = swap_sides(w)
    raters = [3, 7, 8, 20, 33]
    lr = 0.05 if optimizer == "adam" else 0.5
    for init in (None, 2):
        ini = None if init is None else {k: w[k][init] for k in (o.K_ITEM, o.K_GMF_ITEM) if k in w}
        ini_s = None if init is None else {k: s[k][init] for k in (o.K_USER, o.K_GMF_USER) if k in s}
        a, la = fold_in_item(w, raters, 3, 4, 5, l2_0=l2_0, optimizer=optimizer, lr=lr, init=ini)
        b, lb = fold_in_user(s, raters, 3, 4, 5, l2_0=l2_0, optimizer=optimizer, lr=lr, init=ini_s)
        np.testing.assert_allclose(a[o.K_ITEM], b[o.K_USER], rtol=1e-12, atol=1e-15)
        if mf:
            np.testing.assert_allclose(a[o.K_GMF_ITEM], b[o.K_GMF_USER], rtol=1e-12, atol=1e-15)
        assert la == pytest.approx(lb, rel=1e-12)


def test_swapped_model_scores_the_transposed_pairs():
    for layers, mf in (([8, 4], 2), ([6], 3), ([7], 2), ([9, 4], 0)):
        w = _model(layers, mf)
        s = swap_sides(w)
        u, i = np.int64([0, 5, 39, 12]), np.int64([1, 0, 5, 3])
        np.testing.assert_allclose(o.forward(w, u, i)["z"], o.forward(s, i, u)["z"], rtol=1e-13)


def test_reference_one_sgd_step_by_hand_with_odd_width():
    """No hidden layer, no GMF, L[0] = 5: d_u = 2, d_i = 3, z = b + w_u . e_u + w_i . e_i, and from e_i = 0 one SGD
    step moves e_i by -lr * mean(p - y) * w_i."""
    w = _model([5], 0)
    raters = [3, 7, 30]
    negs, seed = 2, 9
    rows, loss = fold_in_item(w, raters, 1, negs, seed, optimizer="sgd", lr=0.5)
    assert rows[o.K_ITEM].shape == (3,)
    rowptr = np.int64([0, 3])
    users = np.concatenate([np.append(o.device_sample_group(rowptr, np.int64(raters), 40, 0, p, negs, seed, 0),
                                      raters[p]) for p in range(3)])
    wu, wi = w[o.K_OUT_W][:2, 0], w[o.K_OUT_W][2:, 0]
    z = w[o.K_OUT_B][0] + w[o.K_USER][users] @ wu
    y = np.tile([0, 0, 1], 3)
    dz = o.sigmoid(z) - y
    np.testing.assert_allclose(rows[o.K_ITEM], -0.5 * dz.mean() * wi, rtol=1e-12)
    np.testing.assert_allclose(loss, o.bce_from_logits(z, y).mean(), rtol=1e-12)
    negatives = users.reshape(3, 3)[:, :2].reshape(-1)
    assert not set(negatives.tolist()) & set(raters)  # negatives avoid the raters


def test_reference_zero_steps_and_float32_tracks_float64():
    w64 = _model([9, 5, 3], 3)
    w32 = {k: v.astype(np.float32) for k, v in w64.items()}
    rows, loss = fold_in_item(w64, [1, 5], 0, 3, 0)
    assert not rows[o.K_ITEM].any() and rows[o.K_ITEM].shape == (5,) and np.isnan(loss)
    init = {o.K_ITEM: w64[o.K_ITEM][2], o.K_GMF_ITEM: w64[o.K_GMF_ITEM][2]}
    raters = [0, 4, 9, 17, 30, 39]
    a, la = fold_in_item(w64, raters, 4, 4, 5, l2_0=0.01, init=init)
    b, lb = fold_in_item(w32, raters, 4, 4, 5, l2_0=0.01, init=init)
    assert b[o.K_ITEM].dtype == np.float32
    for k in a:
        np.testing.assert_allclose(b[k], a[k], rtol=1e-3, atol=1e-5)
    assert lb == pytest.approx(la, rel=1e-4)
