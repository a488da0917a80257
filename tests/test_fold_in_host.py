"""Fold-in's host-side surface, CPU only: the workspace query, the C ABI's refusals before any device work, the parsing
and checking of histories, and the NumPy reference on hand-checkable cases."""

import ctypes

import numpy as np
import pytest

from fold_in_oracle import fold_in, fold_in_user
from movierec import _engine
from movierec import _native as nat
from oracle import movierec_oracle as o
from test_catalogue_targets_host import _model_desc

MR_ERR_INVALID, MR_ERR_WORKSPACE = -1, -2


def test_workspace_query_needs_no_device():
    q = nat.lib.mr_fold_in_workspace_bytes
    for layers, mf in (([256, 128, 64], 64), ([64, 32, 16, 8], 8), ([6, 4], 0), ([7], 3)):
        m = _model_desc(layers, mf, 138493, 26744, fake_params=True)
        a = q(ctypes.byref(m), 10000, 1000000)
        assert a > 0
        if len(layers) > 1:
            assert a >= 26744 * layers[1] * 4  # the item half of the first layer
        assert q(ctypes.byref(m), 20000, 1000000) > a  # grows with the users (their sort)
        assert q(ctypes.byref(m), 10000, 0) == a  # not with the ratings
        assert q(ctypes.byref(m), 0, 0) > 0
        for bad in ((-1, 0), (10, -1), (1 << 31, 0), (10, 1 << 31)):
            assert q(ctypes.byref(m), *bad) == 0, bad
    assert q(None, 10, 10) == 0
    assert q(ctypes.byref(_model_desc([256, 128, 64], 64, 10, 10)), 10, 10) == 0  # no parameters


def _cfg(**kw):
    c = nat.MrFoldIn()
    c.steps, c.negs, c.optimizer, c.lr, c.beta_1, c.beta_2, c.epsilon, c.seed = 3, 4, nat.OPT_ADAM, 0.05, 0.9, 0.999, 1e-7, 1
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def test_argument_validation_needs_no_device():
    fake = ctypes.c_void_p(16)  # never dereferenced: validation fails first
    m = _model_desc([256, 128, 64], 64, 100, 50, fake_params=True)
    ws = (ctypes.c_char * 256)()
    good = dict(rowptr=fake, items=fake, U=4, nnz=8, init=None, cfg=_cfg(), mlp=fake, gmf=fake, ws_bytes=256)

    def call(rowptr, items, U, nnz, init, cfg, mlp, gmf, ws_bytes):
        return nat.lib.mr_fold_in_users(ctypes.byref(m), rowptr, items, U, nnz, init,
                                        ctypes.byref(cfg) if cfg is not None else None, mlp, gmf, None, ws, ws_bytes,
                                        None)

    bad = [dict(cfg=None), dict(cfg=_cfg(steps=-1)), dict(cfg=_cfg(negs=0)), dict(cfg=_cfg(negs=nat.MR_MAX_NEGS + 1)),
           dict(cfg=_cfg(optimizer=2)), dict(cfg=_cfg(lr=float("nan"))), dict(cfg=_cfg(beta_1=1.0)),
           dict(cfg=_cfg(epsilon=0.0)), dict(U=-1), dict(nnz=-1), dict(U=1 << 31), dict(rowptr=None), dict(items=None),
           dict(mlp=None), dict(gmf=None)]
    for change in bad:
        assert call(**dict(good, **change)) == MR_ERR_INVALID, change
        assert "fold_in" in nat.last_error(), change
    # SGD takes no betas; an empty history set needs no items
    assert call(**dict(good, cfg=_cfg(optimizer=nat.OPT_SGD, beta_1=1.0))) == MR_ERR_WORKSPACE
    assert call(**dict(good, items=None, nnz=0)) == MR_ERR_WORKSPACE
    assert call(**good) == MR_ERR_WORKSPACE
    assert "workspace" in nat.last_error()
    m0 = _model_desc([6, 4], 0, 100, 50, fake_params=True)  # no GMF branch: out_user_gmf may be NULL
    assert nat.lib.mr_fold_in_users(ctypes.byref(m0), fake, fake, 4, 8, None, ctypes.byref(_cfg()), fake, None, None,
                                    ws, 256, None) == MR_ERR_WORKSPACE


def test_histories_are_parsed_and_checked():
    rowptr, items = _engine.fold_in_histories([[5, 2, 2, 9], [], np.int64([3])], 10)
    assert rowptr.tolist() == [0, 3, 3, 4] and items.tolist() == [2, 5, 9, 3] and items.dtype == np.int32
    rp, it = _engine.fold_in_histories((np.int64([0, 2, 2]), np.int32([1, 4])), 10)
    assert rp.tolist() == [0, 2, 2] and it.tolist() == [1, 4]
    assert _engine.fold_in_histories([], 10)[0].tolist() == [0]
    with pytest.raises(IndexError):
        _engine.fold_in_histories([[1, 10]], 10)
    with pytest.raises(IndexError):
        _engine.fold_in_histories([[-1]], 10)
    for bad in ((np.int64([1, 2]), np.int32([1, 4])), (np.int64([0, 3]), np.int32([1, 4])),
                (np.int64([0, 2, 1, 2]), np.int32([1, 4])), (np.int64([0, 2]), np.int32([4, 1])),
                (np.int64([0, 2]), np.int32([4, 4]))):
        with pytest.raises(ValueError):
            _engine.fold_in_histories(bad, 10)
    # a list may end where the next starts with a smaller id
    assert _engine.fold_in_histories((np.int64([0, 2, 4]), np.int32([3, 7, 1, 2])), 10)[1].tolist() == [3, 7, 1, 2]
    with pytest.raises(ValueError, match="covers every item"):
        _engine.fold_in_histories([list(range(10))], 10)
    assert _engine.fold_in_histories([list(range(9))], 10)[0].tolist() == [0, 9]


def _model(layers, mf, nu=6, ni=40, seed=3, dtype=np.float64):
    return o.init_weights(nu, ni, layers, mf, np.random.default_rng(seed), dtype)


def test_reference_zero_steps_and_empty_history():
    w = _model([8, 4], 2)
    rows, loss = fold_in_user(w, [1, 5], 0, 3, 0)
    assert not rows[o.K_USER].any() and not rows[o.K_GMF_USER].any() and np.isnan(loss)
    init = {o.K_USER: w[o.K_USER][2], o.K_GMF_USER: w[o.K_GMF_USER][2]}
    rows, _ = fold_in_user(w, [], 4, 3, 0, init=init)  # no rows and no l2: nothing moves
    np.testing.assert_array_equal(rows[o.K_USER], w[o.K_USER][2])
    rows, _ = fold_in_user(w, [], 1, 3, 0, l2_0=0.5, optimizer="sgd", lr=0.1, init=init)  # the l2 term alone
    np.testing.assert_allclose(rows[o.K_USER], w[o.K_USER][2] * (1 - 0.1 * 2 * 0.5))


def test_reference_one_sgd_step_by_hand():
    """No hidden layer, no GMF: z = b + w_u . e_u + w_i . e_i, and from e_u = 0 one SGD step moves e_u by
    -lr * mean(p - y) * w_u."""
    w = _model([4], 0)
    hist = [3, 7]
    negs, seed = 2, 9
    rows, loss = fold_in_user(w, hist, 1, negs, seed, optimizer="sgd", lr=0.5)
    rowptr = np.int64([0, 2])
    items = np.concatenate([np.append(o.device_sample_group(rowptr, np.int64(hist), 40, 0, j, negs, seed, 0), hist[j])
                            for j in range(2)])
    wu, wi = w[o.K_OUT_W][:2, 0], w[o.K_OUT_W][2:, 0]
    z = w[o.K_OUT_B][0] + w[o.K_ITEM][items] @ wi
    y = np.tile([0, 0, 1], 2)
    dz = o.sigmoid(z) - y
    np.testing.assert_allclose(rows[o.K_USER], -0.5 * dz.mean() * wu, rtol=1e-12)
    np.testing.assert_allclose(loss, o.bce_from_logits(z, y).mean(), rtol=1e-12)
    assert not set(items[[0, 1, 3, 4]].tolist()) & set(hist)  # negatives avoid the history


def test_reference_is_per_user_and_float32_tracks_float64():
    w64 = _model([9, 5, 3], 3)
    w32 = {k: v.astype(np.float32) for k, v in w64.items()}
    rowptr, items = np.int64([0, 3, 3, 8]), np.int64([1, 4, 9, 0, 2, 3, 30, 39])
    a = fold_in(w64, rowptr, items, 3, 4, 5, init_users=[-1, 2, 0], l2_0=0.01)
    b = fold_in(w32, rowptr, items, 3, 4, 5, init_users=[-1, 2, 0], l2_0=0.01)
    assert b[0].dtype == np.float32
    np.testing.assert_allclose(b[0], a[0], rtol=1e-3, atol=1e-5)
    np.testing.assert_allclose(b[1], a[1], rtol=1e-3, atol=1e-5)
    assert np.isnan(a[2][1]) and np.isfinite(a[2][[0, 2]]).all()
    alone = fold_in_user(w64, items[3:8], 3, 4, 5, l2_0=0.01, init={o.K_USER: w64[o.K_USER][0],
                                                                    o.K_GMF_USER: w64[o.K_GMF_USER][0]})
    np.testing.assert_array_equal(alone[0][o.K_USER], a[0][2])
