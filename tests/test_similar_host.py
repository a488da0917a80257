"""Similar items / users, host side and CPU only: the version and side constants, the workspace query (its formula and 0
on bad arguments), the C ABI's refusals before any device work, M == 0, and the NumPy reference on a hand-checked
case."""

import ctypes
import math

import numpy as np
import pytest

from movierec import _native as nat
from similar_oracle import representation, similar_select, similarity
from test_catalogue_targets_host import _model_desc

MR_ERR_INVALID, MR_ERR_WORKSPACE = -1, -2
ML20M = (138493, 26744)


def test_version_and_constants():
    assert nat.version() == 107
    assert (nat.SIDE_ITEMS, nat.SIDE_USERS) == (0, 1)


def _a(x):
    return (int(x) + 255) // 256 * 256


def expected_bytes(layers, mf, nu, ni, side, M, k):
    """The header's formula: projection, packed W1 block (tensor-core projection only), the side's operand image, the
    chunk's query image, the score chunk and the selection's workspace for one chunk."""
    items = side == nat.SIDE_ITEMS
    N = ni if items else nu
    L0 = layers[0]
    d = L0 - L0 // 2 if items else L0 // 2
    L1 = layers[1] if len(layers) >= 2 else 0
    C = max(1, min(M, max(1, min((1 << 22) // N, 16384))))
    D = (L1 + mf + 31) // 32 * 32
    tc_tower = (len(layers) >= 2 and L0 % 64 == 0 and all(w % 32 == 0 and w <= 256 for w in layers)
                and all(w % 128 == 0 for w in layers[:-1]) and all(w & (w - 1) == 0 for w in layers[1:])
                and mf + layers[-1] <= 512)
    tc_proj = tc_tower and len(layers) >= 3 and d % 128 == 0 and d <= 256 and L1 == d
    sel = nat.lib.mr_topk_scores_workspace_bytes(C, N, k) - 256
    return (_a(4 * N * L1) + (_a(8 * d * L1) if tc_proj else 0) + _a(8 * D * ((N + 255) // 256 * 256)) +
            _a(8 * D * ((C + 127) // 128 * 128)) + _a(4 * C * N) + _a(sel))


@pytest.mark.parametrize("layers,mf", [([256, 128, 64], 64), ([256, 128, 64], 0), ([64, 32, 16, 8], 8), ([6, 4], 0),
                                       ([8], 4), ([64, 512], 256)])
def test_workspace_formula(layers, mf):
    nu, ni = ML20M
    m = _model_desc(layers, mf, nu, ni, fake_params=True)
    q = lambda side, M, k: nat.lib.mr_similar_workspace_bytes(ctypes.byref(m), side, M, k)
    for side in (nat.SIDE_ITEMS, nat.SIDE_USERS):
        for M, k in ((1, 1), (400, 10), (26744, 1000), (138493, 4096), (0, 10)):
            assert q(side, M, k) == expected_bytes(layers, mf, nu, ni, side, M, k), (side, M, k)
        # bounded in the queries: one chunk
        assert q(side, 10 ** 6, 10) == q(side, 138493, 10)


def test_workspace_ml20m_values_in_the_header():
    nu, ni = ML20M
    m = _model_desc([256, 128, 64], 64, nu, ni, fake_params=True)
    items = nat.lib.mr_similar_workspace_bytes(ctypes.byref(m), nat.SIDE_ITEMS, ni, 10)
    users = nat.lib.mr_similar_workspace_bytes(ctypes.byref(m), nat.SIDE_USERS, nu, 10)
    assert round(items / 1e6, 1) == 72.5
    assert round(users / 1e6) == 301


def test_workspace_query_refuses_bad_arguments():
    nu, ni = 50, 70
    m = _model_desc([64, 32, 16, 8], 8, nu, ni, fake_params=True)
    q = lambda side, M, k, mm=m: nat.lib.mr_similar_workspace_bytes(ctypes.byref(mm) if mm is not None else None,
                                                                     side, M, k)
    assert q(0, 5, 10) > 0 and q(1, 5, 10) > 0
    for side, M, k in ((2, 5, 10), (-1, 5, 10), (0, -1, 10), (0, 1 << 31, 10), (0, 5, 0), (0, 5, 4097)):
        assert q(side, M, k) == 0, (side, M, k)
    assert q(0, 5, 4096) > 0
    assert q(0, 5, 10, None) == 0
    none = _model_desc([8], 0, nu, ni, fake_params=True)  # one layer, no GMF: nothing to compare
    assert q(0, 5, 10, none) == 0 and q(1, 5, 10, none) == 0
    gmf_only = _model_desc([8], 4, nu, ni, fake_params=True)
    assert q(0, 5, 10, gmf_only) > 0


def test_argument_validation_needs_no_device():
    nu, ni = 50, 70
    m = _model_desc([64, 32, 16, 8], 8, nu, ni, fake_params=True)
    fake = ctypes.c_void_p(16)  # never dereferenced: validation fails first
    need = nat.lib.mr_similar_workspace_bytes(ctypes.byref(m), 0, 3, 4)

    def call(model=None, side=0, ids=fake, M=3, k=4, excl_ids=None, excl_rows=0, rowptr=None, lst=None, ws=fake,
             ws_bytes=need):
        mm = ctypes.byref(m) if model is None else model
        return nat.lib.mr_similar(mm, side, ids, M, k, excl_ids, excl_rows, rowptr, lst, fake, fake, None, ws, ws_bytes,
                                  None)

    for change in ({"side": 2}, {"side": -1}, {"k": 0}, {"k": 4097}, {"M": -1}, {"M": 1 << 31}, {"ids": None},
                   {"ws": None}, {"excl_rows": -1}, {"rowptr": fake, "lst": None}):
        assert call(**change) == MR_ERR_INVALID, change
    assert nat.lib.mr_similar(None, 0, fake, 3, 4, None, 0, None, None, fake, fake, None, fake, need, None) == \
        MR_ERR_INVALID
    none = _model_desc([8], 0, nu, ni, fake_params=True)
    assert call(model=ctypes.byref(none)) == MR_ERR_INVALID and "no vector" in nat.last_error()
    assert call(ws_bytes=need - 1) == MR_ERR_WORKSPACE
    # M == 0: a no-op after the checks, whatever the pointers
    assert nat.lib.mr_similar(ctypes.byref(m), 1, None, 0, 4, None, 0, None, None, None, None, None, None, 0, None) == 0
    assert call(M=0, k=0) == MR_ERR_INVALID


def test_oracle_on_a_hand_checked_case():
    # two parts: p = E . W1s, g = w * G; row 2 has a zero MLP part, row 3 is all zero
    E = np.float64([[1, 0], [0, 2], [0, 0], [0, 0]])
    W1s = np.eye(2)
    G = np.float64([[1, 1], [1, -1], [3, 0], [0, 0]])
    w = np.float64([1, 2])
    R = representation(E, W1s, G, w)
    s = 1 / math.sqrt(2)
    np.testing.assert_allclose(R[0], [s, 0, s / math.sqrt(5), 2 * s / math.sqrt(5)])
    np.testing.assert_allclose(R[2], [0, 0, s, 0])
    assert not R[3].any()
    S = R @ R.T
    np.testing.assert_allclose(np.diag(S)[:2], 1.0)
    assert abs(S[2, 2] - 0.5) < 1e-12  # a row with one zero part
    top, sc = similar_select(similarity(R, [0, 3, 9]).astype(np.float32), [0, 3, 9], 4)
    assert 0 not in top[0] and 3 not in top[1]
    assert (top[2] == -1).all() and np.isnan(sc[2]).all()
    assert top[1].tolist() == [0, 1, 2, -1]  # all similarities 0: the lower id first
