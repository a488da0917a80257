"""Many held-out items per user against the whole catalogue: the NumPy reference against catalogue_oracle and against
hand-computed metrics, and the C ABI's host-side surface (workspace queries, argument validation).  CPU only."""

import ctypes
import math

import numpy as np
import pytest

from catalogue_oracle import catalogue_topk, csr
from movierec import _native as nat
from oracle import movierec_oracle as o
from targets_oracle import gain, target_metrics, target_positions

NAN = np.float32(np.nan)
P7 = np.float32([[0.5, 0.9, 0.5, NAN, 0.0, -0.0, 0.9]])  # order without exclusions: 1, 6, 0, 2, 4, 5, 3


def test_one_target_per_user_is_catalogue_topk():
    rng = np.random.default_rng(0)
    vals = np.float32([0.25, 0.5, 0.5, np.nan, np.inf, -np.inf, -0.0, 0.0])
    for N in (1, 7, 100):
        U = 12
        p = rng.choice(vals, (U, N)).astype(np.float32)
        ex_rowptr, ex = csr([sorted(rng.choice(N, rng.integers(0, N + 1), replace=False).tolist()) for _ in range(U)])
        targets = rng.integers(-1, N + 1, U).astype(np.int32)
        tgt_rowptr = np.arange(U + 1, dtype=np.int64)
        for k in (1, 3, 10):
            _, _, pos, sums = catalogue_topk(p, k, ex_rowptr, ex, targets=targets)
            tpos = target_positions(p, tgt_rowptr, targets, ex_rowptr, ex)
            np.testing.assert_array_equal(tpos, pos)
            m = target_metrics(tpos, tgt_rowptr, [k])
            hit, dcg = o.metrics_from_positions(pos, k)
            assert m[0] == U and m[2] == hit
            assert abs(m[5] - dcg) <= 1e-6 * max(dcg, 1.0)  # ndcg of one target = its dcg
            assert abs(m[3] - hit / k) <= 1e-12 and m[4] == hit  # precision, recall


def test_ties_and_a_listed_target():
    # no exclusions, targets 2 and 6: 6 ties with 1 (1 first), 2 ties with 0 (0 first)
    rowptr, items = np.int64([0, 2]), np.int32([2, 6])
    tpos = target_positions(P7, rowptr, items)
    assert tpos.tolist() == [3, 1]
    m = target_metrics(tpos, rowptr, [2])
    g1 = math.log(2) / math.log(3)
    np.testing.assert_allclose(m, [1, 1 / 2, 1, 1 / 2, 1 / 2, g1 / (1 + g1), (1 / 2) / 2], rtol=1e-12)
    # items 1, 2 and 6 excluded; target 6 is listed but never excluded, and item 2 no longer ties with target 0
    ex_rowptr, ex = csr([[1, 2, 6]])
    tpos = target_positions(P7, np.int64([0, 2]), np.int32([0, 6]), ex_rowptr, ex)
    assert tpos.tolist() == [1, 0]


def test_out_of_range_targets_and_cutoffs_beyond_the_catalogue():
    rowptr, items = np.int64([0, 3]), np.int32([-1, 1, 9])
    tpos = target_positions(P7, rowptr, items)
    assert tpos.tolist() == [7, 0, 7]  # N for a target outside [0, N); it still counts in n
    m = target_metrics(tpos, rowptr, [1, 10])
    g = [gain(i) for i in range(8)]
    want_k1 = [1, 1, 1 / 3, 1, 1]
    want_k10 = [1, 3 / 10, 1, (g[0] + 2 * g[7]) / (g[0] + g[1] + g[2]), (1 / 1 + 2 / 8 + 3 / 8) / 3]
    np.testing.assert_allclose(m, [1, 1] + want_k1 + want_k10, rtol=1e-12)
    # every target of an out-of-range user gets N
    assert target_positions(P7, rowptr, items, bad_rows=(0,)).tolist() == [7, 7, 7]


def test_more_targets_than_the_cutoff_and_empty_lists():
    rowptr, items = np.int64([0, 0, 4, 4]), np.int32([0, 1, 2, 6])  # users 0 and 2 have no targets
    p = np.vstack([P7, P7, P7])
    tpos = target_positions(p, rowptr, items)
    assert tpos.tolist() == [2, 0, 3, 1]
    m = target_metrics(tpos, rowptr, [2])
    np.testing.assert_allclose(m, [1, 1, 1, 1, 1 / 2, 1, 1], rtol=1e-12)  # empty lists are not counted
    assert target_metrics(np.zeros(0, np.int32), np.int64([0, 0, 0]), [5]).tolist() == [0.0] * 7


def _model_desc(layers, mf_dim, num_users, num_items, fake_params=False):
    m = nat.MrModel()
    m.n_layers, m.mf_dim, m.num_users, m.num_items = len(layers), mf_dim, num_users, num_items
    for i, w in enumerate(layers):
        m.L[i] = w
    if fake_params:  # addresses never dereferenced, laid out as the dense block requires
        base = 1 << 20
        m.user_mlp = m.item_mlp = m.user_gmf = m.item_gmf = base
        m.dense = base
        off = 0
        for l in range(1, len(layers)):
            m.W[l] = base + 4 * off
            off += layers[l - 1] * layers[l]
            m.b[l] = base + 4 * off
            off += layers[l]
        m.w_out = base + 4 * off
        off += mf_dim + layers[-1]
        m.b_out = base + 4 * off
        m.dense_count = off + 1
    return m


def test_workspace_queries_are_host_only_and_bounded_in_users():
    N, nnz = 26744, 1000
    chunk = (1 << 22) // N
    q = nat.lib.mr_targets_scores_workspace_bytes
    a = q(chunk, N, nnz)
    assert 0 < q(1, N, nnz) <= a
    assert q(10 * chunk, N, nnz) == a == q(138493, N, nnz)
    assert q(chunk, N, 2 * nnz) > a  # a few bytes per target
    assert q(chunk, N, 0) > 0
    for bad in ((-1, N, nnz), (chunk, 0, nnz), (chunk, N, -1), (chunk, N, 1 << 31), (1 << 31, N, nnz)):
        assert q(*bad) == 0, bad
    for layers, mf in (([256, 128, 64], 64), ([64, 32, 16, 8], 8), ([6, 4], 0)):
        m = _model_desc(layers, mf, 138493, N)
        one = nat.lib.mr_catalogue_targets_workspace_bytes(ctypes.byref(m), chunk, nnz)
        assert one >= chunk * N * 8  # item ids and probabilities of a chunk
        assert nat.lib.mr_catalogue_targets_workspace_bytes(ctypes.byref(m), 138493, nnz) == one
        assert nat.lib.mr_catalogue_targets_workspace_bytes(ctypes.byref(m), 1, nnz) < one
        assert nat.lib.mr_catalogue_targets_workspace_bytes(ctypes.byref(m), chunk, -1) == 0
    assert nat.lib.mr_catalogue_targets_workspace_bytes(None, 10, nnz) == 0


MR_ERR_INVALID, MR_ERR_WORKSPACE = -1, -2


def _calls():
    """(name, call(U, N, nnz, ks, n_ks, rowptr, tpos, sums, ws_bytes)) for both entry points, with fake pointers."""
    fake = ctypes.c_void_p(16)  # never dereferenced: validation fails first
    ws = (ctypes.c_char * 256)()

    def scores(U, N, nnz, ks, n_ks, rowptr, tpos, sums, ws_bytes):
        return nat.lib.mr_targets_scores(fake, U, N, None, 0, None, None, rowptr, fake, nnz, ks, n_ks, tpos, sums, ws,
                                         ws_bytes, None)

    def catalogue(U, N, nnz, ks, n_ks, rowptr, tpos, sums, ws_bytes):
        m = _model_desc([256, 128, 64], 64, 100, N, fake_params=True)
        return nat.lib.mr_catalogue_targets(ctypes.byref(m), fake, U, 0, None, None, rowptr, fake, nnz, ks, n_ks, tpos,
                                            sums, ws, ws_bytes, None)
    return [("scores", scores), ("catalogue", catalogue)], fake


@pytest.mark.parametrize("which", ["scores", "catalogue"])
def test_argument_validation_needs_no_device(which):
    calls, fake = _calls()
    call = dict(calls)[which]
    ks = (ctypes.c_int32 * 9)(*([10] * 9))
    good = dict(U=4, N=100, nnz=8, ks=ks, n_ks=1, rowptr=fake, tpos=fake, sums=fake, ws_bytes=256)
    bad = [dict(n_ks=0), dict(n_ks=nat.MR_MAX_CUTOFFS + 1), dict(ks=None), dict(ks=(ctypes.c_int32 * 2)(10, 0), n_ks=2),
           dict(U=-1), dict(U=1 << 31), dict(nnz=-1), dict(nnz=1 << 31), dict(U=0), dict(rowptr=None),
           dict(tpos=None, sums=None)]
    if which == "scores":
        bad.append(dict(N=0))
    for change in bad:
        args = dict(good, **change)
        assert call(**args) == MR_ERR_INVALID, change
        assert "targets" in nat.last_error(), change
    # a workspace below the query is refused before any launch
    assert call(**good) == MR_ERR_WORKSPACE
    assert "workspace" in nat.last_error()


def test_catalogue_call_refuses_a_model_without_parameters():
    fake = ctypes.c_void_p(16)
    ws = (ctypes.c_char * 256)()
    ks = (ctypes.c_int32 * 1)(10)
    m = _model_desc([256, 128, 64], 64, 100, 100)
    assert nat.lib.mr_catalogue_targets(ctypes.byref(m), fake, 4, 0, None, None, fake, fake, 8, ks, 1, fake, fake, ws,
                                        256, None) == MR_ERR_INVALID
