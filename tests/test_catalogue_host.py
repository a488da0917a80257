"""Catalogue top-k: the NumPy reference against the RankLayer rule, and the C ABI's host-side surface (workspace
queries, argument validation).  CPU only."""

import ctypes

import numpy as np

from catalogue_oracle import catalogue_topk, csr
from movierec import _native as nat
from oracle import movierec_oracle as o


def test_oracle_matches_rank_groups_without_exclusions():
    rng = np.random.default_rng(0)
    for N in (1, 7, 100):
        p = rng.choice(np.float32([0.1, 0.5, 0.5, 0.9, np.nan, -0.0, 0.0]), N).astype(np.float32).reshape(1, N)
        items, scores, _, _ = catalogue_topk(p, N, None, None)
        np.testing.assert_array_equal(items[0], o.rank_groups(p, N)[0])
        np.testing.assert_array_equal(scores[0], p[0, items[0]])


def test_oracle_known_cases():
    nan = np.float32(np.nan)
    # ties keep the lower id first, NaN ranks last, -0 and +0 tie
    p = np.float32([[0.5, 0.9, 0.5, nan, 0.0, -0.0, 0.9]])
    items, _, _, _ = catalogue_topk(p, 7, None, None)
    assert items[0].tolist() == [1, 6, 0, 2, 4, 5, 3]
    # k larger than the candidates: -1 / NaN padding; exclusion; target ranked even when listed
    rowptr, ex = csr([[1, 2, 6]])
    items, scores, pos, sums = catalogue_topk(p, 6, rowptr, ex, targets=[6])
    assert items[0].tolist() == [6, 0, 4, 5, 3, -1]
    assert np.isnan(scores[0, 4]) and np.isnan(scores[0, 5])
    assert pos.tolist() == [0] and sums[0] == 1.0
    # every item excluded, the target out of range
    rowptr, ex = csr([list(range(7))])
    items, scores, pos, sums = catalogue_topk(p, 3, rowptr, ex, targets=[7])
    assert items[0].tolist() == [-1, -1, -1] and np.isnan(scores).all()
    assert pos.tolist() == [7] and sums == (0.0, 0.0)
    # ids outside [0, N) in a list and rows outside the table exclude nothing; excl_ids picks the list
    rowptr, ex = csr([[-3, 0, 99], [1]])
    items, _, pos, _ = catalogue_topk(np.vstack([p, p, p]), 2, rowptr, ex, excl_ids=[1, 0, 5], targets=[0, 0, 0])
    assert items.tolist() == [[6, 0], [1, 6], [1, 6]]
    assert pos.tolist() == [1, 2, 2]  # (row 1 excludes item 0, but the target is never excluded)


def _model_desc(layers, mf_dim, num_users, num_items):
    m = nat.MrModel()
    m.n_layers, m.mf_dim, m.num_users, m.num_items = len(layers), mf_dim, num_users, num_items
    for i, w in enumerate(layers):
        m.L[i] = w
    return m


def test_workspace_queries_are_host_only_and_bounded_in_users():
    # one chunk holds about 2^22 rows: beyond that, more users cost no more workspace
    N, k = 26744, 10
    chunk = (1 << 22) // N
    a = nat.lib.mr_topk_scores_workspace_bytes(chunk, N, k)
    assert 0 < nat.lib.mr_topk_scores_workspace_bytes(1, N, k) <= a
    assert nat.lib.mr_topk_scores_workspace_bytes(10 * chunk, N, k) == a
    assert nat.lib.mr_topk_scores_workspace_bytes(138493, N, k) == a
    for layers, mf in (([256, 128, 64], 64), ([64, 32, 16, 8], 8), ([6, 4], 0)):
        m = _model_desc(layers, mf, 138493, N)
        one = nat.lib.mr_catalogue_topk_workspace_bytes(ctypes.byref(m), chunk, k)
        assert one >= chunk * N * 8  # item ids and probabilities of a chunk
        assert nat.lib.mr_catalogue_topk_workspace_bytes(ctypes.byref(m), 138493, k) == one
        assert nat.lib.mr_catalogue_topk_workspace_bytes(ctypes.byref(m), 1, k) < one
    for bad_k in (0, nat.MR_MAX_TOPK + 1):
        assert nat.lib.mr_topk_scores_workspace_bytes(10, N, bad_k) == 0
    assert nat.lib.mr_topk_scores_workspace_bytes(10, 0, k) == 0


def test_argument_validation_needs_no_device():
    MR_ERR_INVALID = -1
    ws = (ctypes.c_char * 256)()
    fake = ctypes.c_void_p(16)  # never dereferenced: validation fails first
    for U, N, k in ((4, 10, 0), (4, 10, nat.MR_MAX_TOPK + 1), (4, 0, 5)):
        rc = nat.lib.mr_topk_scores(fake, U, N, k, None, 0, None, None, None, fake, fake, None, None, ws, 256, None)
        assert rc == MR_ERR_INVALID, (U, N, k)
        assert "topk" in nat.last_error()
    # positions need targets
    rc = nat.lib.mr_topk_scores(fake, 4, 10, 5, None, 0, None, None, None, None, None, fake, None, ws, 256, None)
    assert rc == MR_ERR_INVALID
    # a model description without parameters is refused before anything else
    m = _model_desc([256, 128, 64], 64, 100, 100)
    rc = nat.lib.mr_catalogue_topk(ctypes.byref(m), fake, 4, 10, 0, None, None, None, fake, fake, None, None, None, ws,
                                   256, None)
    assert rc == MR_ERR_INVALID
