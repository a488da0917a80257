"""Ragged-list top-k: the NumPy reference against the RankLayer rule, and the C ABI's host-side surface (workspace
queries, argument refusals) of mr_topk_lists / mr_rank_lists.  CPU only."""

import ctypes

import numpy as np

from lists_oracle import csr, topk_lists
from movierec import _native as nat
from oracle import movierec_oracle as o

MR_ERR_INVALID, MR_ERR_WORKSPACE = -1, -2


def test_oracle_matches_rank_groups_and_label_col_rule_on_uniform_lists():
    rng = np.random.default_rng(0)
    for group in (1, 2, 7, 100):
        G = 13
        p = rng.choice(np.float32([0.1, 0.5, 0.5, 0.9, np.nan, -0.0, 0.0, np.inf, -np.inf]), G * group)
        rowptr = np.arange(G + 1, dtype=np.int64) * group
        top, scores, _, _ = topk_lists(p, rowptr, group)
        np.testing.assert_array_equal(top, o.rank_groups(p, group))
        np.testing.assert_array_equal(scores.view(np.int32),
                                      p.reshape(G, group)[np.arange(G)[:, None], top].view(np.int32))
        # pos = mr_rank_scores' position of label_col: the place of the target in the full permutation
        t = rng.integers(0, group, G)
        _, _, pos, sums = topk_lists(p, rowptr, 10, targets=t)
        want = np.array([int(np.flatnonzero(o.rank_groups(p, group)[g] == t[g])[0]) for g in range(G)])
        np.testing.assert_array_equal(pos, want)
        assert sums == o.metrics_from_positions(want, 10)
        # the target last: mr_rank_eval's rule, where the positive loses ties
        key = np.where(np.isnan(p), -np.inf, p).reshape(G, group)
        _, _, pos, _ = topk_lists(p, rowptr, 10, targets=np.full(G, group - 1))
        np.testing.assert_array_equal(pos, (key[:, :-1] >= key[:, -1:]).sum(axis=1))


def test_oracle_known_cases():
    nan = np.float32(np.nan)
    # ties by position, NaN last, -0 == +0; a duplicated item is two candidates
    rowptr, _ = csr([[0] * 7, [], [5], [3, 3, 4]])
    p = np.float32([0.5, 0.9, 0.5, nan, 0.0, -0.0, 0.9, 0.2, 0.7, 0.7, 0.1])
    top, scores, pos, sums = topk_lists(p, rowptr, 4, targets=[2, 0, 0, 1])
    assert top[0].tolist() == [1, 6, 0, 2]
    assert top[1].tolist() == [-1] * 4 and np.isnan(scores[1]).all()  # an empty list
    assert top[2].tolist() == [0, -1, -1, -1] and scores[2, 0] == np.float32(0.2)  # k larger than the list
    assert top[3].tolist() == [0, 1, 2, -1]  # equal copies: the earlier one first
    assert pos.tolist() == [3, 0, 0, 1]  # an empty list's target is outside it: pos = len = 0
    full, _, _, _ = topk_lists(p, rowptr, 7)
    assert full[0].tolist() == [1, 6, 0, 2, 4, 5, 3]
    # targets outside the list and out-of-range users
    _, _, pos, _ = topk_lists(p, rowptr, 4, targets=[-1, 0, 1, 3])
    assert pos.tolist() == [7, 0, 1, 3]
    top, scores, pos, _ = topk_lists(p, rowptr, 2, targets=[0, 0, 0, 0], bad_lists=[True, False, False, True])
    assert top[0].tolist() == [-1, -1] and np.isnan(scores[3]).all() and pos.tolist() == [7, 0, 0, 3]


def _model_desc(layers, mf_dim, num_users, num_items, base=None):
    """A model description; with `base` its parameter pointers are fake addresses laid out as the dense block
    requires (never dereferenced by the host-side checks)."""
    m = nat.MrModel()
    m.n_layers, m.mf_dim, m.num_users, m.num_items = len(layers), mf_dim, num_users, num_items
    for i, w in enumerate(layers):
        m.L[i] = w
    if base is not None:
        m.user_mlp, m.item_mlp, m.dense = base, base + (1 << 24), base + (1 << 26)
        if mf_dim:
            m.user_gmf, m.item_gmf = base + (1 << 28), base + (1 << 30)
        off = 0
        for i in range(1, len(layers)):
            m.W[i] = m.dense + 4 * off
            off += layers[i - 1] * layers[i]
            m.b[i] = m.dense + 4 * off
            off += layers[i]
        m.w_out = m.dense + 4 * off
        off += mf_dim + layers[-1]
        m.b_out = m.dense + 4 * off
        m.dense_count = off + 1
    return m


def test_workspace_queries_host_only_monotone_and_small_for_small_calls():
    k = 10
    prev = 0
    for nnz in (0, 1, 1000, 1024, 1025, 100003, 1 << 20, 1 << 22, (1 << 22) + 1, 1 << 24):
        w = nat.lib.mr_topk_lists_workspace_bytes(1000, nnz, k)
        assert w >= prev
        prev = w
    assert nat.lib.mr_topk_lists_workspace_bytes(10, 1 << 20, k) <= nat.lib.mr_topk_lists_workspace_bytes(11, 1 << 20, k)
    # staging of the long lists stays below nnz * k / 64 bytes (+ per-list terms and alignment)
    assert nat.lib.mr_topk_lists_workspace_bytes(1, 1 << 24, 256) <= (1 << 24) * 256 // 64 + (1 << 24) // 128 + 4096
    for layers, mf in (([256, 128, 64], 64), ([64, 32, 16, 8], 8), ([6, 4], 0), ([256, 128, 64], 0)):
        m = _model_desc(layers, mf, 138493, 26744)
        prev = 0
        for nnz in (0, 1000, 1 << 20, (1 << 21) + 128, 1 << 22, (1 << 22) + 1, 1 << 24):
            w = nat.lib.mr_rank_lists_workspace_bytes(ctypes.byref(m), 1024, nnz, k)
            assert w >= prev, (layers, nnz)
            prev = w
        prev = 0
        for U in (0, 1, 1024, 138493, 1 << 20):
            w = nat.lib.mr_rank_lists_workspace_bytes(ctypes.byref(m), U, 1 << 20, k)
            assert w >= prev, (layers, U)
            prev = w
        one = nat.lib.mr_rank_lists_workspace_bytes(ctypes.byref(m), 1, 1000, k)
        big = nat.lib.mr_rank_lists_workspace_bytes(ctypes.byref(m), 1, 1 << 22, k)
        assert 0 < one and 3 * one < big, (layers, one, big)  # a serving call: far below a 2^22-row one
    for bad in ((10, 100, 0), (10, 100, nat.MR_MAX_TOPK + 1), (-1, 100, 5), (10, -1, 5)):
        assert nat.lib.mr_topk_lists_workspace_bytes(*bad) == 0
        m = _model_desc([256, 128, 64], 64, 100, 100)
        assert nat.lib.mr_rank_lists_workspace_bytes(ctypes.byref(m), *bad) == 0
    assert nat.lib.mr_rank_lists_workspace_bytes(None, 10, 100, 5) == 0


def test_argument_refusals_need_no_device():
    ws = (ctypes.c_char * 256)()
    fake = ctypes.c_void_p(16)  # never dereferenced: every refusal comes before a launch
    topk = nat.lib.mr_topk_lists
    for U, nnz, k in ((4, 10, 0), (4, 10, nat.MR_MAX_TOPK + 1), (-1, 10, 5), (4, -1, 5), (0, 10, 5)):
        assert topk(fake, U, fake, nnz, k, None, fake, fake, None, None, ws, 256, None) == MR_ERR_INVALID, (U, nnz, k)
        assert "lists" in nat.last_error()
    # pos or sums without targets; a NULL rowptr
    assert topk(fake, 4, fake, 10, 5, None, fake, fake, fake, None, ws, 256, None) == MR_ERR_INVALID
    assert topk(fake, 4, fake, 10, 5, None, fake, fake, None, fake, ws, 256, None) == MR_ERR_INVALID
    assert topk(fake, 4, None, 10, 5, None, fake, fake, None, None, ws, 256, None) == MR_ERR_INVALID
    # a workspace one byte short of the query
    need = nat.lib.mr_topk_lists_workspace_bytes(4, 10, 5)
    assert topk(fake, 4, fake, 10, 5, fake, fake, fake, fake, fake, fake, need - 1, None) == MR_ERR_WORKSPACE
    # mr_rank_lists: a description without parameters first, then the same refusals on a well-formed one
    rank = nat.lib.mr_rank_lists
    m = _model_desc([256, 128, 64], 64, 100, 100)
    assert rank(ctypes.byref(m), fake, 4, fake, fake, 10, 5, None, fake, fake, fake, None, None, None, ws, 256,
                None) == MR_ERR_INVALID
    m = _model_desc([256, 128, 64], 64, 100, 100, base=1 << 32)
    args = lambda k=5, t=None, pos=None, sums=None, ws_bytes=1 << 40: (
        ctypes.byref(m), fake, 4, fake, fake, 10, k, t, fake, fake, fake, pos, sums, None, fake, ws_bytes, None)
    for bad in (dict(k=0), dict(k=nat.MR_MAX_TOPK + 1), dict(pos=fake), dict(sums=fake)):
        assert rank(*args(**bad)) == MR_ERR_INVALID, bad
    need = nat.lib.mr_rank_lists_workspace_bytes(ctypes.byref(m), 4, 10, 5)
    assert need > 0
    assert rank(*args(t=fake, pos=fake, sums=fake, ws_bytes=need - 1)) == MR_ERR_WORKSPACE
    assert "rank_lists workspace" in nat.last_error()
