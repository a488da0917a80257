"""Large k (kTopkSmallK = 256 < k <= MR_MAX_TOPK = 4096): the C ABI's host-side surface of every call that takes k --
the bound, the workspace queries of both paths, and the audience workspace formula.  CPU only."""

import ctypes

from movierec import _native as nat
from test_catalogue_targets_host import _model_desc

MR_ERR_INVALID, MR_ERR_WORKSPACE = -1, -2
L = nat.lib
ML20M = dict(U=138493, N=26744)


def _models():
    return (_model_desc([256, 128, 64], 64, 138493, 26744, fake_params=True),
            _model_desc([64, 32, 16, 8], 8, 6040, 3706, fake_params=True))


def test_bound_is_4096():
    assert nat.MR_MAX_TOPK == 4096
    assert nat.version() >= 106


def test_every_workspace_query_takes_4096_and_refuses_4097():
    m, _ = _models()
    queries = (
        lambda k: L.mr_topk_scores_workspace_bytes(100, 3706, k),
        lambda k: L.mr_catalogue_topk_workspace_bytes(ctypes.byref(m), 100, k),
        lambda k: L.mr_topk_lists_workspace_bytes(100, 5000, k),
        lambda k: L.mr_rank_lists_workspace_bytes(ctypes.byref(m), 100, 5000, k),
        lambda k: L.mr_audience_scores_workspace_bytes(100, 50, k),
        lambda k: L.mr_catalogue_audience_workspace_bytes(ctypes.byref(m), 100, 50, k),
    )
    for i, q in enumerate(queries):
        assert q(257) > 0 and q(1000) > 0 and q(4096) > 0, i
        assert q(4097) == 0 and q(1 << 20) == 0, i


def test_every_call_takes_4096_and_refuses_4097():
    # k = 4096 passes validation and stops at the (too small) workspace; 4097 is refused first.  No launch either way.
    fake = ctypes.c_void_p(16)
    ws = (ctypes.c_char * 256)()
    m, _ = _models()
    mm = _model_desc([256, 128, 64], 64, 100, 50, fake_params=True)
    calls = {
        "topk": lambda k: L.mr_topk_scores(fake, 4, 10, k, None, 0, None, None, None, fake, fake, None, None, ws, 256,
                                           None),
        "catalogue_topk": lambda k: L.mr_catalogue_topk(ctypes.byref(m), fake, 4, k, 0, None, None, None, fake, fake,
                                                        None, None, None, ws, 256, None),
        "lists": lambda k: L.mr_topk_lists(fake, 4, fake, 10, k, None, fake, fake, None, None, ws, 8, None),
        "rank_lists": lambda k: L.mr_rank_lists(ctypes.byref(m), fake, 4, fake, fake, 10, k, None, fake, fake, fake,
                                                None, None, None, ws, 256, None),
        "audience_scores": lambda k: L.mr_audience_scores(fake, 4, 3, k, None, None, 0, None, None, None, fake, fake,
                                                          None, None, ws, 256, None),
        "catalogue_audience": lambda k: L.mr_catalogue_audience(ctypes.byref(mm), fake, 3, k, None, 100, 0, None, None,
                                                                None, fake, fake, None, None, None, ws, 256, None),
    }
    for name, call in calls.items():
        assert call(4096) == MR_ERR_WORKSPACE, (name, nat.last_error())
        assert call(257) == MR_ERR_WORKSPACE, (name, nat.last_error())
        assert call(4097) == MR_ERR_INVALID, name
        assert "4096" in nat.last_error(), (name, nat.last_error())


def test_small_k_workspace_sizes_are_unchanged():
    # values of the same queries at the commit before the large-k path (k <= 256 keeps its path and its sizes)
    m, m1 = _models()
    assert [L.mr_topk_scores_workspace_bytes(U, N, k) for U, N, k in
            ((138493, 26744, 10), (5, 3706, 256), (1, 7, 1))] == [354304, 41472, 768]
    assert [L.mr_catalogue_topk_workspace_bytes(ctypes.byref(d), U, k) for d, U, k in
            ((m, 138493, 10), (m, 138493, 256), (m1, 6040, 100))] == [64520704, 72809728, 38417408]
    assert [L.mr_topk_lists_workspace_bytes(U, nnz, k) for U, nnz, k in
            ((1024, 5120000, 256), (3, 10, 1), (1000, 100000, 50))] == [20532992, 1280, 92160]
    assert [L.mr_rank_lists_workspace_bytes(ctypes.byref(m), U, nnz, k) for U, nnz, k in
            ((1024, 5120000, 256), (3, 10, 1))] == [92815360, 14024704]
    assert [L.mr_audience_scores_workspace_bytes(U, M, k) for U, M, k in
            ((138493, 26744, 10), (138493, 26744, 256), (138493, 100, 256), (7, 1, 1))] == [3316736, 82264832, 9831168,
                                                                                            1024]
    assert [L.mr_catalogue_audience_workspace_bytes(ctypes.byref(d), U, M, k) for d, U, M, k in
            ((m, 138493, 26744, 10), (m, 138493, 100, 256), (m1, 6040, 3706, 20))] == [67483904, 51967488, 41914880]


def test_large_k_row_workspace_is_one_chunk_of_staged_keys():
    U, N = ML20M["U"], ML20M["N"]
    chunk = (1 << 22) // N
    for k in (257, 1000, 4096):
        one = L.mr_topk_scores_workspace_bytes(chunk, N, k)
        assert chunk * N * 8 <= one <= chunk * N * 8 + 1024  # 8 bytes per row of a chunk, whatever k is
        assert L.mr_topk_scores_workspace_bytes(U, N, k) == one
        assert L.mr_topk_scores_workspace_bytes(10 ** 7, N, k) == one
        assert L.mr_topk_scores_workspace_bytes(1, N, k) < one
    m, _ = _models()
    for k in (257, 4096):
        full = L.mr_catalogue_topk_workspace_bytes(ctypes.byref(m), U, k)
        assert L.mr_catalogue_topk_workspace_bytes(ctypes.byref(m), 10 ** 7, k) == full
        assert full >= chunk * N * 16  # staged keys + the sweep's item ids and probabilities


def test_large_k_list_workspace_is_the_positions_only():
    for U, nnz in ((1024, 5_120_000), (1, 1), (100_000, 10 ** 8)):
        w = L.mr_topk_lists_workspace_bytes(U, nnz, 1000)
        assert U * 4 <= w <= U * 4 + 512
        assert L.mr_topk_lists_workspace_bytes(U, nnz, 4096) == w


def _audience_formula(U, M, k):
    C = max(1, min(U, max(1, min((1 << 22) // max(M, 1), 16384))))
    return 12 * max(M, 1) * (2 * k + C) + 8 * max(M, 1)


def test_audience_workspace_follows_the_documented_formula():
    q = L.mr_audience_scores_workspace_bytes
    for U, M, k in ((138493, 26744, 1000), (138493, 26744, 4096), (138493, 100, 1000), (6040, 3706, 257),
                    (5, 1, 300), (0, 7, 4096)):
        f = _audience_formula(U, M, k)
        assert f <= q(U, M, k) <= f + 7 * 256, (U, M, k)
    assert abs(q(138493, 26744, 1000) / 1e9 - 0.69) < 0.01  # C = 156
    assert abs(q(138493, 26744, 4096) / 1e9 - 2.68) < 0.01
    assert abs(q(138493, 100, 1000) / 1e6 - 22.1) < 0.2  # C = 16,384
    for k in (257, 1000, 4096):  # bounded in users by one chunk
        assert q(10 ** 9 // 1000, 26744, k) == q(138493, 26744, k)
        assert q(10 ** 6, 100, k) == q(138493, 100, k)
    m, _ = _models()
    sel = q(138493, 26744, 1000)
    full = L.mr_catalogue_audience_workspace_bytes(ctypes.byref(m), 138493, 26744, 1000)
    assert full > sel + 156 * 26744 * 8  # + one sweep chunk
