"""Audiences' host-side surface, CPU only: the NumPy reference against a brute-force statement of the contract (ties,
NaN, +-0, pools, exclusion, clipped positions), the workspace queries, the C ABI's refusals before any device work, and
the Python argument handling that runs before any launch."""

import ctypes
import math

import numpy as np
import pytest

from audience_oracle import audience
from catalogue_oracle import csr
from movierec import _engine
from movierec import _native as nat
from test_catalogue_targets_host import _model_desc

MR_ERR_INVALID, MR_ERR_WORKSPACE = -1, -2


def brute(p, k, users, num_users, lists, targets):
    """The contract, stated directly: per column, sort the candidates by (-score with NaN as -inf, user id)."""
    U, M = p.shape
    out_u = np.full((M, k), -1, np.int32)
    out_s = np.full((M, k), np.nan, np.float32)
    pos = np.zeros(M, np.int32)
    for j in range(M):
        cand = []
        for r in range(U):
            uid = int(users[r])
            if not 0 <= uid < num_users:
                continue
            if uid in lists[j] and uid != targets[j]:
                continue
            s = float(p[r, j])
            cand.append((math.inf if math.isnan(s) else -s, uid, p[r, j]))
        cand.sort(key=lambda c: (c[0], c[1]))  # -0.0 == 0.0 in the comparison
        for i, c in enumerate(cand[:k]):
            out_u[j, i], out_s[j, i] = c[1], c[2]
        order = [c[1] for c in cand]
        pos[j] = order.index(targets[j]) if targets[j] in order and order.index(targets[j]) < k else k
    return out_u, out_s, pos


@pytest.mark.parametrize("seed", range(6))
def test_oracle_against_the_contract(seed):
    rng = np.random.default_rng(seed)
    U, M, k = int(rng.integers(1, 40)), int(rng.integers(1, 12)), int(rng.integers(1, 8))
    vals = np.float32([0.25, 0.5, np.nan, np.inf, -np.inf, -0.0, 0.0, 1.0])
    p = rng.choice(vals, (U, M)).astype(np.float32)  # nearly everything ties
    pooled = seed % 2 == 1
    users = np.sort(rng.choice(np.arange(-3, 3 * U + 3), U, replace=False)) if pooled else np.arange(U)
    num_users = 2 * U if pooled else U
    lists = [sorted(set(rng.choice(3 * U + 3, int(rng.integers(0, U + 1))).tolist())) for _ in range(M)]
    if M > 1:
        lists[1] = sorted(set(int(u) for u in users if u >= 0))  # the whole pool
    targets = rng.integers(-2, 3 * U + 3, M).astype(np.int32)
    targets[0] = users[U // 2]
    if M > 2 and lists[2]:
        targets[2] = lists[2][0]  # a target on its own exclusion list
    rp, ex = csr(lists)
    got = audience(p, k, users=users if pooled else None, num_users=num_users, excl_rowptr=rp, excl_users=ex,
                   targets=targets)
    want = brute(p, k, users, num_users, [set(x) for x in lists], targets)
    np.testing.assert_array_equal(got[0], want[0])
    np.testing.assert_array_equal(got[1].view(np.int32), want[1].view(np.int32))  # the raw bits: NaN and -0 survive
    np.testing.assert_array_equal(got[2], want[2])
    assert got[3][0] == float((want[2] < k).sum())


def test_oracle_exclusion_rows_and_clipped_positions():
    p = np.float32([[0.9, 0.1], [0.8, 0.2], [0.7, 0.3], [0.6, 0.4]])
    rp, ex = csr([[0, 1], [3]])
    # column 0 uses list 1 ({3}), column 1 a row outside the table (nothing excluded)
    u, s, pos, sums = audience(p, 2, excl_rowptr=rp, excl_users=ex, excl_ids=[1, 7], targets=[2, 0])
    assert u.tolist() == [[0, 1], [3, 2]]
    assert pos.tolist() == [2, 2]  # places 2 and 3: both clipped at k
    assert sums == (0.0, 0.0)
    u, _, pos, _ = audience(p, 3, excl_rowptr=rp, excl_users=ex, targets=[0, 1])
    assert u.tolist() == [[0, 2, 3], [2, 1, 0]] and pos.tolist() == [0, 1]  # target 0 listed but never excluded


def test_workspace_queries_need_no_device():
    q = nat.lib.mr_audience_scores_workspace_bytes
    a = q(138493, 26744, 10)
    assert 26744 * 10 * 12 <= a <= 26744 * 10 * 12 + 26744 * 4 + 4096  # one list per item at the full catalogue
    assert q(138493, 26744, 256) > 26744 * 256 * 12
    assert q(10 ** 6, 26744, 10) == a  # bounded in users
    assert q(0, 5, 1) > 0 and q(5, 0, 1) > 0
    for bad in ((-1, 5, 1), (1 << 31, 5, 1), (5, -1, 1), (5, 5, 0), (5, 5, nat.MR_MAX_TOPK + 1)):
        assert q(*bad) == 0, bad
    qm = nat.lib.mr_catalogue_audience_workspace_bytes
    m = _model_desc([256, 128, 64], 64, 138493, 26744, fake_params=True)
    full = qm(ctypes.byref(m), 138493, 26744, 10)
    assert full > a + 156 * 26744 * 8  # + one sweep chunk
    assert qm(ctypes.byref(m), 10 ** 6, 26744, 10) == full
    assert qm(ctypes.byref(m), 138493, 100, 10) > 0
    assert qm(None, 10, 10, 10) == 0 and qm(ctypes.byref(m), 10, 10, 0) == 0 and qm(ctypes.byref(m), -1, 10, 1) == 0


def test_argument_validation_needs_no_device():
    fake = ctypes.c_void_p(16)  # never dereferenced: validation fails first
    ws = (ctypes.c_char * 256)()
    good = dict(scores=fake, U=4, M=3, k=2, users=None, excl_ids=None, excl_rows=0, rowptr=None, excl=None, targets=fake,
                top_users=fake, top_scores=fake, pos=fake, sums=fake, ws=ws, ws_bytes=256)

    def call(**kw):
        a = dict(good, **kw)
        return nat.lib.mr_audience_scores(a["scores"], a["U"], a["M"], a["k"], a["users"], a["excl_ids"],
                                          a["excl_rows"], a["rowptr"], a["excl"], a["targets"], a["top_users"],
                                          a["top_scores"], a["pos"], a["sums"], a["ws"], a["ws_bytes"], None)

    for change in (dict(U=-1), dict(U=1 << 31), dict(M=-1), dict(k=0), dict(k=nat.MR_MAX_TOPK + 1),
                   dict(excl_rows=-1), dict(rowptr=fake), dict(targets=None), dict(scores=None), dict(ws=None)):
        assert call(**change) == MR_ERR_INVALID, change
        assert "audience" in nat.last_error(), change
    assert call(ws_bytes=8) == MR_ERR_WORKSPACE
    m = _model_desc([256, 128, 64], 64, 100, 50, fake_params=True)
    cat = lambda users, U, items, M: nat.lib.mr_catalogue_audience(ctypes.byref(m), items, M, 2, users, U, 0, None, None,
                                                                   None, fake, fake, None, None, None, ws, 256, None)
    assert cat(None, 99, fake, 3) == MR_ERR_INVALID and "num_users" in nat.last_error()  # no pool: U = num_users
    assert cat(fake, 5, None, 3) == MR_ERR_INVALID
    assert cat(None, 100, fake, 3) == MR_ERR_WORKSPACE


def test_pool_and_exclusion_handling():
    assert _engine.audience_pool(None) is None
    np.testing.assert_array_equal(_engine.audience_pool([5, 1, 5, -2, 1]), np.int32([-2, 1, 5]))
    rp, it = _engine.check_exclusion_csr(np.int64([0, 2, 2, 5]), np.int32([1, 4, 0, 3, 9]))
    assert str(rp.dtype) == "torch.int64" and str(it.dtype) == "torch.int32" and it.tolist() == [1, 4, 0, 3, 9]
    _engine.check_exclusion_csr(np.int64([0]), np.int32([]))
    for rowptr, ids in (([], []), ([1, 2], [3, 4]), ([0, 3], [1, 2]), ([0, 2, 1, 3], [1, 2, 3]),
                        ([0, 3], [1, 3, 2]), ([0, 2], [4, 4])):
        with pytest.raises(ValueError):
            _engine.check_exclusion_csr(np.int64(rowptr), np.int32(ids))


def test_check_csr_refuses_each_malformed_case():
    ok = (np.int64([0, 2, 2, 5]), np.int32([1, 4, 0, 3, 9]))
    rp, it = _engine.check_csr(*ok, "lists", rows=3, ascending=True, limit=10)
    assert rp.tolist() == [0, 2, 2, 5] and it.tolist() == [1, 4, 0, 3, 9] and str(it.dtype) == "torch.int32"
    cases = [  # (rowptr, ids, flags, error): the rule each case breaks, under the flag that asks for it
        ([], [], {}, ValueError),  # no offsets at all
        ([1, 2], [3, 4], {}, ValueError),  # does not start at 0
        ([0, 2, 1, 3], [1, 2, 3], {}, ValueError),  # decreases
        ([0, 1], [1, 2], {}, ValueError),  # ends before len(ids)
        ([0, 3], [1, 2], {}, ValueError),  # ends past len(ids): a kernel would read past the ids
        ([0, 2, 5], [1, 4, 0, 3, 9], dict(rows=3), ValueError),  # wrong row count
        ([0, 2, 5], [1, 4, 0, 3, 9], dict(rows=1), ValueError),
        ([0, 3], [1, 3, 2], dict(ascending=True), ValueError),  # not ascending
        ([0, 2], [4, 4], dict(ascending=True), ValueError),  # not strictly ascending
        ([0, 2], [1, 10], dict(limit=10), IndexError),  # id >= limit
        ([0, 2], [-1, 3], dict(limit=10), IndexError),  # id < 0
    ]
    for rowptr, ids, flags, error in cases:
        with pytest.raises(error):
            _engine.check_csr(np.int64(rowptr), np.int32(ids), "lists", **flags)
    # without their flags, the last four cases pass: lists need not be sorted or in range unless asked
    for rowptr, ids, flags, _ in cases[-4:]:
        _engine.check_csr(np.int64(rowptr), np.int32(ids), "lists")
    # a list may end where the next starts with a smaller id
    _engine.check_csr(np.int64([0, 2, 4]), np.int32([3, 7, 1, 2]), "lists", ascending=True)
