"""Large k on a B200 (256 < k <= 4096, the radix-select path): mr_topk_scores, mr_topk_lists and mr_audience_scores
bit-exact against the NumPy references on adversarial scores, the k <= 256 path as a prefix of the large-k result,
determinism and independence from the rest of a call, and the Python face at large k."""

import numpy as np
import pytest

from movierec.model import _audience_lists, _exclusion_lists

from audience_oracle import audience
from catalogue_oracle import catalogue_topk, csr
from lists_oracle import topk_lists
from oracle import movierec_oracle as o
from test_gpu_audience import _movierec, _raters, check as check_audience
from test_gpu_catalogue import TOWERS, _engine, check_against_oracle, random_lists
from test_gpu_rank_lists import _facade, adversarial, check_selection

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

KS = (257, 1000, 4096)


@pytest.fixture(scope="module")
def eng_mod():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from movierec import _engine as e
    return e


def _bits(ts):
    return [t.cpu().numpy().view(np.int32) if t is not None else None for t in ts]


def _same(a, b):
    for x, y in zip(_bits(a), _bits(b)):
        if x is not None:
            np.testing.assert_array_equal(x, y)


CONST_ROWS, NAN_ROW = (12, 13), 14  # nothing excluded on these rows (after the fully excluded rows 0-3)


def _adversarial_rows(rng, U, N):
    p = adversarial(rng, U * N).reshape(U, N)
    p[CONST_ROWS[0]] = 0.5  # constant rows: the select runs into the id bits
    p[CONST_ROWS[1]] = -0.0
    p[NAN_ROW] = np.nan  # all NaN
    return p


@pytest.mark.parametrize("N", [1, 1000, 5000, 26744])
def test_topk_scores_bit_exact(eng_mod, N):
    rng = np.random.default_rng(N)
    chunk = max(1, min((1 << 22) // N, 16384))
    U = 2 * chunk + 5 if N >= 26744 else 40  # two chunk boundaries at the large catalogue
    p = _adversarial_rows(rng, U, N)
    rows = 9
    rowptr, ex = random_lists(rng, rows, N, full_rows=(3,))
    excl_ids = rng.integers(-1, rows + 2, U).astype(np.int32)
    excl_ids[:4] = 3  # every item excluded
    excl_ids[list(CONST_ROWS) + [NAN_ROW]] = -1  # every item a candidate
    targets = rng.integers(-1, N + 1, U).astype(np.int32)
    for u in range(6, 12):  # targets on their own exclusion list
        r = excl_ids[u]
        if 0 <= r < rows and rowptr[r + 1] > rowptr[r]:
            targets[u] = ex[rowptr[r]]
    for k in KS:
        got = eng_mod.topk_scores(p, k, exclude=(rowptr, ex), excl_ids=excl_ids, targets=targets)
        check_against_oracle(got, catalogue_topk(p, k, rowptr, ex, excl_ids=excl_ids, targets=targets), k)
        _same(got, eng_mod.topk_scores(p, k, exclude=(rowptr, ex), excl_ids=excl_ids, targets=targets))
    # the k <= 256 path is a prefix of the large-k result: ids, score bits and pos
    small = eng_mod.topk_scores(p, 256, exclude=(rowptr, ex), excl_ids=excl_ids, targets=targets)
    large = eng_mod.topk_scores(p, 1000, exclude=(rowptr, ex), excl_ids=excl_ids, targets=targets)
    np.testing.assert_array_equal(large[0].cpu().numpy()[:, :256], small[0].cpu().numpy())
    np.testing.assert_array_equal(large[1].cpu().numpy()[:, :256].view(np.int32), small[1].cpu().numpy().view(np.int32))
    np.testing.assert_array_equal(large[2].cpu().numpy(), small[2].cpu().numpy())
    # a row's result does not depend on the other rows of the call
    sub = np.int64([U - 1, 0, NAN_ROW, CONST_ROWS[0]])
    part = eng_mod.topk_scores(p[sub], 1000, exclude=(rowptr, ex), excl_ids=excl_ids[sub], targets=targets[sub])
    np.testing.assert_array_equal(part[0].cpu().numpy(), large[0].cpu().numpy()[sub])
    np.testing.assert_array_equal(part[2].cpu().numpy(), large[2].cpu().numpy()[sub])


def test_topk_lists_bit_exact(eng_mod):
    rng = np.random.default_rng(4)
    lens = np.array([0, 1, 256, 257, 1024, 1025, 5000, 30000, 4096, 4097, 999, 1000, 1001] * 2, np.int64)
    lens = rng.permutation(lens)
    rowptr = np.zeros(lens.size + 1, np.int64)
    rowptr[1:] = np.cumsum(lens)
    p = adversarial(rng, int(rowptr[-1]))
    big = np.flatnonzero(lens == 30000)
    p[rowptr[big[0]]:rowptr[big[0] + 1]] = 0.25  # a constant list
    p[rowptr[big[1]]:rowptr[big[1] + 1]] = np.nan  # an all-NaN list
    U = lens.size
    kind = np.arange(U) % 5  # first, middle, last, -1, len
    targets = np.where(kind == 0, 0, np.where(kind == 1, lens // 2, np.where(kind == 2, lens - 1,
                                                                              np.where(kind == 3, -1, lens))))
    targets = targets.astype(np.int32)
    for k in KS:
        got = eng_mod.topk_lists(p, rowptr, k, targets=targets)
        check_selection(got, topk_lists(p, rowptr, k, targets=targets))
        _same(got, eng_mod.topk_lists(p, rowptr, k, targets=targets))
    small = eng_mod.topk_lists(p, rowptr, 256, targets=targets)
    large = eng_mod.topk_lists(p, rowptr, 1000, targets=targets)
    np.testing.assert_array_equal(large[0].cpu().numpy()[:, :256], small[0].cpu().numpy())
    np.testing.assert_array_equal(large[1].cpu().numpy()[:, :256].view(np.int32), small[1].cpu().numpy().view(np.int32))
    np.testing.assert_array_equal(large[2].cpu().numpy(), small[2].cpu().numpy())


def _audience_case(rng, U, M, pooled):
    p = adversarial(rng, U * M).reshape(U, M)
    p[:, 0] = 0.5  # a constant column
    if M > 2:
        p[:, 2] = np.nan  # an all-NaN column
    users = np.sort(rng.choice(3 * U, U, replace=False)).astype(np.int32) - 3 if pooled else None
    ids = users if pooled else np.arange(U, dtype=np.int32)
    space = int(ids[-1]) + 4
    rows = 7
    lists = [sorted(rng.choice(space, int(rng.integers(0, min(space, 400))), replace=False).tolist())
             for _ in range(rows)]
    lists[2] = [int(u) for u in ids if u >= 0]  # the whole pool
    rp, ex = csr(lists)
    excl_ids = rng.integers(-1, rows + 2, M).astype(np.int32)
    excl_ids[0] = -1  # the constant column and the all-NaN column: every pool user a candidate
    if M > 2:
        excl_ids[2] = -1
    if M > 1:
        excl_ids[1] = 2  # every pool user excluded
    targets = rng.choice(ids, M).astype(np.int32)
    targets[rng.random(M) < 0.2] = -1
    targets[rng.random(M) < 0.2] = space + 5  # outside the pool
    for j in range(min(M, 5)):  # on their own exclusion list
        r = excl_ids[j]
        if 0 <= r < rows and lists[r]:
            targets[j] = lists[r][0]
    return p, users, (rp, ex), excl_ids, targets


@pytest.mark.parametrize("M,chunks", [(1, 2), (1000, 8), (26744, 2)])
def test_audience_scores_bit_exact(eng_mod, M, chunks):
    # M = 1000 crosses 8 chunk boundaries: buffers fill by atomics and compact several times per item at k = 257
    rng = np.random.default_rng(M)
    chunk = max(1, min((1 << 22) // M, 16384))
    U = chunks * chunk + 5
    for pooled in (False, True):
        p, users, (rp, ex), excl_ids, targets = _audience_case(rng, U, M, pooled)
        for k in KS if M < 26744 else (257, 1000):
            kw = dict(users=users, exclude=(rp, ex), excl_ids=excl_ids, targets=targets)
            got = eng_mod.audience_scores(p, k, **kw)
            check_audience(got, audience(p, k, users=users, excl_rowptr=rp, excl_users=ex, excl_ids=excl_ids,
                                         targets=targets))
            _same(got, eng_mod.audience_scores(p, k, **kw))
        small = eng_mod.audience_scores(p, 256, **kw)
        large = eng_mod.audience_scores(p, 1000, **kw)
        np.testing.assert_array_equal(large[0].cpu().numpy()[:, :256], small[0].cpu().numpy())
        np.testing.assert_array_equal(large[1].cpu().numpy()[:, :256].view(np.int32),
                                      small[1].cpu().numpy().view(np.int32))
        np.testing.assert_array_equal(np.minimum(large[2].cpu().numpy(), 256), small[2].cpu().numpy())
        # an item's audience does not depend on the other items of the call
        if M > 1:
            sub = np.int64([M - 1, 0, 2])
            part = eng_mod.audience_scores(np.ascontiguousarray(p[:, sub]), 1000, users=users, exclude=(rp, ex),
                                           excl_ids=excl_ids[sub], targets=targets[sub])
            np.testing.assert_array_equal(part[0].cpu().numpy(), large[0].cpu().numpy()[sub])
            np.testing.assert_array_equal(part[2].cpu().numpy(), large[2].cpu().numpy()[sub])


@pytest.mark.parametrize("layers,mf", TOWERS, ids=["tc-gmf64", "tc-nogmf", "default-tower", "simt"])
def test_catalogue_calls_start_with_their_small_k_results(eng_mod, layers, mf):
    nu, ni = 5000, 1200
    eng = _engine(eng_mod, layers, mf, nu, ni)
    rng = np.random.default_rng(7)
    users = rng.integers(0, nu, 300).astype(np.int32)
    rowptr, ex = random_lists(rng, nu, ni)
    targets = rng.integers(0, ni, users.size).astype(np.int32)
    s = eng.catalogue_topk(users, 10, exclude=(rowptr, ex), targets=targets)
    big = eng.catalogue_topk(users, 1000, exclude=(rowptr, ex), targets=targets, want_scores=True)
    np.testing.assert_array_equal(big[0].cpu().numpy()[:, :10], s[0].cpu().numpy())
    np.testing.assert_array_equal(big[1].cpu().numpy()[:, :10].view(np.int32), s[1].cpu().numpy().view(np.int32))
    np.testing.assert_array_equal(big[2].cpu().numpy(), s[2].cpu().numpy())
    check_against_oracle(big[:4], catalogue_topk(big[4].cpu().numpy(), 1000, rowptr, ex, excl_ids=users,
                                                 targets=targets), 1000)
    rp, rx = _raters(rng, nu, ni)
    items = rng.integers(0, ni, 64).astype(np.int32)
    at = rng.integers(0, nu, items.size).astype(np.int32)
    s = eng.catalogue_audience(items, 10, exclude=(rp, rx), targets=at)
    big = eng.catalogue_audience(items, 1000, exclude=(rp, rx), targets=at, want_scores=True)
    np.testing.assert_array_equal(big[0].cpu().numpy()[:, :10], s[0].cpu().numpy())
    np.testing.assert_array_equal(big[1].cpu().numpy()[:, :10].view(np.int32), s[1].cpu().numpy().view(np.int32))
    np.testing.assert_array_equal(np.minimum(big[2].cpu().numpy(), 10), s[2].cpu().numpy())
    check_audience(big[:4], audience(big[4].cpu().numpy(), 1000, num_users=nu, excl_rowptr=rp, excl_users=rx,
                                     excl_ids=items, targets=at))
    # over a pool: the reference on the pool's rows of the same probabilities, twice bit-identical
    pool = np.sort(rng.choice(nu, 3000, replace=False)).astype(np.int32)
    whole = eng.catalogue_audience(items, 2000, users=pool, exclude=(rp, rx))
    check_audience(whole[:2] + (None, None), audience(big[4].cpu().numpy()[pool], 2000, users=pool, num_users=nu,
                                                      excl_rowptr=rp, excl_users=rx, excl_ids=items))
    _same(whole[:2], eng.catalogue_audience(items, 2000, users=pool, exclude=(rp, rx))[:2])


def test_python_face(eng_mod, tmp_path):
    import pandas as pd
    from movierec import data_pipeline as dp
    nu, ni = 3000, 1500
    mr = _movierec(tmp_path, nu, ni)
    rng = np.random.default_rng(5)
    users = np.repeat(np.arange(nu), 6)
    items = rng.integers(0, ni, users.size)
    df = pd.DataFrame({dp.COL_USER_ID: users, dp.COL_ITEM_ID: items, dp.COL_RATING: 1.0})
    gen = dp.MovieLensDataGenerator("ml-100k", df, 10, 4, seed=1)
    eng = mr.model.engine
    q = rng.integers(0, nu, 50).astype(np.int32)
    top, sc = mr.model.recommend_for_users(q, top_k=1000, exclude=gen)
    want = eng.catalogue_topk(q, 1000, exclude=_exclusion_lists(gen))
    np.testing.assert_array_equal(top, want[0].cpu().numpy())
    np.testing.assert_array_equal(sc.view(np.int32), want[1].cpu().numpy().view(np.int32))
    its = np.int32([3, 0, ni - 1, 3])
    top, sc = mr.model.audience_for_items(its, top_k=2000, exclude=gen)
    want = eng.catalogue_audience(its, 2000, exclude=_audience_lists(gen))
    np.testing.assert_array_equal(top, want[0].cpu().numpy())
    np.testing.assert_array_equal(sc.view(np.int32), want[1].cpu().numpy().view(np.int32))
    lists = [rng.integers(0, ni, n) for n in (5, 1000, 1500, 4000)]
    f = _facade(eng)
    bi, bs = f.recommend_batch(np.int32([0, 1, 2, 3]), lists, top_k=1000)
    rp = np.cumsum([0] + [len(x) for x in lists]).astype(np.int64)  # the lists as given: positions break ties
    want = eng.rank_lists(np.int32([0, 1, 2, 3]), (rp, np.concatenate(lists).astype(np.int32)), 1000)
    np.testing.assert_array_equal(bi, want[0].cpu().numpy())
    np.testing.assert_array_equal(bs.view(np.int32), want[1].cpu().numpy().view(np.int32))
    # HR / NDCG at 1000 against the reference on the probabilities the call scores with
    held = rng.integers(0, ni, nu).astype(np.int32)
    allu = np.arange(nu, dtype=np.int32)
    hr, ndcg = mr.evaluate_full_catalogue(allu, held, exclude=gen, k=1000)
    full = eng.catalogue_topk(allu, 5, exclude=_exclusion_lists(gen), want_scores=True)[4].cpu().numpy()
    erp, eit = [x.cpu().numpy() for x in _exclusion_lists(gen)]
    pos = catalogue_topk(full, 1000, erp, eit, targets=held)[2]
    h, d = o.metrics_from_positions(pos, 1000)
    assert hr == h / nu
    assert abs(ndcg - d / nu) <= 1e-6 * max(d / nu, 1e-3)
    # the extended catalogue of an item fold-in
    raters = [np.sort(rng.choice(nu, n, replace=False)) for n in (30, 12, 0)]
    folded = mr.fold_in_items(raters, steps=3)
    fe = folded.model.engine
    F = fe.catalogue_topk(allu, 5, want_scores=True)[4].cpu().numpy()[:, folded.new_item_ids]
    top, sc = folded.audience_for_new_items(top_k=1000)
    rp, it = csr(raters)
    want = audience(F, 1000, num_users=nu, excl_rowptr=rp, excl_users=it)
    np.testing.assert_array_equal(top, want[0])
    np.testing.assert_array_equal(sc.view(np.int32), want[1].view(np.int32))
