"""Audiences on a B200: mr_audience_scores bit-exact against the NumPy reference on adversarial scores,
mr_catalogue_audience bit-identical to mr_catalogue_topk's probabilities on every tower, independence from the other
items and the pool, the extended catalogue of an item fold-in, and the Python face."""

import numpy as np
import pytest

from audience_oracle import audience
from catalogue_oracle import csr
from oracle import movierec_oracle as o
from test_gpu_catalogue import TOWERS, _engine, close_to_truth

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def eng_mod():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from movierec import _engine as e
    return e


def _np(ts):
    return [t.cpu().numpy() if t is not None else None for t in ts]


def check(got, want):
    users, scores, pos, sums = _np(got[:3]) + [got[3]]
    np.testing.assert_array_equal(users, want[0])
    np.testing.assert_array_equal(scores.view(np.int32), want[1].view(np.int32))
    if want[2] is not None:
        np.testing.assert_array_equal(pos, want[2])
        s = sums.cpu().numpy().astype(np.float64)
        assert s[0] == want[3][0]
        assert abs(s[1] - want[3][1]) <= 1e-6 * max(abs(want[3][1]), 1.0)


@pytest.mark.parametrize("M", [1, 31, 32, 1000, 26744])
def test_audience_scores_bit_exact_on_adversarial_scores(eng_mod, M):
    rng = np.random.default_rng(M)
    chunk = max(1, min((1 << 22) // M, 16384))
    U = 2 * chunk + 5  # crosses two chunk boundaries
    vals = np.float32([0.25, 0.5, 0.5, 0.75, np.nan, np.inf, -np.inf, -0.0, 0.0, 1.0])
    p = np.where(rng.random((U, M)) < 0.5, rng.choice(vals, (U, M)),
                 rng.integers(0, 64, (U, M)).astype(np.float32) / 64).astype(np.float32)  # many exact ties
    for pooled in (False, True):
        users = np.sort(rng.choice(3 * U, U, replace=False)).astype(np.int32) - 3 if pooled else None
        ids = users if pooled else np.arange(U, dtype=np.int32)
        space = int(ids[-1]) + 4
        rows = 7
        lists = [sorted(rng.choice(space, int(rng.integers(0, min(space, 400))), replace=False).tolist())
                 for _ in range(rows)]
        lists[2] = [int(u) for u in ids if u >= 0]  # the whole pool
        rp, ex = csr(lists)
        excl_ids = rng.integers(-1, rows + 2, M).astype(np.int32)  # rows outside the table
        excl_ids[: max(1, M // 8)] = 2
        targets = rng.choice(ids, M).astype(np.int32)
        targets[rng.random(M) < 0.2] = -1
        off = rng.random(M) < 0.2
        targets[off] = space + 5  # outside the pool
        for j in range(min(M, 5)):  # targets on their own exclusion list
            r = excl_ids[j]
            if 0 <= r < rows and lists[r]:
                targets[j] = lists[r][0]
        for k in (1, 10, 256):
            got = eng_mod.audience_scores(p, k, users=users, exclude=(rp, ex), excl_ids=excl_ids, targets=targets)
            check(got, audience(p, k, users=users, excl_rowptr=rp, excl_users=ex, excl_ids=excl_ids, targets=targets))
    u, s, pos, sums = eng_mod.audience_scores(p, 10)
    np.testing.assert_array_equal(u.cpu().numpy(), audience(p, 10)[0])
    assert pos is None and sums is None


def _raters(rng, nu, ni):
    return csr([sorted(rng.choice(nu, int(rng.integers(0, 60)), replace=False).tolist()) for _ in range(ni)])


@pytest.mark.parametrize("layers,mf", TOWERS, ids=["tc-gmf64", "tc-nogmf", "default-tower", "simt"])
def test_catalogue_audience_against_catalogue_topk(eng_mod, layers, mf):
    ni = 1000
    nu = 2 * ((1 << 22) // ni) + 7  # two chunk boundaries
    eng = _engine(eng_mod, layers, mf, nu, ni)
    rng = np.random.default_rng(3)
    rp, ex = _raters(rng, nu, ni)
    items = np.arange(ni, dtype=np.int32)
    targets = rng.integers(0, nu, ni).astype(np.int32)
    targets[:5] = [ex[rp[j]] if rp[j + 1] > rp[j] else 0 for j in range(5)]  # on their own lists
    _, _, _, _, full = eng.catalogue_topk(np.arange(nu, dtype=np.int32), 10, want_scores=True)
    F = full.cpu().numpy()
    for k in (1, 10):
        top, sc, pos, sums, mat, pool = eng.catalogue_audience(items, k, exclude=(rp, ex), targets=targets,
                                                              want_scores=True)
        assert pool is None
        np.testing.assert_array_equal(mat.cpu().numpy().view(np.int32), F.view(np.int32))
        check((top, sc, pos, sums), audience(F, k, num_users=nu, excl_rowptr=rp, excl_users=ex, targets=targets))
    assert float(eng.last_catalogue_bad.item()) == 0.0
    sample = rng.choice(nu, 12, replace=False)
    w = eng.get_weights()
    w64 = {key: np.asarray(v, np.float64) for key, v in w.items()}
    uu, ii = np.repeat(sample, ni), np.tile(items, sample.size)
    close_to_truth(F[sample].reshape(-1), o.forward(w, uu, ii)["p"], o.forward(w64, uu, ii)["p"],
                   "audience probabilities {} / {}".format(layers, mf))


@pytest.mark.parametrize("layers,mf", [TOWERS[0], TOWERS[2]], ids=["tc-gmf64", "default-tower"])
def test_independent_of_the_other_items_and_the_pool(eng_mod, layers, mf):
    nu, ni, k = 9000, 300, 10
    eng = _engine(eng_mod, layers, mf, nu, ni)
    rng = np.random.default_rng(9)
    rp, ex = _raters(rng, nu, ni)
    allu, alls, _, _, _, _ = _np(eng.catalogue_audience(np.arange(ni), k, exclude=(rp, ex)))
    for sub in (np.int32([7]), rng.integers(0, ni, 31).astype(np.int32), np.int32([5, 5, 299, 0, 5]),
                rng.permutation(ni).astype(np.int32)):
        u, s, _, _, _, _ = _np(eng.catalogue_audience(sub, k, exclude=(rp, ex)))
        np.testing.assert_array_equal(u, allu[sub])
        np.testing.assert_array_equal(s.view(np.int32), alls[sub].view(np.int32))
    # an ascending pool subset (given unsorted, with duplicates and ids outside the users) = the restricted matrix
    pool = np.sort(rng.choice(nu, 4000, replace=False)).astype(np.int32)
    given = np.concatenate([rng.permutation(pool), pool[:50], np.int32([-4, nu, nu + 3])])
    items = rng.integers(0, ni, 40).astype(np.int32)
    targets = rng.choice(nu, 40).astype(np.int32)
    got = eng.catalogue_audience(items, k, users=given, exclude=(rp, ex), targets=targets, want_scores=True)
    assert float(eng.last_catalogue_bad.item()) > 0  # the out-of-range pool ids
    _, _, _, _, full = eng.catalogue_topk(np.arange(nu, dtype=np.int32), 10, want_scores=True)
    F = full.cpu().numpy()
    ids = got[5].cpu().numpy()
    np.testing.assert_array_equal(ids, np.unique(given))
    restricted = np.full((ids.size, items.size), np.nan, np.float32)
    valid = (ids >= 0) & (ids < nu)
    restricted[valid] = F[ids[valid]][:, items]
    np.testing.assert_array_equal(got[4].cpu().numpy()[valid].view(np.int32), restricted[valid].view(np.int32))
    check(got[:4], audience(restricted, k, users=ids, num_users=nu, excl_rowptr=rp, excl_users=ex, excl_ids=items,
                            targets=targets))
    again = eng.catalogue_audience(items, k, users=given, exclude=(rp, ex), targets=targets)
    for x, y in zip(got[:4], again[:4]):
        np.testing.assert_array_equal(x.cpu().numpy().view(np.int32), y.cpu().numpy().view(np.int32))
    # out-of-range items: -1 / NaN rows, pos = k
    u, s, pos, _, _, _ = _np(eng.catalogue_audience(np.int32([ni, 3, -1]), k, targets=[0, 1, 2]))
    assert (u[[0, 2]] == -1).all() and np.isnan(s[[0, 2]]).all() and pos[[0, 2]].tolist() == [k, k]
    np.testing.assert_array_equal(u[1], eng.catalogue_audience(np.int32([3]), k)[0][0].cpu().numpy())


def _movierec(tmp_path, nu, ni):
    from movierec.model import MovierecModel
    params = dict(num_users=nu, num_items=ni, layers_sizes=[64, 32, 16, 8], layers_l2reg=[0] * 4, optimizer="adam",
                  lr=0.001, batch_size=10, num_negs_per_pos=4, batch_size_eval=10, num_negs_per_pos_eval=4, k=5,
                  mf_dim=8, seed=1)
    return MovierecModel(params, output_dir=str(tmp_path))


def test_extended_catalogue(eng_mod, tmp_path):
    nu, ni = 500, 40
    mr = _movierec(tmp_path, nu, ni)
    rng = np.random.default_rng(2)
    raters = [np.sort(rng.choice(nu, n, replace=False)) for n in (30, 12, 0)]
    folded = mr.fold_in_items(raters, steps=3)
    new = folded.new_item_ids
    eng = folded.model.engine
    _, _, _, _, full = eng.catalogue_topk(np.arange(nu, dtype=np.int32), 5, want_scores=True)
    F = full.cpu().numpy()[:, new]
    top, sc = folded.audience_for_new_items(top_k=15)
    rp, it = csr(raters)
    want = audience(F, 15, num_users=nu, excl_rowptr=rp, excl_users=it)
    np.testing.assert_array_equal(top, want[0])
    np.testing.assert_array_equal(sc.view(np.int32), want[1].view(np.int32))
    for j, r in enumerate(raters):
        assert not np.isin(top[j], r).any()
    pool = np.arange(0, nu, 3)
    top, _ = folded.audience_for_new_items(top_k=5, users=pool)
    assert np.isin(top, pool).all()


def test_python_face(eng_mod, tmp_path):
    import pandas as pd
    from movierec import data_pipeline as dp
    nu, ni = 300, 60
    mr = _movierec(tmp_path, nu, ni)
    rng = np.random.default_rng(5)
    users = np.repeat(np.arange(nu), 6)
    items = rng.integers(0, ni, users.size)
    df = pd.DataFrame({dp.COL_USER_ID: users, dp.COL_ITEM_ID: items, dp.COL_RATING: 1.0})
    gen = dp.MovieLensDataGenerator("ml-100k", df, 10, 4, seed=1)
    irp, iu = gen.item_user_lists()
    irp, iu = irp.cpu().numpy(), iu.cpu().numpy()
    for j in range(items.max() + 1):
        np.testing.assert_array_equal(iu[irp[j]:irp[j + 1]], np.unique(users[items == j]))
    eng = mr.model.engine
    _, _, _, _, full = eng.catalogue_topk(np.arange(nu, dtype=np.int32), 5, want_scores=True)
    F = full.cpu().numpy()
    q = np.int32([3, 0, 59, 3])
    top, sc = mr.model.audience_for_items(q, top_k=8, exclude=gen)
    want = audience(F[:, q], 8, num_users=nu, excl_rowptr=irp, excl_users=iu, excl_ids=q)
    np.testing.assert_array_equal(top, want[0])
    np.testing.assert_array_equal(sc.view(np.int32), want[1].view(np.int32))
    held = rng.integers(0, nu, 20).astype(np.int32)
    its = rng.integers(0, ni, 20).astype(np.int32)
    hr, ndcg = mr.evaluate_item_audiences(its, held, exclude=gen, k=10)
    pos = audience(F[:, its], 10, num_users=nu, excl_rowptr=irp, excl_users=iu, excl_ids=its, targets=held)[2]
    h, d = o.metrics_from_positions(pos, 10)
    assert hr == h / its.size
    assert abs(ndcg - d / its.size) <= 1e-6 * max(d / its.size, 1e-3)
    with pytest.raises(IndexError):
        mr.model.audience_for_items([ni], top_k=5)
    with pytest.raises(IndexError):
        mr.model.audience_for_items([1], top_k=5, users=[0, nu])
    with pytest.raises(IndexError):
        mr.evaluate_item_audiences([1, 2], [0, nu], k=5)
    with pytest.raises(ValueError):
        mr.model.audience_for_items([1], top_k=5, exclude=(np.int64([0, 2]), np.int32([4, 1])))
    with pytest.raises(ValueError):
        mr.model.audience_for_items([1], top_k=5, exclude=(np.int64([0, 3]), np.int32([1, 4])))
    with pytest.raises(ValueError):
        mr.evaluate_item_audiences([1, 2], [0], k=5)
