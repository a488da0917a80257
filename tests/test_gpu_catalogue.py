"""Catalogue top-k on a B200: mr_topk_scores and mr_catalogue_topk against the NumPy reference (selection
bit-exact, probabilities within the parity tolerance), bit-identity with mr_rank_eval, exclusion, chunking,
determinism and the Python face."""

import copy

import numpy as np
import pandas as pd
import pytest

from catalogue_oracle import catalogue_topk, csr
from oracle import movierec_oracle as o

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

RTOL = 1e-5  # north_star: fp32 logits, probabilities within 1e-5 relative

TOWERS = [  # (layers, mf_dim): fused eval path, tensor cores without GMF, default tower, SIMT tile kernel
    ([256, 128, 64], 64), ([256, 128, 64], 0), ([64, 32, 16, 8], 8), ([6, 4], 0)]


@pytest.fixture(scope="module")
def eng_mod():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from movierec import _engine
    return _engine


def close_to_truth(got, ref32, ref64, what, rtol=RTOL, k=4.0):
    """The kernel against the float64 oracle, calibrated by the float32 oracle's own distance from it (the rule of
    test_gpu_parity.close_to_truth, per tensor and per element, without the slack term)."""
    got = np.asarray(got, np.float64).reshape(-1)
    ref32 = np.asarray(ref32, np.float64).reshape(-1)
    ref64 = np.asarray(ref64, np.float64).reshape(-1)
    scale = max(float(np.max(np.abs(ref64))), 1e-30)
    e32 = float(np.max(np.abs(ref32 - ref64)))
    err = np.abs(got - ref64)
    assert float(err.max()) <= max(k * e32, rtol * scale), "{}: max err {:.3e} (fp32-oracle err {:.3e})".format(
        what, float(err.max()), e32)
    big = np.abs(ref64) > 1e-3 * scale
    excess = err[big] - (rtol * np.abs(ref64[big]) + k * e32)
    assert excess.size == 0 or excess.max() <= 0, "{}: element error {:.3e} over the bound".format(what, excess.max())


def random_lists(rng, rows, N, full_rows=()):
    lists = []
    for r in range(rows):
        if r in full_rows:
            lists.append(list(range(N)))
        else:
            n = int(rng.integers(0, max(1, min(N, 300))))
            lists.append(sorted(rng.choice(N, size=n, replace=False).tolist()))
    return csr(lists)


def check_against_oracle(got, want, k):
    items, scores, pos, sums = got
    w_items, w_scores, w_pos, w_sums = want
    np.testing.assert_array_equal(items.cpu().numpy(), w_items)
    np.testing.assert_array_equal(scores.cpu().numpy(), w_scores)
    if w_pos is not None:
        np.testing.assert_array_equal(pos.cpu().numpy(), w_pos)
        s = sums.cpu().numpy().astype(np.float64)
        assert s[0] == w_sums[0]
        assert abs(s[1] - w_sums[1]) <= 1e-6 * max(abs(w_sums[1]), 1.0)


@pytest.mark.parametrize("N", [1, 31, 32, 1000, 26744, 100003])
def test_topk_scores_bit_exact_on_adversarial_scores(eng_mod, N):
    rng = np.random.default_rng(N)
    chunk = max(1, min((1 << 22) // N, 16384))
    U = min(chunk + 3, 45) if N >= 26744 else 37  # crosses a chunk boundary for the large catalogues
    vals = np.float32([0.25, 0.5, 0.5, 0.75, np.nan, np.inf, -np.inf, -0.0, 0.0, 1.0])
    p = np.where(rng.random((U, N)) < 0.5, rng.choice(vals, (U, N)),
                 rng.integers(0, 64, (U, N)).astype(np.float32) / 64).astype(np.float32)  # many exact ties
    rows = 9
    rowptr, ex = random_lists(rng, rows, N, full_rows=(3,))
    excl_ids = rng.integers(-1, rows + 2, U).astype(np.int32)  # duplicated rows, rows outside the table
    excl_ids[:4] = 3  # users with every item excluded
    targets = rng.integers(-1, N + 1, U).astype(np.int32)
    for k in (1, 10, 100, 256):
        got = eng_mod.topk_scores(p, k, exclude=(rowptr, ex), excl_ids=excl_ids, targets=targets)
        check_against_oracle(got, catalogue_topk(p, k, rowptr, ex, excl_ids=excl_ids, targets=targets), k)
    # without exclusion lists or targets
    items, scores, pos, sums = eng_mod.topk_scores(p, 10)
    w = catalogue_topk(p, 10, None, None)
    np.testing.assert_array_equal(items.cpu().numpy(), w[0])
    assert pos is None and sums is None


def _engine(eng_mod, layers, mf, nu, ni, seed=11, **kw):
    return eng_mod.NeuMFEngine(nu, ni, layers, [0] * len(layers), mf_dim=mf, seed=seed, **kw)


def _truth(eng, users, ni):
    w = eng.get_weights()
    w64 = {k: np.asarray(v, np.float64) for k, v in w.items()}
    uu = np.repeat(np.asarray(users), ni)
    ii = np.tile(np.arange(ni), len(users))
    return o.forward(w, uu, ii)["p"], o.forward(w64, uu, ii)["p"]


@pytest.mark.parametrize("layers,mf,proj", [(L, f, None) for L, f in TOWERS] + [([256, 128, 64], 64, "off")],
                         ids=["tc-gmf64", "tc-nogmf", "default-tower", "simt", "tc-gmf64-unprojected"])
def test_catalogue_against_oracle(eng_mod, layers, mf, proj):
    nu, ni, k = 70, 1000, 10
    eng = _engine(eng_mod, layers, mf, nu, ni, item_projection=proj)
    rng = np.random.default_rng(5)
    users = rng.integers(0, nu, 40).astype(np.int32)
    rowptr, ex = random_lists(rng, nu, ni)
    targets = rng.integers(0, ni, 40).astype(np.int32)
    items, scores, pos, sums, full = eng.catalogue_topk(users, k, exclude=(rowptr, ex), targets=targets, want_scores=True)
    p = full.cpu().numpy()
    want = catalogue_topk(p, k, rowptr, ex, excl_ids=users, targets=targets)
    check_against_oracle((items, scores, pos, sums), want, k)
    p32, p64 = _truth(eng, users, ni)
    close_to_truth(p, p32, p64, "catalogue probabilities {} / {}".format(layers, mf))
    got_items = items.cpu().numpy()
    for u in range(len(users)):  # no returned item is on the user's list (the target is never excluded)
        listed = np.setdiff1d(ex[rowptr[users[u]]:rowptr[users[u] + 1]], [targets[u]])
        assert not np.isin(got_items[u], listed).any()


@pytest.mark.parametrize("layers,mf", [([256, 128, 64], 64), ([64, 32, 16, 8], 8)], ids=["tc-gmf64", "default-tower"])
def test_catalogue_probabilities_equal_rank_eval_bit_for_bit(eng_mod, layers, mf):
    nu, ni, group = 300, 2000, 100
    eng = _engine(eng_mod, layers, mf, nu, ni, item_projection="on")
    rng = np.random.default_rng(8)
    users = rng.integers(0, nu, 64).astype(np.int32)
    cand = rng.integers(0, ni, (64, group)).astype(np.int32)
    _, _, _, probs = eng.rank_eval(torch.from_numpy(users).cuda(), torch.from_numpy(cand.ravel()).cuda(), group, 10,
                                   want_probs=True)
    _, _, _, _, full = eng.catalogue_topk(users, 10, want_scores=True)
    got = full.cpu().numpy()[np.arange(64)[:, None], cand]
    np.testing.assert_array_equal(got.view(np.int32), probs.cpu().numpy().reshape(64, group).view(np.int32))


def test_exclusion_targets_and_recommend(eng_mod):
    nu, ni, K = 50, 1000, 10  # (recommend() ranks at most 1,024 candidates)
    eng = _engine(eng_mod, [256, 128, 64], 64, nu, ni)
    rng = np.random.default_rng(3)
    users = np.arange(nu, dtype=np.int32)
    rowptr, ex = random_lists(rng, nu, ni)
    targets = np.array([ex[rowptr[u]] if rowptr[u + 1] > rowptr[u] else 0 for u in range(nu)], np.int32)  # listed
    items, _, pos, _, full = eng.catalogue_topk(users, K, exclude=(rowptr, ex), targets=targets, want_scores=True)
    w = catalogue_topk(full.cpu().numpy(), K, rowptr, ex, targets=targets)
    np.testing.assert_array_equal(pos.cpu().numpy(), w[2])
    for u in range(nu):
        assert not np.isin(items.cpu().numpy()[u], np.setdiff1d(ex[rowptr[u]:rowptr[u + 1]], [targets[u]])).any()
    # no exclusion: the same top-K as recommend() over every item, where the truth separates the scores
    from movierec import model as mm
    top, _, _, _, _ = eng.catalogue_topk(users, K)
    _, p64 = _truth(eng, users, ni)
    p64 = p64.reshape(nu, ni)
    checked = 0
    for u in range(nu):
        s = np.sort(p64[u])[::-1][:K + 1]
        if np.min(s[:-1] - s[1:]) <= 1e-5:
            continue
        facade = mm.NeuMFModel.__new__(mm.NeuMFModel)
        facade.engine = eng
        rec_items, _ = facade.recommend(int(u), np.arange(ni), K)
        np.testing.assert_array_equal(top.cpu().numpy()[u], rec_items)
        checked += 1
    assert checked >= 5


def test_deterministic_and_chunking_invisible(eng_mod):
    ni = 1000
    chunk = (1 << 22) // ni
    nu = chunk + 2
    for layers, mf in (([256, 128, 64], 64), ([64, 32, 16, 8], 8)):
        eng = _engine(eng_mod, layers, mf, nu, ni)
        rng = np.random.default_rng(1)
        rowptr, ex = random_lists(rng, nu, ni)
        sample = rng.integers(0, chunk - 1, 4).tolist() + [chunk - 1, chunk, chunk + 1]
        singles = {}
        for u in sample:
            it, sc, _, _, _ = eng.catalogue_topk([u], 10, exclude=(rowptr, ex))
            singles[u] = (it.cpu().numpy()[0], sc.cpu().numpy()[0])
        for U in (chunk - 1, chunk, chunk + 1, chunk + 2):
            users = np.arange(U, dtype=np.int32)
            a = eng.catalogue_topk(users, 10, exclude=(rowptr, ex), targets=users % ni)
            b = eng.catalogue_topk(users, 10, exclude=(rowptr, ex), targets=users % ni)
            for x, y in zip(a[:4], b[:4]):
                np.testing.assert_array_equal(x.cpu().numpy().view(np.int32), y.cpu().numpy().view(np.int32))
            for u in sample:
                if u < U:
                    np.testing.assert_array_equal(a[0].cpu().numpy()[u], singles[u][0])
                    np.testing.assert_array_equal(a[1].cpu().numpy()[u].view(np.int32), singles[u][1].view(np.int32))


def _ml100k(tmp_path):
    from movierec import data_pipeline as dp, model as mm
    from movierec.util import movielens_utils as ml
    nu, ni = ml.NUM_USERS["ml-100k"], ml.NUM_ITEMS["ml-100k"]
    rng = np.random.default_rng(4)
    users = np.repeat(np.arange(1, nu, dtype=np.int64), 20)
    items = rng.integers(1, ni, users.size)
    df = pd.DataFrame({dp.COL_USER_ID: users, dp.COL_ITEM_ID: items, dp.COL_RATING: 1.0})
    gen = dp.MovieLensDataGenerator("ml-100k", df, 25, 4, seed=1)
    params = {"num_users": nu, "num_items": ni, "layers_sizes": [64, 32, 16, 8], "layers_l2reg": [0, 0, 0, 0],
              "optimizer": "adam", "lr": 0.001, "batch_size": 25, "num_negs_per_pos": 4, "batch_size_eval": 100,
              "num_negs_per_pos_eval": 99, "k": 5, "mf_dim": 8, "seed": 2}
    return mm.MovierecModel(copy.deepcopy(params), output_dir=str(tmp_path)), gen, nu, ni


def test_evaluate_full_catalogue_through_generator(eng_mod, tmp_path):
    m, gen, nu, ni = _ml100k(tmp_path)
    rng = np.random.default_rng(6)
    users = np.arange(1, nu, dtype=np.int32)
    held = rng.integers(1, ni, users.size).astype(np.int32)
    hr, ndcg = m.evaluate_full_catalogue(users, held, exclude=gen, k=10)
    eng = m.model.engine
    rowptr, lists = gen.user_item_lists()
    _, _, _, _, full = eng.catalogue_topk(users, 10, targets=held, want_scores=True)
    _, _, pos, sums = catalogue_topk(full.cpu().numpy(), 10, rowptr.cpu().numpy(), lists.cpu().numpy(),
                                     excl_ids=users, targets=held)
    assert hr == sums[0] / users.size
    assert abs(ndcg - sums[1] / users.size) <= 1e-6 * max(sums[1] / users.size, 1e-3)
    top, _ = m.model.recommend_for_users(users[:5], top_k=10, exclude=gen)
    r, li = rowptr.cpu().numpy(), lists.cpu().numpy()
    for i, u in enumerate(users[:5]):
        assert not np.isin(top[i], li[r[u]:r[u + 1]]).any()


def test_out_of_range_ids_raise(eng_mod, tmp_path):
    m, gen, nu, ni = _ml100k(tmp_path)
    with pytest.raises(IndexError):
        m.model.recommend_for_users([1, nu], top_k=5)
    with pytest.raises(IndexError):
        m.model.recommend_for_users([-1], top_k=5)
    with pytest.raises(IndexError):
        m.evaluate_full_catalogue([1, 2], [3, ni], k=10)
    with pytest.raises(IndexError):
        m.evaluate_full_catalogue([1, nu + 5], [3, 4], k=10)
    # the device call itself marks the bad user's rows
    items, scores, pos, _, _ = m.model.engine.catalogue_topk([nu, 1], 5, targets=[2, -1])
    assert (items.cpu().numpy()[0] == -1).all() and np.isnan(scores.cpu().numpy()[0]).all()
    assert pos.cpu().numpy().tolist() == [ni, ni]


def test_malformed_exclusion_lists_raise_before_any_launch(eng_mod):
    eng = _engine(eng_mod, [64, 32, 16, 8], 8, 6, 40)
    scores = torch.rand((6, 40), device="cuda")
    users = np.arange(6, dtype=np.int32)
    targets = (np.int64([0, 1, 1, 1, 2, 2, 2]), np.int32([3, 5]))
    # an unsorted list, and rowptr[-1] < len(items): neither can make a kernel leave its arrays
    for bad in ((np.int64([0, 2, 2, 2, 2, 2, 2]), np.int32([7, 3])),
                (np.int64([0, 1, 1, 1, 1, 1, 1]), np.int32([3, 7]))):
        for call in (lambda: eng.catalogue_topk(users, 5, exclude=bad),
                     lambda: eng_mod.topk_scores(scores, 5, exclude=bad),
                     lambda: eng.catalogue_targets(users, targets, [5], exclude=bad),
                     lambda: eng_mod.targets_scores(scores, targets, [5], exclude=bad)):
            with pytest.raises(ValueError, match="exclusion lists"):
                call()
