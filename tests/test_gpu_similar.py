"""Similar items and users on a B200 (mr_similar): similarities against the float64 oracle, the selection bit-exact
against the NumPy selection on the call's own scores, sizes across chunks and k paths, duplicated / out-of-range
queries, exclusion lists, zero rows, determinism and independence from the other queries, folded-in rows, the Python
face and neighbour quality on planted clusters."""

import numpy as np
import pytest

from catalogue_oracle import csr
from similar_oracle import side_parts, similar_select, truth
from test_gpu_catalogue import TOWERS, _engine, close_to_truth

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

SIM_TOWERS = TOWERS + [([8], 4), ([64, 512], 256)]  # + the GMF part alone, and D = 768 (24 K-chunks)
SIDES = ("items", "users")


@pytest.fixture(scope="module")
def eng_mod():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from movierec import _engine
    return _engine


def _np(t):
    return t.cpu().numpy() if t is not None else None


def run(eng, ids, k, side="items", exclude=None, excl_ids=None):
    """One call with every output, its selection checked bit for bit against the NumPy selection on its own scores."""
    top, sims, full = eng.similar(ids, k, side=side, exclude=exclude, excl_ids=excl_ids, want_scores=True)
    top, sims, S = _np(top), _np(sims), _np(full)
    rp, ex = exclude if exclude is not None else (None, None)
    w_top, w_sims = similar_select(S, ids, k, rp, ex, excl_ids)
    np.testing.assert_array_equal(top, w_top)
    np.testing.assert_array_equal(sims.view(np.int32), w_sims.view(np.int32))
    N = S.shape[1]
    ids = np.asarray(ids, np.int64)
    for j in range(ids.size):
        assert ids[j] not in top[j][top[j] >= 0] or not 0 <= ids[j] < N
    return top, sims, S


@pytest.mark.parametrize("side", SIDES)
@pytest.mark.parametrize("layers,mf", SIM_TOWERS, ids=["tc-gmf64", "tc-nogmf", "default-tower", "simt", "gmf-only",
                                                       "wide-d768"])
def test_towers_against_oracle(eng_mod, layers, mf, side):
    nu, ni = 300, 257
    eng = _engine(eng_mod, layers, mf, nu, ni)
    N = ni if side == "items" else nu
    rng = np.random.default_rng(3)
    ids = rng.integers(0, N, 60).astype(np.int32)
    ids[5] = ids[7]      # duplicated query
    ids[9] = N           # out of range
    ids[11] = -3
    top, sims, S = run(eng, ids, 10, side)
    s32, s64 = truth(eng.get_weights(), side, mf, ids)
    close_to_truth(S, s32, s64, "similarities {} / {} {}".format(layers, mf, side))
    ok = (ids >= 0) & (ids < N)
    np.testing.assert_allclose(S[np.flatnonzero(ok), ids[ok]], 1.0, atol=1e-5)  # self-similarity
    assert (S[~ok] == 0).all() and (top[~ok] == -1).all() and np.isnan(sims[~ok]).all()
    assert np.array_equal(top[5], top[7])
    assert np.all(np.abs(S) <= 1 + 1e-5)


@pytest.mark.parametrize("N", [1, 2, 31, 257, 3706, 26744])
def test_sizes_and_k(eng_mod, N):
    eng = _engine(eng_mod, [256, 128, 64], 64, 10, N)
    rng = np.random.default_rng(N)
    M = 400 if N == 26744 else min(N + 3, 50)  # 26,744 items: 156 queries per chunk, three chunks
    ids = rng.integers(0, N, M).astype(np.int32)
    ids[0] = N - 1
    ks = [1, 10, 256, 257, 1000] + ([N + 5] if N + 5 <= 4096 else [])
    S0 = None
    for k in ks:
        top, sims, S = run(eng, ids, k)
        if S0 is None:
            S0 = S
            s32, s64 = truth(eng.get_weights(), "items", 64, ids)
            close_to_truth(S, s32, s64, "similarities N={}".format(N))
        np.testing.assert_array_equal(S.view(np.int32), S0.view(np.int32))  # scores do not depend on k
        n_cand = N - 1
        if k > n_cand:
            assert (top[:, n_cand:] == -1).all() and np.isnan(sims[:, n_cand:]).all()
        assert (top[:, :min(k, n_cand)] >= 0).all()


def test_exclusion_lists(eng_mod):
    N = 1000
    eng = _engine(eng_mod, [64, 32, 16, 8], 8, 20, N)
    rng = np.random.default_rng(7)
    lists = [sorted(rng.choice(N, int(rng.integers(0, 300)), replace=False).tolist()) for _ in range(9)]
    lists[3] = list(range(N))  # covers every id
    rp, ex = csr(lists)
    M = 40
    ids = rng.integers(0, N, M).astype(np.int32)
    excl_ids = rng.integers(-1, 11, M).astype(np.int32)  # duplicated rows, rows outside the table
    excl_ids[0] = 3
    for k in (10, 300):
        top, sims, _ = run(eng, ids, k, exclude=(rp, ex), excl_ids=excl_ids)
        assert (top[0] == -1).all() and np.isnan(sims[0]).all()
    top, _, _ = run(eng, ids[:9], 12, exclude=(rp, ex))  # default: query j uses list j
    with pytest.raises(ValueError):
        eng.similar(ids, 5, exclude=(np.int64([0, 2]), np.int32([3, 1])))


@pytest.mark.parametrize("side", SIDES)
def test_zero_rows(eng_mod, side):
    nu, ni = 90, 80
    eng = _engine(eng_mod, [256, 128, 64], 64, nu, ni)
    w = eng.get_weights()
    mlp = "item_embedding/embeddings" if side == "items" else "user_embedding/embeddings"
    gmf = "gmf_item_embedding/embeddings" if side == "items" else "gmf_user_embedding/embeddings"
    w[mlp][[1, 4]] = 0
    w[gmf][[1, 6]] = 0  # row 1 all zero, row 4 without its MLP part, row 6 without its GMF part
    eng.set_weights(w)
    N = ni if side == "items" else nu
    ids = np.int32([1, 4, 6, 0, 1])
    top, sims, S = run(eng, ids, N + 2, side)
    assert not np.isnan(S).any() and not np.isnan(sims[:, :N - 1]).any()
    assert (S[0] == 0).all() and (S[:, 1] == 0).all()
    assert abs(S[1, 4] - 0.5) <= 1e-5 and abs(S[2, 6] - 0.5) <= 1e-5  # one part of two
    assert abs(S[3, 0] - 1.0) <= 1e-5
    s32, s64 = truth(eng.get_weights(), side, 64, ids)
    close_to_truth(S, s32, s64, "similarities with zero rows")


def test_determinism_and_independence(eng_mod):
    N = 26744
    eng = _engine(eng_mod, [256, 128, 64], 64, 10, N)
    rng = np.random.default_rng(1)
    crowd = rng.integers(0, N, 1000).astype(np.int32)
    probe = int(crowd[500])
    for k in (20, 500):
        a = eng.similar(crowd, k, want_scores=True)
        b = eng.similar(crowd, k, want_scores=True)
        for x, y in zip(a, b):
            np.testing.assert_array_equal(_np(x).view(np.int32), _np(y).view(np.int32))
        alone = [_np(t) for t in eng.similar([probe], k, want_scores=True)]
        perm = rng.permutation(crowd.size)
        shuf = [_np(t) for t in eng.similar(crowd[perm], k, want_scores=True)]
        at = int(np.flatnonzero(perm == 500)[0])
        for got_alone, got_crowd, got_shuf in zip(alone, a, shuf):
            np.testing.assert_array_equal(got_alone[0].view(np.int32), _np(got_crowd)[500].view(np.int32))
            np.testing.assert_array_equal(got_alone[0].view(np.int32), got_shuf[at].view(np.int32))


def test_folded_in_rows(eng_mod):
    nu, ni = 400, 300
    eng = _engine(eng_mod, [64, 32, 16, 8], 8, nu, ni)
    rng = np.random.default_rng(4)
    raters = [np.sort(rng.choice(nu, n, replace=False)) for n in (40, 15)]
    mlp, gmf, _ = eng.fold_in_items(raters, 5, 0.05, 4)
    view = eng.item_view(mlp, gmf)
    ids = np.int32([ni, ni + 1, 0, 17])  # the new items as queries; they are candidates of every query
    top, _, S = run(view, ids, 20)
    s32, s64 = truth(view.get_weights(), "items", 8, ids)
    close_to_truth(S, s32, s64, "similarities on the extended catalogue")
    assert S.shape == (4, ni + 2)
    hist = [np.sort(rng.choice(ni, n, replace=False)) for n in (30, 8)]
    umlp, ugmf, _ = eng.fold_in(hist, 5, 0.05, 4)
    uview = eng.user_view(umlp, ugmf)
    _, _, Su = run(uview, np.int32([0, 1]), 1, side="users")
    s32, s64 = truth(uview.get_weights(), "users", 8, [0, 1])
    close_to_truth(Su, s32, s64, "similarities of folded-in users")


def test_python_face(eng_mod, tmp_path):
    from test_gpu_audience import _movierec
    nu, ni = 300, 60
    mr = _movierec(tmp_path, nu, ni)
    eng = mr.model.engine
    q = np.int32([3, 0, 59, 3])
    rp, ex = csr([[1, 2], [], [58], [0]])
    top, sims = mr.model.similar_items(q, top_k=8, exclude=(rp, ex))
    _, _, full = eng.similar(q, 8, want_scores=True)
    want = similar_select(_np(full), q, 8, rp, ex)
    np.testing.assert_array_equal(top, want[0])
    np.testing.assert_array_equal(sims.view(np.int32), want[1].view(np.int32))
    assert isinstance(top, np.ndarray) and top.shape == (4, 8)
    utop, _ = mr.model.similar_users([5, 299], top_k=3)
    assert utop.shape == (2, 3) and 5 not in utop[0]
    with pytest.raises(IndexError):
        mr.model.similar_items([ni], top_k=5)
    with pytest.raises(IndexError):
        mr.model.similar_users([-1], top_k=5)
    with pytest.raises(ValueError):
        eng.similar(q, 5, side="movies")


def test_planted_clusters(eng_mod):
    from test_gpu_fold_in import planted_dataset, train_planted
    uc, ic, hist = planted_dataset()
    eng = train_planted(eng_mod, hist, 480)
    items = np.arange(480, dtype=np.int32)
    top = _np(eng.similar(items, 10)[0])
    prec = float(np.mean(ic[top] == ic[items][:, None]))
    w = eng.get_weights()
    E, _, G, _ = side_parts(w, "items", 8)
    raw = np.concatenate([E, G], axis=1).astype(np.float64)
    raw /= np.maximum(np.linalg.norm(raw, axis=1, keepdims=True), 1e-30)
    C = raw @ raw.T
    np.fill_diagonal(C, -np.inf)
    raw_top = np.argsort(-C, axis=1, kind="stable")[:, :10]
    raw_prec = float(np.mean(ic[raw_top] == ic[:, None]))
    print("planted clusters item neighbour precision@10: representation {:.3f} raw embeddings {:.3f} chance {:.3f}".format(
        prec, raw_prec, 1 / 8))
    assert prec >= 2 / 8
