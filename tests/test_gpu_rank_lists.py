"""Ragged candidate lists on a B200: mr_topk_lists and mr_rank_lists against the NumPy reference (selection
bit-exact, probabilities within the parity tolerance), bit-identity with mr_rank_eval, independence of a list's
outputs from the rest of the call, out-of-range ids and the Python face (recommend_batch, evaluate_candidate_lists)."""

import numpy as np
import pytest

from lists_oracle import csr, topk_lists
from oracle import movierec_oracle as o
from test_gpu_catalogue import TOWERS, close_to_truth

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

INT32_MIN, INT32_MAX = -2 ** 31, 2 ** 31 - 1
# the four towers of the catalogue tests, plus the projected tower with the projection off (plain forward)
KINDS = [(layers, mf, "auto") for layers, mf in TOWERS] + [([256, 128, 64], 64, "off")]
KIND_IDS = ["tc-gmf64", "tc-nogmf", "default-tower", "simt", "tc-proj-off"]


@pytest.fixture(scope="module")
def eng_mod():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from movierec import _engine
    return _engine


def adversarial(rng, n):
    vals = np.float32([0.25, 0.5, 0.5, 0.75, np.nan, np.inf, -np.inf, -0.0, 0.0, 1.0])
    return np.where(rng.random(n) < 0.5, rng.choice(vals, n),
                    rng.integers(0, 64, n).astype(np.float32) / 64).astype(np.float32)  # many exact ties


def check_selection(got, want):
    top_pos, top_scores, pos, sums = got
    w_pos, w_scores, w_p, w_sums = want
    np.testing.assert_array_equal(top_pos.cpu().numpy(), w_pos)
    np.testing.assert_array_equal(top_scores.cpu().numpy().view(np.int32), w_scores.view(np.int32))
    if w_p is not None:
        np.testing.assert_array_equal(pos.cpu().numpy(), w_p)
        s = sums.cpu().numpy().astype(np.float64)
        assert s[0] == w_sums[0]
        assert abs(s[1] - w_sums[1]) <= 1e-6 * max(abs(w_sums[1]), 1.0)


def test_topk_lists_bit_exact_on_adversarial_scores(eng_mod):
    rng = np.random.default_rng(1)
    lens = []
    for k in (1, 10, 32, 33, 100, 256):
        lens += [0, 1, max(k - 1, 0), k, k + 1]
    lens += [31, 32, 33, 1023, 1024, 1025, 32 * 1024 + 1, 100003, (1 << 20) + 3]
    lens = rng.permutation(np.array(lens * 2, np.int64))
    rowptr = np.zeros(lens.size + 1, np.int64)
    rowptr[1:] = np.cumsum(lens)
    p = adversarial(rng, int(rowptr[-1]))
    U = lens.size
    kind = np.arange(U) % 5  # first, middle, last, -1, len
    targets = np.where(kind == 0, 0, np.where(kind == 1, lens // 2, np.where(kind == 2, lens - 1,
                                                                              np.where(kind == 3, -1, lens))))
    targets = targets.astype(np.int32)
    for k in (1, 10, 32, 33, 100, 256):
        got = eng_mod.topk_lists(p, rowptr, k, targets=targets)
        check_selection(got, topk_lists(p, rowptr, k, targets=targets))
    # without targets; from device offsets
    got = eng_mod.topk_lists(torch.from_numpy(p).cuda(), torch.from_numpy(rowptr).cuda(), 10)
    w = topk_lists(p, rowptr, 10)
    np.testing.assert_array_equal(got[0].cpu().numpy(), w[0])
    assert got[2] is None and got[3] is None


def test_topk_lists_many_tiny_lists_next_to_a_giant_one(eng_mod):
    rng = np.random.default_rng(2)
    lens = rng.integers(0, 4, 1 << 20).astype(np.int64)
    lens[rng.integers(0, lens.size)] = (1 << 20) + 7
    rowptr = np.zeros(lens.size + 1, np.int64)
    rowptr[1:] = np.cumsum(lens)
    p = adversarial(rng, int(rowptr[-1]))
    targets = (rng.integers(-1, 5, lens.size)).astype(np.int32)
    for k in (3, 100):
        check_selection(eng_mod.topk_lists(p, rowptr, k, targets=targets), topk_lists(p, rowptr, k, targets=targets))


def test_topk_lists_pos_equals_rank_scores_label_col(eng_mod):
    rng = np.random.default_rng(3)
    for group in (5, 100, 1000):
        G = 300
        p = adversarial(rng, G * group)
        lc = rng.integers(0, group, G).astype(np.int32)
        _, pos_rs, _ = eng_mod.rank_scores(p, group, 10, label_col=lc, want_rank=False)
        _, _, pos, _ = eng_mod.topk_lists(p, np.arange(G + 1, dtype=np.int64) * group, 10, targets=lc)
        np.testing.assert_array_equal(pos.cpu().numpy(), pos_rs.cpu().numpy())


def _engine(eng_mod, layers, mf, nu, ni, proj="auto", seed=11):
    return eng_mod.NeuMFEngine(nu, ni, layers, [0] * len(layers), mf_dim=mf, seed=seed, item_projection=proj)


def _random_lists(rng, U, ni, max_len=700):
    lens = rng.integers(0, max_len, U)
    lens[:3] = [0, 1, 2000]  # an empty list, a single candidate, one long list (two selection slices)
    return csr([rng.integers(0, ni, n) for n in lens])  # duplicates included


@pytest.mark.parametrize("layers,mf,proj", KINDS, ids=KIND_IDS)
def test_rank_lists_against_oracle(eng_mod, layers, mf, proj):
    nu, ni, k = 70, 1000, 10
    eng = _engine(eng_mod, layers, mf, nu, ni, proj)
    rng = np.random.default_rng(5)
    U = 40
    users = rng.integers(0, nu, U).astype(np.int32)
    rowptr, items = _random_lists(rng, U, ni)
    lens = np.diff(rowptr)
    targets = (rng.random(U) * np.maximum(lens, 1)).astype(np.int32)
    top_items, top_scores, top_pos, pos, sums, probs = eng.rank_lists(users, (rowptr, items), k, targets=targets,
                                                                      want_probs=True)
    assert float(eng.last_lists_bad.item()) == 1  # the empty list's target lies outside it
    p = probs.cpu().numpy()
    w = topk_lists(p, rowptr, k, targets=targets)
    check_selection((top_pos, top_scores, pos, sums), w)
    tp = top_pos.cpu().numpy()
    want_items = np.where(tp >= 0, items[np.clip(rowptr[:-1, None] + tp, 0, items.size - 1)], -1)
    np.testing.assert_array_equal(top_items.cpu().numpy(), want_items)
    wts = eng.get_weights()
    row_users = np.repeat(users, lens)
    p32 = o.forward(wts, row_users, items)["p"]
    p64 = o.forward({a: np.asarray(b, np.float64) for a, b in wts.items()}, row_users, items)["p"]
    close_to_truth(p, p32, p64, "list probabilities {} / {} / {}".format(layers, mf, proj))


@pytest.mark.parametrize("layers,mf", [([256, 128, 64], 64), ([64, 32, 16, 8], 8)], ids=["tc-gmf64", "default-tower"])
def test_rank_lists_equals_rank_eval_bit_for_bit(eng_mod, layers, mf):
    nu, ni = 300, 2000
    eng = _engine(eng_mod, layers, mf, nu, ni, "on")
    rng = np.random.default_rng(8)
    for group in (5, 100, 256):
        G = 97
        users = rng.integers(0, nu, G).astype(np.int32)
        cand = rng.integers(0, ni, (G, group)).astype(np.int32)
        pos_e, _, _, probs_e = eng.rank_eval(torch.from_numpy(users).cuda(), torch.from_numpy(cand.ravel()).cuda(), group,
                                             10, want_probs=True)
        rowptr = np.arange(G + 1, dtype=np.int64) * group
        _, _, _, pos, _, probs = eng.rank_lists(users, (rowptr, cand.ravel()), 10,
                                                targets=np.full(G, group - 1, np.int32), want_probs=True)
        np.testing.assert_array_equal(probs.cpu().numpy().view(np.int32), probs_e.cpu().numpy().view(np.int32))
        np.testing.assert_array_equal(pos.cpu().numpy(), pos_e.cpu().numpy())


def _bits(outs):
    return [x.cpu().numpy().view(np.int32).copy() if x is not None else None for x in outs]


@pytest.mark.parametrize("layers,mf,proj", KINDS, ids=KIND_IDS)
def test_list_outputs_do_not_depend_on_the_batch(eng_mod, layers, mf, proj):
    nu, ni, k = 90, 1500, 10
    eng = _engine(eng_mod, layers, mf, nu, ni, proj)
    rng = np.random.default_rng(9)
    U = 60
    users = rng.integers(0, nu, U).astype(np.int32)
    rowptr, items = _random_lists(rng, U, ni, 1200)
    lens = np.diff(rowptr)
    targets = (rng.random(U) * np.maximum(lens, 1)).astype(np.int32)
    lists = [items[rowptr[u]:rowptr[u + 1]] for u in range(U)]
    a = _bits(eng.rank_lists(users, (rowptr, items), k, targets=targets, want_probs=True))
    b = _bits(eng.rank_lists(users, (rowptr, items), k, targets=targets, want_probs=True))
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    perm = rng.permutation(U)
    pr, pi = csr([lists[u] for u in perm])
    c = _bits(eng.rank_lists(users[perm], (pr, pi), k, targets=targets[perm], want_probs=True))
    for i, u in enumerate(perm):
        for j in range(3):  # top items, scores, positions
            np.testing.assert_array_equal(c[j][i], a[j][u])
        assert c[3][i] == a[3][u]
        np.testing.assert_array_equal(c[5][pr[i]:pr[i + 1]], a[5][rowptr[u]:rowptr[u + 1]])
    for u in (0, 1, 2, 7, U - 1):
        r1, i1 = csr([lists[u]])
        s = _bits(eng.rank_lists(users[u:u + 1], (r1, i1), k, targets=targets[u:u + 1], want_probs=True))
        for j in range(3):
            np.testing.assert_array_equal(s[j][0], a[j][u])
        assert s[3][0] == a[3][u]
        np.testing.assert_array_equal(s[5], a[5][rowptr[u]:rowptr[u + 1]])


@pytest.mark.parametrize("layers,mf,proj", KINDS, ids=KIND_IDS)
def test_out_of_range_ids_in_the_device_call(eng_mod, layers, mf, proj):
    nu, ni, k = 50, 800, 5
    eng = _engine(eng_mod, layers, mf, nu, ni, proj)
    rng = np.random.default_rng(10)
    lists = [rng.integers(0, ni, 30) for _ in range(6)]
    lists[5][[3, 17]] = [ni, -1]  # out-of-range items in a valid user's list
    rowptr, items = csr(lists)
    users = np.array([-1, nu, INT32_MIN, INT32_MAX, 3, 4], np.int32)
    targets = np.array([0, 1, 2, 3, 4, 3], np.int32)
    top_items, top_scores, top_pos, pos, _, probs = eng.rank_lists(users, (rowptr, items), k, targets=targets,
                                                                    want_probs=True)
    assert float(eng.last_lists_bad.item()) > 0
    ti, ts, tp = top_items.cpu().numpy(), top_scores.cpu().numpy(), top_pos.cpu().numpy()
    assert (ti[:4] == -1).all() and (tp[:4] == -1).all() and np.isnan(ts[:4]).all()
    assert pos.cpu().numpy().tolist()[:4] == [30] * 4
    p = probs.cpu().numpy()
    assert np.isnan(p[rowptr[5] + 3]) and np.isnan(p[rowptr[5] + 17])
    assert np.isfinite(np.delete(p[rowptr[5]:rowptr[6]], [3, 17])).all()
    assert pos.cpu().numpy()[5] == 28  # the target is the first NaN candidate: after the 28 valid ones
    _, p_ok, _, _, _, _ = eng.rank_lists(users[4:5], csr([lists[4]]), k)
    np.testing.assert_array_equal(p_ok.cpu().numpy()[0], ts[4])


def _facade(eng):
    from movierec import model as mm
    f = mm.NeuMFModel.__new__(mm.NeuMFModel)
    f.engine = eng
    f._owner = mm.MovierecModel.__new__(mm.MovierecModel)
    f._owner._num_users, f._owner._num_items = eng.num_users, eng.num_items
    return f


@pytest.mark.parametrize("layers,mf,proj", KINDS, ids=KIND_IDS)
def test_recommend_batch_against_recommend(eng_mod, layers, mf, proj):
    nu, ni, K = 60, 1000, 10
    eng = _engine(eng_mod, layers, mf, nu, ni, proj)
    rng = np.random.default_rng(12)
    users = rng.integers(0, nu, 24).astype(np.int32)
    lists = [rng.integers(0, ni, n) for n in rng.integers(1, 1000, 24)]  # recommend() ranks <= 1,024 candidates
    lists[0] = lists[0][:3]  # shorter than K: -1 / NaN padding
    f = _facade(eng)
    items, scores = f.recommend_batch(users, lists, top_k=K)
    r2, s2 = f.recommend_batch(users, csr(lists), top_k=K)
    np.testing.assert_array_equal(items, r2)
    exact = proj == "off" or mf == 0  # the plain-forward sequence: the same kernels as recommend()
    for u in range(len(users)):
        ri, rs = f.recommend(int(users[u]), lists[u], K)
        n = ri.size
        assert (items[u, n:] == -1).all() and np.isnan(scores[u, n:]).all()
        if exact:
            np.testing.assert_array_equal(items[u, :n], ri)
            np.testing.assert_array_equal(scores[u, :n].view(np.int32), rs.view(np.int32))
        else:
            np.testing.assert_allclose(scores[u, :n], rs, rtol=1e-5, atol=1e-6)
            # the orders agree wherever the scores are farther apart than the tolerance
            mine = dict(zip(items[u, :n].tolist(), scores[u, :n].tolist()))
            for a in range(n):
                for b in range(a + 1, n):
                    if rs[a] - rs[b] > 1e-5 and ri[a] in mine and ri[b] in mine:
                        assert mine[ri[a]] > mine[ri[b]]
    with pytest.raises(IndexError):
        f.recommend_batch([0, nu], [[1], [2]])
    with pytest.raises(IndexError):
        f.recommend_batch([INT32_MIN], [[1]])
    with pytest.raises(IndexError):
        f.recommend_batch([0, 1], [[1, ni], [2]])
    with pytest.raises(IndexError):
        f.recommend_batch([0], [[-1]])
    with pytest.raises(ValueError):
        f.recommend_batch([0, 1], (np.array([0, 3, 2]), np.arange(2)))
    with pytest.raises(ValueError):
        eng.rank_lists([0, 1], (np.array([1, 2, 2]), np.arange(2)), 5)
    with pytest.raises(ValueError):
        eng.rank_lists([0, 1], (torch.tensor([0, 2, 3]).cuda(), np.arange(2)), 5)


def test_chunked_calls_equal_one_call(eng_mod, monkeypatch):
    from movierec import model as mm
    nu, ni = 200, 3000
    for layers, mf, proj in (([256, 128, 64], 64, "auto"), ([64, 32, 16, 8], 8, "auto"), ([6, 4], 0, "auto")):
        eng = _engine(eng_mod, layers, mf, nu, ni, proj)
        rng = np.random.default_rng(13)
        users = rng.integers(0, nu, 300).astype(np.int32)
        lists = [rng.integers(0, ni, n) for n in rng.integers(1, 400, 300)]
        lists[7] = rng.integers(0, ni, 5000)  # longer than a small chunk: a call of its own
        targets = np.array([rng.integers(0, len(x)) for x in lists], np.int32)
        f = _facade(eng)
        a = f.recommend_batch(users, lists, top_k=10)
        owner = f._owner
        owner.model, owner._k = f, 10
        e1 = owner.evaluate_candidate_lists(users, lists, targets)
        monkeypatch.setattr(mm, "LISTS_CALL_ROWS", 3000)
        assert len(mm._list_chunks(csr(lists)[0])) > 5
        b = f.recommend_batch(users, lists, top_k=10)
        e2 = owner.evaluate_candidate_lists(users, lists, targets)
        monkeypatch.undo()
        np.testing.assert_array_equal(a[0], b[0])
        np.testing.assert_array_equal(a[1].view(np.int32), b[1].view(np.int32))
        assert e1[0] == e2[0] and abs(e1[1] - e2[1]) <= 1e-6


def test_evaluate_candidate_lists_reproduces_evaluate(eng_mod, tmp_path):
    import copy
    from movierec import model as mm
    nu, ni = 943, 1682
    for layers, mf in (([256, 128, 64], 64), ([64, 32, 16, 8], 8)):
        params = {"num_users": nu, "num_items": ni, "layers_sizes": layers, "layers_l2reg": [0] * len(layers),
                  "optimizer": "adam", "lr": 0.001, "batch_size": 25, "num_negs_per_pos": 4, "batch_size_eval": 100,
                  "num_negs_per_pos_eval": 99, "k": 5, "mf_dim": mf, "seed": 2}
        eng_mod.set_item_projection("on")
        try:
            m = mm.MovierecModel(copy.deepcopy(params), output_dir=str(tmp_path))
        finally:
            eng_mod.set_item_projection("auto")
        rng = np.random.default_rng(14)
        users = rng.integers(0, nu, 500).astype(np.int32)
        items = rng.integers(0, ni, 500 * 100).astype(np.int32)
        hr, ndcg = m.evaluate(users, items)
        hr2, ndcg2 = m.evaluate_candidate_lists(users, (np.arange(501, dtype=np.int64) * 100, items),
                                                np.full(500, 99, np.int32))
        assert hr == hr2
        assert abs(ndcg - ndcg2) <= 1e-6 * max(ndcg, 1e-3)
        with pytest.raises(IndexError):
            m.evaluate_candidate_lists([1, nu], [[1, 2], [3]], [0, 0])
        with pytest.raises(IndexError):
            m.evaluate_candidate_lists([1, 2], [[1, 2], [3]], [0, 1])  # a target outside its list
