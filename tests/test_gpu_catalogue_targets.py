"""Many held-out items per user on a B200: mr_targets_scores bit-exact against the NumPy reference on adversarial scores,
mr_catalogue_targets against mr_catalogue_topk (one target per user) and against mr_targets_scores on the same
probabilities, determinism, chunking, and MovierecModel.evaluate_full_catalogue_sets."""

import copy
import ctypes

import numpy as np
import pandas as pd
import pytest

from catalogue_oracle import csr
from targets_oracle import target_metrics, target_positions

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

TOWERS = [([256, 128, 64], 64), ([256, 128, 64], 0), ([64, 32, 16, 8], 8), ([6, 4], 0)]
TOWER_IDS = ["tc-gmf64", "tc-nogmf", "default-tower", "simt"]


@pytest.fixture(scope="module")
def eng_mod():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from movierec import _engine
    return _engine


def sums_close(got, want, rtol=1e-6):
    got = np.asarray(got.cpu().numpy() if hasattr(got, "cpu") else got, np.float64)
    want = np.asarray(want, np.float64)
    assert got.shape == want.shape
    err = np.abs(got - want) / np.maximum(np.abs(want), 1.0)
    assert float(err.max()) <= rtol, "sums {} vs {}".format(got.tolist(), want.tolist())


def target_lists(rng, U, N, lengths):
    """U ascending target lists: lengths cycle through `lengths` (capped at N; "all" = every item of the catalogue),
    some lists with ids -1 and N around them."""
    lists = []
    for u in range(U):
        n = lengths[u % len(lengths)]
        t = list(range(N)) if n == "all" else sorted(rng.choice(N, min(n, N), replace=False).tolist())
        if u % 7 == 3:
            t = [-1] + t + [N]
        lists.append(t)
    rowptr = np.zeros(U + 1, np.int64)
    rowptr[1:] = np.cumsum([len(x) for x in lists])
    items = np.concatenate([np.asarray(x, np.int32) for x in lists]) if lists else np.zeros(0, np.int32)
    return rowptr, items.astype(np.int32)


@pytest.mark.parametrize("N", [1, 31, 32, 1000, 26744, 100003])
def test_targets_scores_bit_exact_on_adversarial_scores(eng_mod, N):
    rng = np.random.default_rng(N)
    chunk = max(1, min((1 << 22) // N, 16384))
    U = min(chunk + 3, 45) if N >= 26744 else 37  # crosses a chunk boundary for the largest catalogue
    vals = np.float32([0.25, 0.5, 0.5, 0.75, np.nan, np.inf, -np.inf, -0.0, 0.0, 1.0])
    p = np.where(rng.random((U, N)) < 0.5, rng.choice(vals, (U, N)),
                 rng.integers(0, 64, (U, N)).astype(np.float32) / 64).astype(np.float32)  # many exact ties
    rowptr, items = target_lists(rng, U, N, [0, 1, 2, 33, 1025, 3, "all" if N <= 1000 or U > 40 else 5])
    ex_lists = []
    for u in range(9):  # exclusion lists overlapping the targets of the rows that use them
        own = items[rowptr[u]:rowptr[u + 1]]
        own = own[(own >= 0) & (own < N)]
        pick = rng.choice(N, min(N, 200), replace=False)
        ex_lists.append(sorted(set(pick.tolist()) | set(own[::2].tolist())))
    ex_lists[3] = list(range(N))  # a row with every item excluded
    ex_rowptr, ex = csr(ex_lists)
    excl_ids = rng.integers(-1, 11, U).astype(np.int32)  # duplicated rows, rows outside the table
    excl_ids[:9] = np.arange(9)
    ks = [1, 5, 10, 100, N + 7]
    tpos, sums = eng_mod.targets_scores(p, (rowptr, items), ks, exclude=(ex_rowptr, ex), excl_ids=excl_ids)
    want = target_positions(p, rowptr, items, ex_rowptr, ex, excl_ids=excl_ids)
    np.testing.assert_array_equal(tpos.cpu().numpy(), want)
    sums_close(sums, target_metrics(want, rowptr, ks))
    # without exclusion lists, one cutoff
    tpos, sums = eng_mod.targets_scores(p, (rowptr, items), [10])
    want = target_positions(p, rowptr, items)
    np.testing.assert_array_equal(tpos.cpu().numpy(), want)
    sums_close(sums, target_metrics(want, rowptr, [10]))


def test_malformed_rowptr_stays_in_bounds(eng_mod):
    from movierec import _native as nat
    U, N, nnz = 6, 500, 40
    dev = torch.device("cuda")
    p = torch.rand((U, N), device=dev)
    items = torch.arange(nnz, dtype=torch.int32, device=dev) * 3
    guard = torch.full((nnz + 64,), -7, dtype=torch.int32, device=dev)
    tpos = guard[:nnz]
    sums = torch.zeros(7, device=dev)
    for rp in ([0, 30, 10, 60, -5, 40, 1 << 40], [5, 3, 2, 1, 0, 0, 0], [0, 40, 40, 40, 40, 40, 90]):
        rowptr = torch.tensor(rp, dtype=torch.int64, device=dev)
        nbytes = nat.lib.mr_targets_scores_workspace_bytes(U, N, nnz)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        ks = (ctypes.c_int32 * 1)(10)
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        rc = nat.lib.mr_targets_scores(ctypes.c_void_p(p.data_ptr()), U, N, None, 0, None, None,
                                       ctypes.c_void_p(rowptr.data_ptr()), ctypes.c_void_p(items.data_ptr()), nnz, ks, 1,
                                       ctypes.c_void_p(tpos.data_ptr()), ctypes.c_void_p(sums.data_ptr()),
                                       ctypes.c_void_p(ws.data_ptr()), nbytes, st)
        assert rc == 0
        torch.cuda.synchronize()
        assert (guard[nnz:] == -7).all()  # nothing written past the target array
    # an unsorted list: results unspecified, the call completes
    items_rev = items.flip(0).contiguous()
    eng_mod.targets_scores(p, (torch.tensor([0, 10, 20, 20, 30, 35, 40]), items_rev), [5])
    torch.cuda.synchronize()


def _engine(eng_mod, layers, mf, nu, ni, seed=11, **kw):
    return eng_mod.NeuMFEngine(nu, ni, layers, [0] * len(layers), mf_dim=mf, seed=seed, **kw)


def random_lists(rng, rows, N, most=300):
    return csr([sorted(rng.choice(N, int(rng.integers(0, min(N, most))), replace=False).tolist()) for _ in range(rows)])


@pytest.mark.parametrize("layers,mf,proj", [(L, f, None) for L, f in TOWERS] + [([256, 128, 64], 64, "off")],
                         ids=TOWER_IDS + ["tc-gmf64-unprojected"])
def test_one_target_per_user_equals_catalogue_topk(eng_mod, layers, mf, proj):
    nu, ni, k = 70, 1000, 10
    eng = _engine(eng_mod, layers, mf, nu, ni, item_projection=proj)
    rng = np.random.default_rng(5)
    users = rng.integers(0, nu, 40).astype(np.int32)
    users[7] = nu  # an out-of-range user: every target gets N
    rowptr, ex = random_lists(rng, nu, ni)
    targets = rng.integers(0, ni, 40).astype(np.int32)
    targets[3], targets[11] = -1, ni  # out-of-range targets
    for u in range(0, 40, 5):  # targets on the user's exclusion list
        lst = ex[rowptr[users[u] % nu]:rowptr[users[u] % nu + 1]]
        if lst.size and u not in (3, 11):
            targets[u] = lst[0]
    _, _, pos, sums, _ = eng.catalogue_topk(users, k, exclude=(rowptr, ex), targets=targets)
    tpos, tsums = eng.catalogue_targets(users, (np.arange(41, dtype=np.int64), targets), [k], exclude=(rowptr, ex))
    np.testing.assert_array_equal(tpos.cpu().numpy(), pos.cpu().numpy())
    s, t = sums.cpu().numpy().astype(np.float64), tsums.cpu().numpy().astype(np.float64)
    assert t[0] == 40 and t[2] == s[0]
    assert abs(t[5] - s[1]) <= 1e-6 * max(s[1], 1.0)
    assert float(eng.last_catalogue_bad.item()) > 0


@pytest.mark.parametrize("layers,mf", [([256, 128, 64], 64), ([64, 32, 16, 8], 8)], ids=["tc-gmf64", "default-tower"])
def test_catalogue_targets_equal_targets_scores_on_its_probabilities(eng_mod, layers, mf):
    nu, ni = 90, 2000
    eng = _engine(eng_mod, layers, mf, nu, ni)
    rng = np.random.default_rng(9)
    users = np.arange(nu, dtype=np.int32)
    ex_rowptr, ex = random_lists(rng, nu, ni)
    rowptr, items = target_lists(rng, nu, ni, [0, 1, 2, 33, 600, 1025, 4])
    ks = [1, 10, 50]
    tpos, sums = eng.catalogue_targets(users, (rowptr, items), ks, exclude=(ex_rowptr, ex))
    _, _, _, _, full = eng.catalogue_topk(users, 10, want_scores=True)
    tpos2, sums2 = eng_mod.targets_scores(full, (rowptr, items), ks, exclude=(ex_rowptr, ex), excl_ids=users)
    np.testing.assert_array_equal(tpos.cpu().numpy(), tpos2.cpu().numpy())
    np.testing.assert_array_equal(sums.cpu().numpy().view(np.int32), sums2.cpu().numpy().view(np.int32))
    want = target_positions(full.cpu().numpy(), rowptr, items, ex_rowptr, ex, excl_ids=users)
    np.testing.assert_array_equal(tpos.cpu().numpy(), want)
    sums_close(sums, target_metrics(want, rowptr, ks))


def test_deterministic_and_chunking_invisible(eng_mod):
    ni = 1000
    chunk = (1 << 22) // ni
    nu = 2 * chunk + 5  # three chunks
    for layers, mf in (([256, 128, 64], 64), ([64, 32, 16, 8], 8)):
        eng = _engine(eng_mod, layers, mf, nu, ni)
        rng = np.random.default_rng(1)
        ex_rowptr, ex = random_lists(rng, nu, ni, most=60)
        users = np.arange(nu, dtype=np.int32)
        rowptr, items = target_lists(rng, nu, ni, [0, 1, 5, 17, 40])
        a = eng.catalogue_targets(users, (rowptr, items), [3, 10], exclude=(ex_rowptr, ex))
        b = eng.catalogue_targets(users, (rowptr, items), [3, 10], exclude=(ex_rowptr, ex))
        for x, y in zip(a, b):
            np.testing.assert_array_equal(x.cpu().numpy().view(np.int32), y.cpu().numpy().view(np.int32))
        tpos = a[0].cpu().numpy()
        sums_close(a[1], target_metrics(tpos, rowptr, [3, 10]))
        sample = sorted(set(rng.integers(0, nu, 6).tolist()) | {chunk - 1, chunk, 2 * chunk, nu - 1})
        single_sums = np.zeros(12)
        for u in sample:
            b0, b1 = int(rowptr[u]), int(rowptr[u + 1])
            t1, s1 = eng.catalogue_targets([u], (np.int64([0, b1 - b0]), items[b0:b1]), [3, 10], exclude=(ex_rowptr, ex))
            np.testing.assert_array_equal(t1.cpu().numpy(), tpos[b0:b1])
            single_sums += s1.cpu().numpy()
        sub = np.concatenate([np.arange(rowptr[u], rowptr[u + 1]) for u in sample]).astype(np.int64)
        sub_rowptr = np.concatenate([[0], np.cumsum([rowptr[u + 1] - rowptr[u] for u in sample])])
        sums_close(single_sums, target_metrics(tpos[sub], sub_rowptr, [3, 10]))


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


def test_evaluate_full_catalogue_sets(eng_mod, tmp_path):
    from movierec import data_pipeline as dp
    m, gen, nu, ni = _ml100k(tmp_path)
    rng = np.random.default_rng(6)
    # held-out ratings: 0 to 6 items for most users, repeats and file order as a ratings file has them
    tu = np.repeat(np.arange(1, nu), rng.integers(0, 7, nu - 1)).astype(np.int64)
    ti = rng.integers(1, ni, tu.size).astype(np.int64)
    test = pd.DataFrame({dp.COL_USER_ID: tu, dp.COL_ITEM_ID: ti, dp.COL_RATING: 1.0}).sample(frac=1.0, random_state=3)
    ks = (1, 5, 20)
    got = m.evaluate_full_catalogue_sets(test, exclude=gen, ks=ks)
    # the reference on the model's own probabilities
    eng = m.model.engine
    lists = [sorted(set(ti[tu == u].tolist())) for u in range(nu)]
    rowptr, items = csr(lists)
    users = np.flatnonzero(np.diff(rowptr) > 0).astype(np.int32)
    _, _, _, _, full = eng.catalogue_topk(users, 5, want_scores=True)
    sub_rowptr, sub_items = csr([lists[u] for u in users])
    ex_rowptr, ex = gen.user_item_lists()
    want_pos = target_positions(full.cpu().numpy(), sub_rowptr, sub_items, ex_rowptr.cpu().numpy(), ex.cpu().numpy(),
                                excl_ids=users)
    want = target_metrics(want_pos, sub_rowptr, ks)
    G = want[0]
    assert G == users.size
    expect = {"mrr": want[1] / G}
    for c, k in enumerate(ks):
        for j, name in enumerate(("hr", "precision", "recall", "ndcg", "map")):
            expect["{}@{}".format(name, k)] = want[2 + 5 * c + j] / G
    assert set(got) == set(expect)
    for key in expect:
        assert abs(got[key] - expect[key]) <= 1e-6 * max(abs(expect[key]), 1e-3), key
    # the same lists as a CSR indexed by user id
    got_csr = m.evaluate_full_catalogue_sets((rowptr, items), exclude=gen, ks=ks)
    for key in expect:
        assert got_csr[key] == got[key]
    # one held-out item per user: the leave-one-out evaluation
    held = rng.integers(1, ni, nu - 1).astype(np.int32)
    one = pd.DataFrame({dp.COL_USER_ID: np.arange(1, nu), dp.COL_ITEM_ID: held, dp.COL_RATING: 1.0})
    hr, ndcg = m.evaluate_full_catalogue(np.arange(1, nu, dtype=np.int32), held, exclude=gen, k=10)
    sets = m.evaluate_full_catalogue_sets(one, exclude=gen, ks=[10])
    assert sets["hr@10"] == hr
    assert abs(sets["ndcg@10"] - ndcg) <= 1e-6 * max(ndcg, 1e-3)
    assert m.evaluate_full_catalogue_sets(one.iloc[:0], exclude=gen)["mrr"] == 0.0


def test_evaluate_full_catalogue_sets_out_of_range_ids_raise(eng_mod, tmp_path):
    from movierec import data_pipeline as dp
    m, gen, nu, ni = _ml100k(tmp_path)
    for u, i in ((nu, 3), (-1, 3), (2, ni), (2, -1)):
        df = pd.DataFrame({dp.COL_USER_ID: [1, u], dp.COL_ITEM_ID: [4, i], dp.COL_RATING: 1.0})
        with pytest.raises(IndexError):
            m.evaluate_full_catalogue_sets(df, exclude=gen)
    with pytest.raises(IndexError):
        m.evaluate_full_catalogue_sets((np.int64([0, 1, 2]), np.int32([3, ni])))
    rowptr = np.zeros(nu + 2, np.int64)
    rowptr[-1] = 1  # a list for user nu
    with pytest.raises(IndexError):
        m.evaluate_full_catalogue_sets((rowptr, np.int32([3])))
    # the device call itself gives every target of a bad user position num_items
    tpos, _ = m.model.engine.catalogue_targets([nu, 1], (np.int64([0, 2, 3]), np.int32([2, 5, ni])), [5])
    assert tpos.cpu().numpy().tolist()[0:2] == [ni, ni] and tpos.cpu().numpy()[2] == ni
