"""The GMF item gradient of the fused train step, bit for bit.

The fused kernel (tc_fused.cu) stages dz per row instead of the row's GMF item gradient (dz * w_out[:f]) * gmf_u, and
level 0 of the item-side segmented reduction (segreduce.cu) forms that product from dz and the user's GMF row.  With
w_out[f:] = 0, b_out = 0 and a zero GMF item table every logit is exactly 0, so p = 0.5 and dz = (0.5 - y) / B are
known exactly; the test then restates the products in fp32 and the reduction's fixed summation tree (chunks of 32
sorted entries, runs summed in batch order, partial sums of runs that cross a chunk reduced again by the next level)
and requires the gradient table to be equal bit for bit."""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

SKIP, NO_NEIGHBOUR = -1, -3


@pytest.fixture(scope="module")
def eng_mod():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from movierec import _engine
    return _engine


def segment_sums(keys, vals, num_rows):
    """launch_segreduce's result for sorted `keys` and rows `vals` [n, d] (float32): every level splits its entries
    into chunks of 32, sums each run in order from +0, writes a run that lies inside its chunk and hands the partial
    sums of runs that cross a chunk boundary (two slots per chunk) to the next level."""
    out = np.zeros((num_rows, vals.shape[1]), np.float32)
    keys, vals = np.asarray(keys, np.int64), np.asarray(vals, np.float32)
    while True:
        n = len(keys)
        nchunks = (n + 31) // 32
        nkeys = np.full(2 * nchunks, SKIP, np.int64)
        nvals = np.zeros((2 * nchunks, vals.shape[1]), np.float32)
        for ch in range(nchunks):
            b = 32 * ch
            ks = keys[b:b + 32]
            nvalid = len(ks)
            kprev = keys[b - 1] if b > 0 else NO_NEIGHBOUR
            knext = keys[b + 32] if b + 32 < n else NO_NEIGHBOUR
            first_inc = ks[0] != SKIP and kprev == ks[0]
            last_inc = nvalid == 32 and ks[-1] != SKIP and knext == ks[-1]
            nkeys[2 * ch] = ks[0] if first_inc else SKIP
            nkeys[2 * ch + 1] = ks[-1] if last_inc else SKIP
            s = 0
            while s < nvalid:
                t = s + 1
                while t < nvalid and ks[t] == ks[s]:
                    t += 1
                key = ks[s]
                acc = np.zeros(vals.shape[1], np.float32)
                for j in range(s, t):
                    acc = acc + (vals[b + j] if key != SKIP else np.float32(0))
                if key != SKIP and 0 <= key < num_rows:
                    inc_first, inc_last = s == 0 and first_inc, t == nvalid and last_inc
                    if not inc_first and not inc_last:
                        out[key] = acc
                    elif inc_first:
                        nvals[2 * ch] = acc
                        if inc_last:
                            nvals[2 * ch + 1] = 0
                    else:
                        nvals[2 * ch + 1] = acc
                s = t
        if nchunks == 1:
            return out
        keys, vals = nkeys, nvals


@pytest.mark.parametrize("bad_user", [False, True], ids=["ids_in_range", "one_group_with_an_out_of_range_user"])
def test_fused_step_gmf_item_gradient_is_bit_exact(eng_mod, bad_user):
    nu, ni, L, f, group = 1500, 700, [256, 128, 64], 64, 5
    B = group * 2048
    rng = np.random.default_rng(11)
    eng = eng_mod.NeuMFEngine(nu, ni, L, [0] * 3, mf_dim=f, seed=3)
    assert eng.uses_tensor_cores() and eng.uses_item_projection(B) and eng.uses_user_projection(B, group)
    w = eng.get_weights()
    w[eng_mod.K_OUT_W] = np.asarray(w[eng_mod.K_OUT_W], np.float32).copy()
    w[eng_mod.K_OUT_W].reshape(-1)[f:] = 0
    w[eng_mod.K_OUT_W].reshape(-1)[:f] = rng.normal(0, 1, f).astype(np.float32)
    w[eng_mod.K_OUT_B] = np.zeros_like(np.asarray(w[eng_mod.K_OUT_B], np.float32))
    w[eng_mod.K_GMF_ITEM] = np.zeros_like(np.asarray(w[eng_mod.K_GMF_ITEM], np.float32))
    w[eng_mod.K_GMF_USER] = rng.normal(0, 1, (nu, f)).astype(np.float32)
    eng.set_weights(w)

    group_users = rng.integers(0, nu, B // group)
    if bad_user:
        group_users[17] = nu + 5
    users = np.repeat(group_users, group).astype(np.int32)
    # a few hot items (runs across many chunks: every level of the reduction) among many rare ones
    items = np.where(rng.random(B) < 0.4, rng.integers(0, 6, B), rng.integers(0, ni, B)).astype(np.int32)
    y = np.tile([0] * (group - 1) + [1], B // group).astype(np.float32)
    out = eng.train_grads(users, items, y, group=group, k=3, grouped=True).cpu().numpy()
    torch.cuda.synchronize()
    assert (out[4] != 0) == bad_user
    got = eng.g_tables[eng_mod.K_GMF_ITEM].cpu().numpy()

    ok = users < nu
    dz = np.where(ok, (np.float32(0.5) - y) * np.float32(1.0 / B), np.float32(0)).astype(np.float32)
    w_gmf = np.asarray(w[eng_mod.K_OUT_W], np.float32).reshape(-1)[:f]
    gmf_u = np.where(ok[:, None], w[eng_mod.K_GMF_USER][np.where(ok, users, 0)], np.float32(0)).astype(np.float32)
    rows = ((dz[:, None] * w_gmf[None, :]).astype(np.float32) * gmf_u).astype(np.float32)
    order = np.argsort(items, kind="stable")
    want = segment_sums(items[order], rows[order], ni)
    assert np.count_nonzero(want) > 0
    bad = np.flatnonzero(want.view(np.int32).reshape(-1) != got.view(np.int32).reshape(-1))
    assert bad.size == 0, "{} of {} GMF item gradient elements differ, first at {}: {} vs {}".format(
        bad.size, want.size, bad[:5], got.reshape(-1)[bad[:5]], want.reshape(-1)[bad[:5]])
