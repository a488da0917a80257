"""The update half of the train step against plain references, on one GPU: out-of-range ids in the sort and the
segmented reduction, the owner-side sparse-row update, the flat optimizer sweep, the data-parallel exchange kernel on
emulated ranks (W gradient buffers and W parameter replicas on one device: a peer pointer is just a device pointer)
and the row-sharded gather.

Comparison rule (test_gpu_parity.close_to_truth): the float64 truth, calibrated by an fp32 evaluation's own distance
from it; wherever the arithmetic is fixed, bit equality as well."""

import ctypes as C

import numpy as np
import pytest

from test_gpu_parity import OraclePair, check_step_against_oracles, close_to_truth, make_batch

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

INT32_MIN, INT32_MAX = -2 ** 31, 2 ** 31 - 1
B1, B2, EPS = 0.9, 0.999, 1e-7


@pytest.fixture(scope="module")
def eng_mod():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from movierec import _engine
    return _engine


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _bits(a):
    """float32 array -> its bit patterns (NaN-safe bitwise comparison)."""
    return np.ascontiguousarray(np.asarray(a, np.float32)).view(np.int32)


def _same(a, b, what):
    a, b = _bits(a), _bits(b)
    assert a.shape == b.shape, what
    bad = np.flatnonzero(a.reshape(-1) != b.reshape(-1))
    assert bad.size == 0, "{}: {} elements differ, first at {}".format(what, bad.size, bad[:5])


def _lr_t(lr, t):
    """Adam's step size as the C side computes it (float-valued hyper-parameters, double arithmetic) -> float32."""
    f = lambda x: float(np.float32(x))
    return f(f(lr) * np.sqrt(1.0 - f(B2) ** t) / (1.0 - f(B1) ** t))


# ---- out-of-range ids -------------------------------------------------------------------------------------------------
# The row-id sort used to run ceil(bits_for(num_rows) / 8) 8-bit passes over the RAW ids, so an out-of-range id sorted
# among the entries of the valid id that shares its low 8 * passes bits and split that id's run in the segmented
# reduction: two partial sums written to one gradient row (dense tables) or two updates of one row (sparse tables).

def old_sort_bits(n):
    """Key bits the row-id sort covered before out-of-range ids were mapped to a sentinel: whole 8-bit digits over
    the bits of the largest valid id."""
    b = 1
    while b < 31 and (1 << b) < n:
        b += 1
    return 8 * ((b + 7) // 8)


def alias_of(x, n):
    """The valid id that out-of-range id x shares its sorted bits with in a table of n rows, or None."""
    low = x & ((1 << old_sort_bits(n)) - 1)
    return low if low < n else None


BAD_KINDS = ["plus", "int32_min", "minus_one", "int32_max"]


def bad_id(kind, n, hot):
    """(out-of-range id, the valid id it aliases or None)."""
    x = {"plus": hot + (1 << old_sort_bits(n)), "int32_min": INT32_MIN, "minus_one": -1, "int32_max": INT32_MAX}[kind]
    return x, alias_of(x, n)


def place_around(ids, pos_bad, x, a, many, n, rng):
    """ids with x at pos_bad and the valid id a many (runs across 32-entry chunks) or a few (one chunk) times both
    before and after it in arrival order; a appears nowhere else."""
    ids = ids.copy()
    ids[ids == a] = (a + 1) % n if n > 1 else a
    if many:
        before, after = np.arange(0, pos_bad, 3), np.arange(pos_bad + 1, len(ids), 3)
    else:
        before, after = np.array([pos_bad - 5, pos_bad - 2]), np.array([pos_bad + 1, pos_bad + 4])
    ids[before] = a
    ids[after] = a
    ids[pos_bad] = x
    return ids


def aliasing_batch(rng, nu, ni, groups, negs, kind, many):
    """A grouped batch with one aliasing bad id on the item side and one (a whole group) on the user side, and its twin
    with the bad ids replaced by the non-aliasing num_rows + 1."""
    users, items, y = make_batch(rng, nu, ni, groups, negs)
    g = negs + 1
    xi, ai = bad_id(kind, ni, hot=7 % ni)
    xu, au = bad_id(kind, nu, hot=5 % nu)
    if ai is None:  # kind has no valid alias in this table: the bad id still has to leave the step as its twin does
        ai = 7 % ni
    if au is None:
        au = 5 % nu
    items = place_around(items, len(items) // 2 + 2, xi, ai, many, ni, rng)
    ug = place_around(users[::g], groups // 2, xu, au, many, nu, rng)
    users = np.repeat(ug, g)
    tw_items, tw_users = items.copy(), users.copy()
    tw_items[items == xi] = ni + 1
    tw_users[users == xu] = nu + 1
    return (users, items, y), (tw_users, tw_items, y)


# (name, (num_users, num_items, layers, mf_dim), engine kwargs, grouped, table modes, path check)
ALIAS_PATHS = [
    ("fused", (256, 256, [256, 128, 64], 64), {}, True, ("dense",),
     lambda e, B, g: e.uses_user_projection(B, g)),
    ("tc-unfused", (256, 256, [256, 128, 64], 64), {"fused_train": "off"}, True, ("dense", "sparse"),
     lambda e, B, g: e.uses_tensor_cores()),
    ("tc-per-row", (256, 256, [256, 128, 64], 64), {"item_projection": "off"}, False, ("dense", "sparse"),
     lambda e, B, g: e.uses_tensor_cores() and not e.uses_item_projection(B)),
    ("small-tower", (256, 256, [64, 32, 16, 8], 8), {}, True, ("dense",),
     lambda e, B, g: e.uses_small_tower(B, g)),
    ("simt", (256, 700, [9, 5, 3], 3), {}, False, ("dense", "sparse"),
     lambda e, B, g: not e.uses_tensor_cores()),
]
ALIAS_CASES = [(p, mode, kind) for p in ALIAS_PATHS for mode in p[4] for kind in BAD_KINDS]


def _step_record(eng, batch, grouped, negs):
    users, items, y = batch
    out = eng.train_grads(users, items, y, group=negs + 1, k=3, grouped=grouped).cpu().numpy()
    rec = {"step_out": out, "g_dense": eng.g_dense.cpu().numpy()}
    for k, t in eng.g_tables.items():
        rec["g " + k] = t.cpu().numpy()
    eng.apply()
    for k, w in eng.get_weights().items():
        rec["w " + k] = w
    st = eng.get_optimizer_state()
    for k in st:
        if k != "iterations":
            rec["state " + k] = st[k]
    return rec


@pytest.mark.parametrize("case", ALIAS_CASES, ids=lambda c: "{}-{}-{}".format(c[0][0], c[1], c[2]))
def test_aliasing_bad_ids_leave_the_step_as_a_non_aliasing_bad_id_does(eng_mod, case):
    (name, (nu, ni, L, f), kw, grouped, _, selected), mode, kind = case
    negs, groups = 4, 600
    B = groups * (negs + 1)
    engines = [eng_mod.NeuMFEngine(nu, ni, L, [0] * len(L), mf_dim=f, optimizer="adam", lr=0.01, table_mode=mode,
                                   seed=3, **kw) for _ in range(3)]
    assert selected(engines[0], B, negs + 1), name
    rng = np.random.default_rng(BAD_KINDS.index(kind))
    for step, many in enumerate((True, False)):
        batch, twin = aliasing_batch(rng, nu, ni, groups, negs, kind, many)
        got = _step_record(engines[0], batch, grouped, negs)
        again = _step_record(engines[1], batch, grouped, negs)
        want = _step_record(engines[2], twin, grouped, negs)
        assert int(got["step_out"][4]) & 1, "bad ids not flagged"
        for k in want:
            _same(got[k], want[k], "{} step {}: {} vs non-aliasing twin".format(name, step, k))
            _same(got[k], again[k], "{} step {}: {} run twice".format(name, step, k))


# ---- mr_sparse_rows_update ----------------------------------------------------------------------------------------------

def sparse_state(rng, num_rows, d0, d1, adam):
    mk = lambda d, s: torch.from_numpy(rng.normal(0, s, (num_rows, d)).astype(np.float32)).cuda() if d else None
    p = [mk(d0, 0.1), mk(d1, 0.1)]
    m = [mk(d0, 0.01), mk(d1, 0.01)] if adam else [None, None]
    v = [None, None]
    if adam:
        v = [torch.from_numpy(rng.uniform(0, 1e-3, (num_rows, d)).astype(np.float32)).cuda() if d else None
             for d in (d0, d1)]
    return p, m, v


def run_sparse(nat, p, m, v, d0, d1, num_rows, ids, grads, adam, lr, lr_t):
    n = int(ids.numel())
    nbytes = max(int(nat.lib.mr_sparse_rows_workspace_bytes(n, d0, d1)), 256)
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    nat.check(nat.lib.mr_sparse_rows_update(_p(p[0]), _p(m[0]), _p(v[0]), d0, _p(p[1]), _p(m[1]), _p(v[1]), d1, num_rows,
                                            _p(ids), _p(grads), n, nat.OPT_ADAM if adam else nat.OPT_SGD, lr, lr_t, B1,
                                            B2, EPS, _p(ws), nbytes, _stream()), "mr_sparse_rows_update")
    torch.cuda.synchronize()


def _host(ts):
    return [t.cpu().numpy() if t is not None else None for t in ts]


def _clone(ts):
    return [t.clone() if t is not None else None for t in ts]


def _sparse_ids(rng, n, num_rows, pattern):
    if pattern == "same":
        return np.full(n, min(17, num_rows - 1), np.int32)
    ids = rng.integers(0, num_rows, n).astype(np.int32)
    if pattern == "zipf":  # one hot id owning ~10^5 pairs, scattered through the list
        ids[rng.choice(n, 100000, replace=False)] = 123
    return ids


SPARSE_CASES = [
    # n, num_rows, d0, d1, optimizer, t, id pattern
    (1, 300, 64, 64, "adam", 1, "uniform"),
    (31, 300, 6, 3, "adam", 3, "uniform"),
    (33, 1, 4, 2, "sgd", 0, "uniform"),          # one row: every pair on it
    (5000, 300, 64, 64, "adam", 3, "uniform"),
    (5000, 70000, 128, 0, "sgd", 0, "uniform"),  # three sort passes
    (5000, 1, 128, 0, "adam", 1, "uniform"),
    (2 ** 21 + 7, 300, 4, 2, "adam", 1, "uniform"),  # several levels of the recursive reduction, scalar path
    (200000, 70000, 64, 64, "adam", 3, "zipf"),
    (100000, 300, 6, 3, "sgd", 0, "same"),
]


@pytest.mark.parametrize("case", SPARSE_CASES, ids=lambda c: "n{}-rows{}-d{}x{}-{}{}-{}".format(*c))
def test_sparse_rows_update_matches_float64(eng_mod, case):
    nat = eng_mod.nat
    n, num_rows, d0, d1, opt, t, pattern = case
    adam = opt == "adam"
    lr = 0.01
    lr_t = _lr_t(lr, t) if adam else lr
    rng = np.random.default_rng(n + num_rows)
    ids_h = _sparse_ids(rng, n, num_rows, pattern)
    g_h = rng.normal(0, 1, (n, d0 + d1)).astype(np.float32)
    p, m, v = sparse_state(rng, num_rows, d0, d1, adam)
    p_in, m_in, v_in = _host(p), _host(m), _host(v)
    ids, grads = torch.from_numpy(ids_h).cuda(), torch.from_numpy(g_h).cuda()
    runs = []
    for _ in range(2):
        pr, mr, vr = _clone(p), _clone(m), _clone(v)
        run_sparse(nat, pr, mr, vr, d0, d1, num_rows, ids, grads, adam, lr, lr_t)
        runs.append((_host(pr), _host(mr), _host(vr)))
    for a, b in zip(runs[0], runs[1]):
        for x, y in zip(a, b):
            if x is not None:
                _same(x, y, "two calls from the same state")
    cnt = np.bincount(ids_h, minlength=num_rows)
    touched = cnt > 0
    col0 = 0
    for j, d in enumerate((d0, d1)):
        if d == 0:
            continue
        gsum = np.stack([np.bincount(ids_h, weights=g_h[:, col0 + c].astype(np.float64), minlength=num_rows)
                         for c in range(d)], axis=1)
        gabs = np.stack([np.bincount(ids_h, weights=np.abs(g_h[:, col0 + c]).astype(np.float64), minlength=num_rows)
                         for c in range(d)], axis=1)
        col0 += d
        got_p = runs[0][0][j]
        # untouched rows: bitwise unchanged
        _same(got_p[~touched], p_in[j][~touched], "untouched rows of table {}".format(j))
        if adam:
            _same(runs[0][1][j][~touched], m_in[j][~touched], "untouched rows of m{}".format(j))
            _same(runs[0][2][j][~touched], v_in[j][~touched], "untouched rows of v{}".format(j))
        # touched rows: float64 truth; the fp32 reference applies the update in fp32 to the exact sum rounded once
        # slack: the tree sum's own error (~log2(count) roundings of sum |g|) pushed through the update
        sum_tol = (np.ceil(np.log2(np.maximum(cnt, 1)))[:, None] + 1) * 2.0 ** -24 * gabs
        gs64, gs32 = gsum[touched], gsum[touched].astype(np.float32)
        p64, p32 = p_in[j][touched].astype(np.float64), p_in[j][touched]
        if adam:
            m64 = B1 * m_in[j][touched].astype(np.float64) + (1 - B1) * gs64
            v64 = B2 * v_in[j][touched].astype(np.float64) + (1 - B2) * gs64 * gs64
            ref64 = p64 - lr_t * m64 / (np.sqrt(v64) + EPS)
            f = np.float32
            m32 = f(B1) * m_in[j][touched] + (f(1) - f(B1)) * gs32
            v32 = f(B2) * v_in[j][touched] + (f(1) - f(B2)) * gs32 * gs32
            ref32 = p32 - f(lr_t) * m32 / (np.sqrt(v32) + f(EPS))
            sv = np.sqrt(v64)
            jac = lr_t * ((1 - B1) / (sv + EPS) - m64 * (1 - B2) * gs64 / (np.maximum(sv, 1e-300) * (sv + EPS) ** 2))
            close_to_truth(runs[0][1][j][touched], m32, m64, "m{}".format(j),
                           slack=(1 - B1) * sum_tol[touched])
            close_to_truth(runs[0][2][j][touched], v32, v64, "v{}".format(j),
                           slack=(1 - B2) * 2 * np.abs(gs64) * sum_tol[touched])
        else:
            ref64 = p64 - lr_t * gs64
            ref32 = p32 - np.float32(lr_t) * gs32
            jac = np.full(gs64.shape, lr_t)
        close_to_truth(got_p[touched], ref32, ref64, "table {}".format(j), slack=np.abs(jac) * sum_tol[touched])


@pytest.mark.parametrize("num_rows", [256, 300, 70000])
@pytest.mark.parametrize("kind", BAD_KINDS)
def test_sparse_rows_update_ignores_aliasing_bad_ids(eng_mod, num_rows, kind):
    nat = eng_mod.nat
    rng = np.random.default_rng(num_rows)
    for (d0, d1), adam, many in (((64, 64), True, True), ((6, 3), True, False), ((128, 0), False, True)):
        n = 5000
        x, a = bad_id(kind, num_rows, hot=11)
        if a is None:
            a = 11
        ids_h = place_around(rng.integers(0, num_rows, n).astype(np.int32), n // 2, x, a, many, num_rows, rng)
        twin_h = ids_h.copy()
        twin_h[ids_h == x] = num_rows + 1
        g = torch.from_numpy(rng.normal(0, 1, (n, d0 + d1)).astype(np.float32)).cuda()
        p, m, v = sparse_state(rng, num_rows, d0, d1, adam)
        res = []
        for ids_x in (ids_h, twin_h, ids_h):
            pr, mr, vr = _clone(p), _clone(m), _clone(v)
            run_sparse(nat, pr, mr, vr, d0, d1, num_rows, torch.from_numpy(ids_x).cuda(), g, adam, 0.01,
                       _lr_t(0.01, 2) if adam else 0.01)
            res.append(_host(pr) + _host(mr) + _host(vr))
        for i, (got, want, again) in enumerate(zip(*res)):
            if got is not None:
                _same(got, want, "d={} buffer {}: aliasing bad id vs non-aliasing twin".format((d0, d1), i))
                _same(got, again, "d={} buffer {}: run twice".format((d0, d1), i))


# ---- mr_optimizer_flat --------------------------------------------------------------------------------------------------

def flat_reference(p, g, m, v, adam, lr_t, l2):
    """(fp32 reference, float64 truth) of one flat sweep: (p, m, v) each."""
    f = np.float32
    g32 = g + f(2 * l2) * p if l2 else g.copy()
    g64 = g.astype(np.float64) + 2 * float(f(l2)) * p.astype(np.float64) if l2 else g.astype(np.float64)
    if not adam:
        return (p - f(lr_t) * g32, None, None), (p.astype(np.float64) - lr_t * g64, None, None)
    m32 = f(B1) * m + (f(1) - f(B1)) * g32
    v32 = f(B2) * v + (f(1) - f(B2)) * g32 * g32
    m64 = B1 * m.astype(np.float64) + (1 - B1) * g64
    v64 = B2 * v.astype(np.float64) + (1 - B2) * g64 * g64
    return ((p - f(lr_t) * m32 / (np.sqrt(v32) + f(EPS)), m32, v32),
            (p.astype(np.float64) - lr_t * m64 / (np.sqrt(v64) + EPS), m64, v64))


@pytest.mark.parametrize("n", [0, 1, 3, 4, 5, 1023, 2 ** 20 + 3])
def test_optimizer_flat_vector_and_scalar_paths(eng_mod, n):
    nat = eng_mod.nat
    rng = np.random.default_rng(n)
    canary = np.float32(-777.0)
    for adam in (True, False):
        for l2 in (0.0, 0.01):
            lr_t = _lr_t(0.01, 2) if adam else 0.01
            host = {"p": rng.normal(0, 0.1, n), "g": rng.normal(0, 1, n), "m": rng.normal(0, 0.01, n),
                    "v": rng.uniform(0, 1e-3, n)}
            host = {k: x.astype(np.float32) for k, x in host.items()}
            outs = {}
            for shift in (0, 1):  # 16-byte aligned buffers, and buffers one float off (the launcher's scalar path)
                bufs = {}
                for k, x in host.items():
                    b = torch.full((n + 8,), float(canary), dtype=torch.float32, device="cuda")
                    b[shift:shift + n] = torch.from_numpy(x).cuda()
                    bufs[k] = b
                    assert (b[shift:].data_ptr() % 16 == 0) == (shift == 0)
                view = lambda k: bufs[k][shift:]
                nat.check(nat.lib.mr_optimizer_flat(_p(view("p")), _p(view("g")), _p(view("m")) if adam else None,
                                                    _p(view("v")) if adam else None, n,
                                                    nat.OPT_ADAM if adam else nat.OPT_SGD, lr_t, B1, B2, EPS, l2,
                                                    _stream()), "mr_optimizer_flat")
                torch.cuda.synchronize()
                res = {k: b.cpu().numpy() for k, b in bufs.items()}
                for k, b in res.items():  # nothing outside [0, n) is touched
                    _same(np.delete(b, np.arange(shift, shift + n)), np.full(n + 8 - n, canary), "canary " + k)
                outs[shift] = {k: b[shift:shift + n] for k, b in res.items()}
            what = "adam" if adam else "sgd"
            for k in ("p", "m", "v") if adam else ("p",):
                _same(outs[0][k], outs[1][k], "{} l2={} {}: vector vs scalar path".format(what, l2, k))
            _same(outs[0]["g"], host["g"], "gradient is read only")
            if n == 0:
                continue
            ref32, ref64 = flat_reference(host["p"], host["g"], host["m"], host["v"], adam, lr_t, l2)
            for i, k in enumerate(("p", "m", "v") if adam else ("p",)):
                close_to_truth(outs[0][k], ref32[i], ref64[i], "{} l2={} {} n={}".format(what, l2, k, n))


# ---- mr_dp_reduce_apply on emulated ranks -----------------------------------------------------------------------------

def peer_array(ts, order=None):
    order = list(range(len(ts))) if order is None else order
    return (C.c_void_p * len(ts))(*[ts[r].data_ptr() for r in order])


def dp_call(nat, gp, pp, world, rank, m, v, lo, hi, adam, lr_t, l2):
    return nat.lib.mr_dp_reduce_apply(gp, pp, world, rank, _p(m) if adam else None, _p(v) if adam else None, lo, hi,
                                      nat.OPT_ADAM if adam else nat.OPT_SGD, lr_t, B1, B2, EPS, l2, None, None,
                                      _stream())


def dp_exchange(nat, grads, params, ms, vs, slices, adam, lr_t, order=None, skip_rank=None, drop_l2=False):
    """Every emulated rank's launches over its owner slices (what DataParallelNeuMF._reduce_apply issues); the
    perturbations are there to show that the checks below notice them."""
    W = len(grads)
    for r in range(W):
        if r == skip_rank:
            continue
        gp, pp = peer_array(grads, order), peer_array(params, order)
        for lo, hi, l2, _ in slices[r]:
            nat.check(dp_call(nat, gp, pp, W, r, ms[r] if adam else None, vs[r] if adam else None, lo, hi, adam, lr_t,
                              0.0 if drop_l2 else l2), "mr_dp_reduce_apply")
    torch.cuda.synchronize()


def dp_expected(nat, grads, p0, m0, v0, regions, adam, lr_t):
    """mr_optimizer_flat over every region on the fp32 rank-order sum g0 + g1 + ... + g(W-1) (torch adds)."""
    gsum = grads[0].clone()
    for g in grads[1:]:
        gsum += g
    p, m, v = p0.clone(), m0.clone() if adam else None, v0.clone() if adam else None
    for _, off, count, l2 in regions:
        sl = slice(off, off + count)
        nat.check(nat.lib.mr_optimizer_flat(_p(p[sl]), _p(gsum[sl]), _p(m[sl]) if adam else None,
                                            _p(v[sl]) if adam else None, count, nat.OPT_ADAM if adam else nat.OPT_SGD,
                                            lr_t, B1, B2, EPS, l2, _stream()), "mr_optimizer_flat")
    torch.cuda.synchronize()
    return p, m, v


def check_dp(params, ms, vs, slices, regions, want, p0, m0, v0, adam):
    """Replicas bit-identical and equal to `want` on the regions, untouched elsewhere; every rank's m / v equal to
    `want` on its own slices and untouched elsewhere."""
    W = len(params)
    got = [x.cpu().numpy() for x in params]
    for r in range(1, W):
        _same(got[r], got[0], "replica {} vs replica 0".format(r))
    inside = np.zeros(got[0].size, bool)
    for _, off, count, _ in regions:
        inside[off:off + count] = True
    wp = want[0].cpu().numpy()
    _same(got[0][inside], wp[inside], "replicas vs optimizer_flat on the rank-order sum")
    _same(got[0][~inside], p0.cpu().numpy()[~inside], "parameter padding between regions")
    if adam:
        for r in range(W):
            own = np.zeros(got[0].size, bool)
            for lo, hi, _, _ in slices[r]:
                own[lo:hi] = True
            for buf, w, init, tag in ((ms[r], want[1], m0, "m"), (vs[r], want[2], v0, "v")):
                b = buf.cpu().numpy()
                _same(b[own], w.cpu().numpy()[own], "rank {} {} on its slices".format(r, tag))
                _same(b[~own], init.cpu().numpy()[~own], "rank {} {} outside its slices".format(r, tag))


def synthetic_regions():
    """Regions of 4, 64 and 2^20 + 64 elements, 64-float (256-byte) aligned, with canary gaps between them."""
    regions, off = [], 64
    for count, l2 in ((4, 0.01), (64, 0.0), (2 ** 20 + 64, 0.02)):
        regions.append(("r{}".format(count), off, count, l2))
        off = (off + count + 63) // 64 * 64 + 64
    return regions, off


def engine_regions(eng_mod):
    eng = eng_mod.NeuMFEngine(300, 200, [256, 128, 64], [0.01, 0, 0], mf_dim=64, seed=1)
    eng.rebind_flat()
    return eng.flat_regions(), eng.g_flat.numel()


def dp_setup(rng, W, total, adam):
    mk = lambda x: torch.from_numpy(x.astype(np.float32)).cuda()
    p0 = mk(rng.normal(0, 0.1, total))
    grads = [mk(rng.normal(0, 1e-2, total)) for _ in range(W)]
    m0 = mk(rng.normal(0, 1e-3, total)) if adam else None
    v0 = mk(rng.uniform(0, 1e-4, total)) if adam else None
    return p0, grads, m0, v0


def run_dp_case(eng_mod, W, regions, total, adam, rng, **perturb):
    from movierec import _distributed
    nat = eng_mod.nat
    p0, grads, m0, v0 = dp_setup(rng, W, total, adam)
    inside = np.zeros(total, bool)
    for _, off, count, _ in regions:
        inside[off:off + count] = True
    gap = torch.from_numpy(~inside).cuda()
    for t in (p0, m0, v0):  # canaries in the padding between regions
        if t is not None:
            t[gap] = 1234.5
    lr_t = _lr_t(0.01, 2) if adam else 0.01
    slices = [_distributed.owner_slices(regions, W, r, lambda name: 0) for r in range(W)]
    params = [p0.clone() for _ in range(W)]
    ms = [m0.clone() for _ in range(W)] if adam else [None] * W
    vs = [v0.clone() for _ in range(W)] if adam else [None] * W
    dp_exchange(nat, grads, params, ms, vs, slices, adam, lr_t, **perturb)
    want = dp_expected(nat, grads, p0, m0, v0, regions, adam, lr_t)
    check_dp(params, ms, vs, slices, regions, want, p0, m0, v0, adam)
    # float64 truth
    g = [x.cpu().numpy() for x in grads]
    g32 = g[0].copy()
    for x in g[1:]:
        g32 = g32 + x
    g64 = np.sum(np.stack(g).astype(np.float64), axis=0)
    got = params[0].cpu().numpy()
    ph, mh, vh = p0.cpu().numpy(), m0.cpu().numpy() if adam else None, v0.cpu().numpy() if adam else None
    for name, off, count, l2 in regions:
        sl = slice(off, off + count)
        m_sl, v_sl = (mh[sl], vh[sl]) if adam else (None, None)
        ref32, _ = flat_reference(ph[sl], g32[sl], m_sl, v_sl, adam, lr_t, l2)
        _, ref64 = flat_reference(ph[sl], g64[sl], m_sl, v_sl, adam, lr_t, l2)  # the truth sums the ranks exactly
        close_to_truth(got[sl], ref32[0], ref64[0], "region {} W={}".format(name, W))


DP_WORLDS = [1, 2, 3, 4, 5, 6, 7, 8, 16]


@pytest.mark.parametrize("regions", ["engine", "synthetic"])
@pytest.mark.parametrize("world", DP_WORLDS)
def test_dp_reduce_apply_on_emulated_ranks(eng_mod, world, regions):
    rng = np.random.default_rng(world)
    regs, total = engine_regions(eng_mod) if regions == "engine" else synthetic_regions()
    for adam in (True, False):
        run_dp_case(eng_mod, world, regs, total, adam, rng)


@pytest.mark.parametrize("perturb", [{"order": [0, 2, 1]}, {"drop_l2": True}, {"skip_rank": 1}],
                         ids=["rank-order", "no-l2", "rank-skips-slice"])
def test_dp_checks_notice_a_wrong_exchange(eng_mod, perturb):
    regs, total = synthetic_regions()
    with pytest.raises(AssertionError):
        run_dp_case(eng_mod, 3, regs, total, True, np.random.default_rng(5), **perturb)


def test_dp_reduce_apply_refusals(eng_mod):
    nat = eng_mod.nat
    bufs = [torch.zeros(256, dtype=torch.float32, device="cuda") for _ in range(9)]
    m, v = torch.zeros(256, device="cuda"), torch.zeros(256, device="cuda")
    gp, pp = peer_array(bufs[:2]), peer_array(bufs[2:4])
    MR_ERR_INVALID = -1
    assert dp_call(nat, peer_array(bufs), peer_array(bufs), 9, 0, m, v, 0, 64, True, 1e-3, 0.0) == MR_ERR_INVALID
    assert dp_call(nat, gp, pp, 2, 0, m, v, 2, 64, True, 1e-3, 0.0) == MR_ERR_INVALID   # lo % 4 != 0
    assert dp_call(nat, gp, pp, 2, 2, m, v, 0, 64, True, 1e-3, 0.0) == MR_ERR_INVALID   # rank >= world
    off = (C.c_void_p * 2)(bufs[0].data_ptr(), bufs[1].data_ptr() + 4)
    assert dp_call(nat, off, pp, 2, 0, m, v, 0, 64, True, 1e-3, 0.0) == MR_ERR_INVALID
    assert dp_call(nat, gp, off, 2, 0, m, v, 0, 64, True, 1e-3, 0.0) == MR_ERR_INVALID
    assert dp_call(nat, gp, pp, 2, 0, m[1:], v, 0, 64, True, 1e-3, 0.0) == MR_ERR_INVALID
    assert dp_call(nat, gp, pp, 2, 0, m, v[1:], 0, 64, True, 1e-3, 0.0) == MR_ERR_INVALID
    torch.cuda.synchronize()
    for b in bufs:  # nothing was launched
        assert not b.any()


# ---- a data-parallel train step on emulated ranks (the single-GPU restatement of tools/dp_gpu_check.py) ----------------

# (name, (num_users, num_items, layers, mf_dim, negs, global groups), l2, grouped, fast-path check on rank-local rows)
DP_TOWERS = [
    ("fused", (60, 40, [256, 128, 64], 64, 4, 384), [0, 0, 0], True,
     lambda e, B, g: e.uses_user_projection(B, g)),
    ("default", (60, 40, [64, 32, 16, 8], 8, 4, 384), [0, 0, 0, 0], True,
     lambda e, B, g: e.uses_small_tower(B, g)),
    ("simt", (5, 10, [6, 4], 0, 3, 12), [0.01, 0.01], False,
     lambda e, B, g: not e.uses_tensor_cores()),
]
DP_STEP_CASES = [(t, W, "adam") for t in DP_TOWERS for W in (2, 3)] + [(DP_TOWERS[1], 3, "sgd"), (DP_TOWERS[2], 2, "sgd")]


def dp_train(eng_mod, tower, W, opt, steps=3, perturb=None):
    from movierec import _distributed
    nat = eng_mod.nat
    name, (nu, ni, L, f, negs, groups), l2, grouped, fast = tower
    g = negs + 1
    lr = 0.001
    params = {"layers_sizes": L, "layers_l2reg": l2, "optimizer": opt, "lr": lr, "beta_1": B1, "beta_2": B2,
              "num_negs_per_pos": negs, "k": 2}
    engines = [eng_mod.NeuMFEngine(nu, ni, L, l2, mf_dim=f, optimizer=opt, lr=lr, table_mode="dense", seed=7)
               for _ in range(W)]
    for e in engines:
        e.rebind_flat()
    adam = opt == "adam"
    regions = engines[0].flat_regions()
    slices = [_distributed.owner_slices(regions, W, r, lambda n: 0) for r in range(W)]
    pair = OraclePair(engines[0].get_weights())
    rng = np.random.default_rng(40 + W)
    for step in range(steps):
        users, items, y = make_batch(rng, nu, ni, groups, negs)
        B = len(y)
        for r, e in enumerate(engines):
            u, i, yy = _distributed.shard_batch(users, items, y, g, W, r)
            assert fast(e, len(yy), g), "{}: rank {} of {} left the fast path".format(name, r, W)
            e.train_grads(u, i, yy, group=g, k=2, inv_global_batch=1.0 / B, grouped=grouped, dense_l2=(r == 0))
        torch.cuda.synchronize()
        lr_t = engines[0].step_lr_t()
        assert all(e.step_lr_t() == lr_t for e in engines)
        grads = [e.g_flat for e in engines]
        p0 = engines[0].p_flat.clone()
        own_m = engines[0].m_flat.clone() if adam else None  # the full Adam state, assembled from the owners
        own_v = engines[0].v_flat.clone() if adam else None
        if adam:
            for r, e in enumerate(engines):
                for lo, hi, _, _ in slices[r]:
                    own_m[lo:hi] = e.m_flat[lo:hi]
                    own_v[lo:hi] = e.v_flat[lo:hi]
        want = dp_expected(nat, grads, p0, own_m, own_v, regions, adam, lr_t)
        kw = perturb if (perturb and step == steps - 1) else {}
        dp_exchange(nat, grads, [e.p_flat for e in engines], [e.m_flat for e in engines],
                    [e.v_flat for e in engines], slices, adam, lr_t, **kw)
        for e in engines:
            e.finish_apply()
        params_now = [e.p_flat for e in engines]
        for r in range(1, W):
            assert torch.equal(params_now[r], params_now[0]), "replica {} differs".format(r)
        _same(params_now[0].cpu().numpy(), want[0].cpu().numpy(), "{} step {}: vs optimizer_flat on the rank-order sum"
              .format(name, step))
        if adam:
            for r, e in enumerate(engines):
                for lo, hi, _, _ in slices[r]:
                    _same(e.m_flat[lo:hi].cpu().numpy(), want[1][lo:hi].cpu().numpy(), "m of rank {}".format(r))
                    _same(e.v_flat[lo:hi].cpu().numpy(), want[2][lo:hi].cpu().numpy(), "v of rank {}".format(r))
        gg, g64 = pair.grads(users, items, y, l2)
        pair.step(users, items, y, params, adam_mode="dense", g64=g64)
        got = engines[0].get_weights()
        for k in pair.w:
            close_to_truth(got[k], pair.w[k], pair.w64[k], "{} W={} weight {} after step {}".format(name, W, k, step + 1),
                           slack=pair.slack[k])
    assert all(e.iterations == steps for e in engines)


@pytest.mark.parametrize("case", DP_STEP_CASES, ids=lambda c: "{}-W{}-{}".format(c[0][0], c[1], c[2]))
def test_data_parallel_step_on_emulated_ranks(eng_mod, case):
    tower, W, opt = case
    dp_train(eng_mod, tower, W, opt)


@pytest.mark.parametrize("perturb", [{"order": [0, 2, 1]}, {"drop_l2": True}, {"skip_rank": 0}],
                         ids=["rank-order", "no-l2", "rank-skips-slice"])
def test_data_parallel_step_checks_notice_a_wrong_exchange(eng_mod, perturb):
    with pytest.raises(AssertionError):
        dp_train(eng_mod, DP_TOWERS[2], 3, "adam", steps=1, perturb=perturb)


# ---- mr_gather_rows_sharded -------------------------------------------------------------------------------------------

@pytest.mark.parametrize("world", [1, 2, 3, 5, 8, 16])
def test_gather_rows_sharded_bit_exact(eng_mod, world):
    nat = eng_mod.nat
    rng = np.random.default_rng(world)
    total = 37 * world + 1 if world > 1 else 37
    rows_max = (total + world - 1) // world
    for dim in (1, 3, 4, 33, 64, 128):
        full = rng.normal(size=(total, dim)).astype(np.float32)
        shards = []
        for r in range(world):  # separate allocations: every shard base 16-byte aligned (the kernel's precondition)
            s = torch.full((rows_max, dim), float("inf"), dtype=torch.float32, device="cuda")
            mine = full[r::world]
            s[:mine.shape[0]] = torch.from_numpy(mine).cuda()
            shards.append(s)
        ptrs = torch.tensor([s.data_ptr() for s in shards], dtype=torch.int64, device="cuda")
        last_short = 36 * world + world - 1 if world > 1 else total - 1  # last row of rank W-1 (37 rows, rank 0 38)
        bad = [-1, total, INT32_MIN, INT32_MAX]
        ids_h = np.concatenate([rng.permutation(total), [total - 1, last_short], bad, rng.integers(0, total, 50)])
        ids_h = ids_h.astype(np.int32)
        ids = torch.from_numpy(ids_h).cuda()
        n = ids_h.size
        is_bad = np.isin(ids_h, bad)
        for shift in (0, 1):  # out 16-byte aligned (float4 rows when dim % 4 == 0), and one float off (scalar path)
            buf = torch.zeros(n * dim + 4, dtype=torch.float32, device="cuda")
            out = buf[shift:shift + n * dim]
            nat.check(nat.lib.mr_gather_rows_sharded(_p(ptrs), world, total, dim, _p(ids), n, _p(out), _stream()),
                      "mr_gather_rows_sharded")
            torch.cuda.synchronize()
            got = out.cpu().numpy().reshape(n, dim)
            _same(got[~is_bad], full[ids_h[~is_bad]], "W={} dim={} shift={}".format(world, dim, shift))
            assert np.isnan(got[is_bad]).all(), "W={} dim={}: bad ids must give NaN rows".format(world, dim)
            rest = buf.cpu().numpy()
            assert not rest[:shift].any() and not rest[shift + n * dim:].any(), "wrote outside out"


# ---- row-sharded step size ------------------------------------------------------------------------------------------

def test_apply_dense_only_takes_the_single_gpu_step_size(eng_mod):
    """Sparse tables: train_grads + apply_dense_only() moves the dense block exactly as train_step does (the row-sharded
    step's dense update then equals the single-GPU one)."""
    nu, ni, L, f, negs = 200, 300, [64, 32, 16, 8], 8, 4
    rng = np.random.default_rng(8)
    batches = [make_batch(rng, nu, ni, 77, negs) for _ in range(3)]
    ref = eng_mod.NeuMFEngine(nu, ni, L, [0] * 4, mf_dim=f, table_mode="sparse", lr=0.001, seed=4)
    split = eng_mod.NeuMFEngine(nu, ni, L, [0] * 4, mf_dim=f, table_mode="sparse", lr=0.001, seed=4)
    for users, items, y in batches:
        ref.train_step(users, items, y, group=negs + 1, k=2)
        split.train_grads(users, items, y, group=negs + 1, k=2)
        split.apply_dense_only()
        _same(split.dense.cpu().numpy(), ref.dense.cpu().numpy(), "dense block")
        for k, w in ref.get_weights().items():
            _same(split.get_weights()[k], w, k)
    assert split.iterations == ref.iterations == 3


# ---- the train step itself still matches the oracle on the batches above ------------------------------------------------

def test_aliasing_batches_without_bad_ids_match_the_oracle(eng_mod):
    """The hot-id layout of the aliasing batches (a valid id's run across many 32-entry chunks, with a single-chunk
    run in the next step) with the bad ids replaced by valid ones: the fused tower against the oracle pair."""
    nu, ni, L, f, negs, groups = 256, 256, [256, 128, 64], 64, 4, 600
    params = {"layers_sizes": L, "layers_l2reg": [0, 0, 0], "optimizer": "adam", "lr": 0.01, "beta_1": B1,
              "beta_2": B2, "num_negs_per_pos": negs, "k": 2}
    eng = eng_mod.NeuMFEngine(nu, ni, L, [0, 0, 0], mf_dim=f, optimizer="adam", lr=0.01, seed=3)
    pair = OraclePair(eng.get_weights())
    rng = np.random.default_rng(2)
    for step, many in enumerate((True, False)):
        (users, items, y), _ = aliasing_batch(rng, nu, ni, groups, negs, "plus", many)
        items[items >= ni] = 7
        users[users >= nu] = 5
        check_step_against_oracles(eng, pair, users, items, y, params, [0, 0, 0], "dense", step, True, 2)
