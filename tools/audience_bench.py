"""Audiences (mr_catalogue_audience): the k best users of every item over the whole user base, timed alternately with
the full-catalogue top-k (mr_catalogue_topk) on the same seeded weights, plus the cold-start shape (100 folded-in items
x all users).  GPU only.

Workload shapes of bench.py; k = 10; exclusion lists = the per-item raters of the synthetic ratings (bench.synth_ratings)
for audiences, the per-user lists for the top-k.  CUDA events around each call after a warm-up call; the two calls
alternate `reps` times in one process.  Before any number is printed, the audiences of >= 8 sampled items are checked
against the NumPy reference (tests/audience_oracle.py on the kernel's scores, which must equal mr_catalogue_topk's bit
for bit; the scores of sampled users against oracle.forward); a failed check exits non-zero.  With --quality: audience
HR@10 of held-out raters on the planted clusters of tests/test_gpu_fold_in_items.py, for folded-in rows, zero rows and
mean rows.  Prints one JSON line.

    python tools/audience_bench.py --workload ml-20m [--reps 3] [--quality]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "movierecommender-tf-trt_b200"), os.path.join(ROOT, "tests")]

import torch  # noqa: E402

import bench  # noqa: E402
from audience_oracle import audience  # noqa: E402
from movierec import _engine, _native as nat  # noqa: E402
from oracle import movierec_oracle as o  # noqa: E402


def gpu_info():
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def phases(fn):
    nat.profile_begin()
    fn()
    ph, launches = nat.profile_end()
    ph = {k: round(v[0], 4) for k, v in ph.items() if v[1]}
    return ph, launches, (round(ph.get("rank", 0.0) / sum(ph.values()), 4) if ph else None)


def quality():
    """Audience HR@10 / NDCG@10 of the held-out (new item, rater) pairs of the planted clusters."""
    import tempfile
    import test_gpu_fold_in_items as t
    eng, setup = t.planted_items_setup(_engine)
    with tempfile.TemporaryDirectory() as tmp:
        mr = t.planted_items_model(eng, setup, tmp)
        ni = setup["num_items"]
        items = np.concatenate([np.full(len(x), ni + j, np.int32) for j, x in enumerate(setup["test"])])
        users = np.concatenate([np.asarray(x, np.int32) for x in setup["test"]])
        lists = [np.int32([])] * ni + [np.asarray(f, np.int32) for f in setup["fold"]]
        rowptr = np.concatenate([[0], np.cumsum([len(x) for x in lists])]).astype(np.int64)
        excl = (rowptr, np.concatenate(lists).astype(np.int32))
        out = {}
        for name, model in (("folded", mr.fold_in_items(setup["fold"], seed=3)),
                            ("zero_rows", mr.fold_in_items(setup["fold"], steps=0)),
                            ("mean_rows", t.mean_rows_model(mr, t.HELD_ITEMS))):
            hr, ndcg = model.evaluate_item_audiences(items, users, exclude=excl, k=10)
            out[name] = {"hr@10": round(float(hr), 4), "ndcg@10": round(float(ndcg), 4)}
        out["pairs"] = int(items.size)
        return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="ml-20m", choices=["ml-20m", "ml-1m"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--check-items", type=int, default=8)
    ap.add_argument("--cold-items", type=int, default=100)
    ap.add_argument("--quality", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("audience_bench: needs a CUDA device")
    wl = bench.WORKLOADS[args.workload]
    nu, ni, k = wl["num_users"], wl["num_items"], args.k
    dev = torch.device("cuda")
    eng = _engine.NeuMFEngine(nu, ni, wl["layers"], [0] * len(wl["layers"]), mf_dim=wl["mf_dim"], seed=1)
    ru, ri = bench.synth_ratings(wl, 0)
    u_rowptr, u_lists = _engine.build_user_csr(ru, ri, nu, ni)
    i_rowptr, i_lists = _engine.build_user_csr(ri, ru, ni, nu)
    rng = np.random.default_rng(2)
    all_users = torch.arange(nu, dtype=torch.int32, device=dev)
    all_items = torch.arange(ni, dtype=torch.int32, device=dev)
    u_targets = torch.from_numpy(rng.integers(0, ni, nu).astype(np.int32)).to(dev)
    i_targets = torch.from_numpy(rng.integers(0, nu, ni).astype(np.int32)).to(dev)

    def aud():
        return eng.catalogue_audience(all_items, k, exclude=(i_rowptr, i_lists), targets=i_targets)

    def top():
        return eng.catalogue_topk(all_users, k, exclude=(u_rowptr, u_lists), targets=u_targets)

    # oracle check: sampled items' audiences from their own scores, which must be mr_catalogue_topk's
    check = np.sort(rng.choice(ni, args.check_items, replace=False)).astype(np.int32)
    a_users, a_scores, a_pos, _ = aud()[:4]
    c = eng.catalogue_audience(check, k, exclude=(i_rowptr, i_lists), targets=i_targets[check], want_scores=True)
    p = c[4].cpu().numpy()
    rp, li = i_rowptr.cpu().numpy(), i_lists.cpu().numpy()
    want = audience(p, k, num_users=nu, excl_rowptr=rp, excl_users=li, excl_ids=check,
                    targets=i_targets.cpu().numpy()[check])
    su = np.sort(rng.choice(nu, 8, replace=False)).astype(np.int32)
    t_full = eng.catalogue_topk(su, k, want_scores=True)[4].cpu().numpy()[:, check]
    w = eng.get_weights()
    p_or = o.forward({n: np.asarray(v, np.float64) for n, v in w.items()}, np.repeat(su, check.size),
                     np.tile(check, su.size))["p"].reshape(su.size, check.size)
    ok = (np.array_equal(c[0].cpu().numpy(), want[0]) and np.array_equal(c[2].cpu().numpy(), want[2])
          and np.array_equal(c[1].cpu().numpy().view(np.int32), want[1].view(np.int32))
          and np.array_equal(a_users.cpu().numpy()[check], want[0]) and np.array_equal(a_pos.cpu().numpy()[check], want[2])
          and np.array_equal(a_scores.cpu().numpy()[check].view(np.int32), want[1].view(np.int32))
          and np.array_equal(p[su].view(np.int32), t_full.view(np.int32))
          and float(np.max(np.abs(p[su] - p_or))) <= 1e-5 * float(np.max(np.abs(p_or))) + 1e-6)
    if not ok:
        sys.exit("audience_bench: oracle check FAILED on items {}".format(check.tolist()))

    # cold start: new items folded in from the raters of existing items, then their audiences over all users
    M = args.cold_items
    src = np.sort(rng.choice(ni, M, replace=False))
    raters = [li[rp[j]:rp[j + 1]] for j in src]
    mlp, gmf, _ = eng.fold_in_items(raters, 2, 0.05, 4, seed=1)
    view = eng.item_view(mlp, gmf)
    new = torch.arange(ni, ni + M, dtype=torch.int32, device=dev)
    cold_rp = np.concatenate([np.zeros(ni, np.int64), np.concatenate([[0], np.cumsum([r.size for r in raters])])])
    cold_excl = (torch.from_numpy(cold_rp).to(dev), torch.from_numpy(np.concatenate(raters).astype(np.int32)).to(dev))

    def cold():
        return view.catalogue_audience(new, k, exclude=cold_excl)

    for fn in (aud, top, cold):
        fn()
    torch.cuda.synchronize()
    t_aud, t_top, t_cold = [], [], []
    for _ in range(args.reps):
        t_aud.append(event_ms(aud))
        t_top.append(event_ms(top))
        t_cold.append(event_ms(cold))
    aud_ph, aud_launch, aud_share = phases(aud)
    top_ph, _, top_share = phases(top)
    cold_ph, cold_launch, cold_share = phases(cold)
    name, power = gpu_info()
    pairs = nu * ni
    a_ms, t_ms, c_ms = float(np.median(t_aud)), float(np.median(t_top)), float(np.median(t_cold))
    out = {
        "tool": "audience_bench", "workload": args.workload, "gpu": name, "power_limit": power,
        "users": nu, "items": ni, "k": k, "layers": wl["layers"], "mf_dim": wl["mf_dim"], "reps": args.reps,
        "excluded_pairs": int(li.size),
        "audience_ms": round(a_ms, 3), "audience_ms_runs": [round(x, 3) for x in t_aud],
        "audience_pairs_per_s": pairs / (a_ms / 1e3), "audience_phase_ms": aud_ph,
        "audience_kernel_launches": aud_launch, "audience_selection_share": aud_share,
        "catalogue_topk_ms": round(t_ms, 3), "catalogue_topk_ms_runs": [round(x, 3) for x in t_top],
        "catalogue_topk_phase_ms": top_ph, "catalogue_topk_selection_share": top_share,
        "audience_over_topk": round(a_ms / t_ms, 4),
        "cold_items": M, "cold_ms": round(c_ms, 3), "cold_ms_runs": [round(x, 3) for x in t_cold],
        "cold_pairs_per_s": nu * M / (c_ms / 1e3), "cold_phase_ms": cold_ph, "cold_kernel_launches": cold_launch,
        "cold_selection_share": cold_share,
        "oracle_check_items": check.tolist(), "oracle_check": "passed",
    }
    if args.quality:
        out["planted_quality"] = quality()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
