"""Large-k selection (k > 256, csrc/topk_large.cu) timed next to the k <= 256 path in one run.  GPU only.

On the workload's shape with seeded weights and the per-user / per-item CSR of the synthetic ratings
(bench.synth_ratings) as exclusion lists:
  - mr_catalogue_topk over every user at each of --ks, alternated round by round, with the RANK share of each;
  - mr_catalogue_audience, every item x every user at k = 10 and K (alternated), and 100 items x every user at
    k = 10 and K (the narrow call: 100 items folded in after training);
  - mr_rank_lists, 1024 requests of 5,000 candidates, k = 256 against K.
CUDA events around each call after a warm-up call of every shape.  Before any number is printed, sampled users'
top-k / positions, sampled items' audiences and sampled lists are checked against the NumPy references
(tests/catalogue_oracle.py, audience_oracle.py, lists_oracle.py) on the kernels' own probabilities; a failed
check exits non-zero.  K = min(1000, the largest of --ks) is the k of the checks and of the audience and list
timings, so that `--ks 10,256` also measures a library without large k (the previous build, alternated with this one
in one session).  Prints one JSON line.

    python tools/topk_large_bench.py --workload ml-20m [--reps 3] [--ks 10,256,1000,4096]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "movierecommender-tf-trt_b200"), os.path.join(ROOT, "tests"),
                os.path.join(ROOT, "tools")]

import torch  # noqa: E402

import bench  # noqa: E402
from audience_oracle import audience  # noqa: E402
from catalogue_oracle import catalogue_topk  # noqa: E402
from catalogue_topk_bench import gpu_info  # noqa: E402
from lists_oracle import topk_lists  # noqa: E402
from movierec import _engine, _native as nat  # noqa: E402


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def alternated(fns, reps):
    """{name: (mean ms, rank share of one extra profiled call)}: every fn warmed up, then reps rounds of one call each."""
    for fn in fns.values():
        fn()
    torch.cuda.synchronize()
    ms = {n: [] for n in fns}
    for _ in range(reps):
        for n, fn in fns.items():
            ms[n].append(event_ms(fn))
    out = {}
    for n, fn in fns.items():
        nat.profile_begin()
        fn()
        phases, _ = nat.profile_end()
        total = sum(v[0] for v in phases.values() if v[1])
        share = phases["rank"][0] / total if total > 0 else None
        out[n] = {"ms": round(float(np.mean(ms[n])), 3), "ms_min": round(float(np.min(ms[n])), 3),
                  "ms_max": round(float(np.max(ms[n])), 3), "rank_ms": round(phases["rank"][0], 3),
                  "rank_share": round(share, 4) if share is not None else None}
    return out


def fail(what):
    sys.exit("topk_large_bench: oracle check FAILED: " + what)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="ml-20m", choices=["ml-20m", "ml-1m"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--ks", default="10,256,1000,4096")
    ap.add_argument("--no-audience", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("topk_large_bench: needs a CUDA device")
    ks = [int(x) for x in args.ks.split(",")]
    wl = bench.WORKLOADS[args.workload]
    nu, ni = wl["num_users"], wl["num_items"]
    dev = torch.device("cuda")
    eng = _engine.NeuMFEngine(nu, ni, wl["layers"], [0] * len(wl["layers"]), mf_dim=wl["mf_dim"], seed=1)
    ru, ri = bench.synth_ratings(wl, 0)
    rowptr, lists = _engine.build_user_csr(ru, ri, nu, ni)
    irowptr, iusers = _engine.build_user_csr(ri, ru, ni, nu)  # per item: its raters, ascending
    rng = np.random.default_rng(2)
    users = torch.arange(nu, dtype=torch.int32, device=dev)
    targets = torch.from_numpy(rng.integers(0, ni, nu).astype(np.int32)).to(dev)
    all_items = torch.arange(ni, dtype=torch.int32, device=dev)
    new_items = torch.from_numpy(rng.choice(ni, 100, replace=False).astype(np.int32)).to(dev)
    held = torch.from_numpy(rng.integers(0, nu, ni).astype(np.int32)).to(dev)
    rp, li = rowptr.cpu().numpy(), lists.cpu().numpy()
    irp, iu = irowptr.cpu().numpy(), iusers.cpu().numpy()
    K = min(1000, max(ks))

    # checks at k = K on the kernels' own probabilities
    check = np.sort(rng.choice(nu, 8, replace=False)).astype(np.int32)
    top, top_s, pos = eng.catalogue_topk(users, K, exclude=(rowptr, lists), targets=targets)[:3]
    c = eng.catalogue_topk(check, K, exclude=(rowptr, lists), targets=targets[check], want_scores=True)
    w = catalogue_topk(c[4].cpu().numpy(), K, rp, li, excl_ids=check, targets=targets.cpu().numpy()[check])
    if not (np.array_equal(top.cpu().numpy()[check], w[0]) and np.array_equal(pos.cpu().numpy()[check], w[2])
            and np.array_equal(top_s.cpu().numpy()[check].view(np.int32), w[1].view(np.int32))):
        fail("catalogue_topk users {}".format(check.tolist()))
    del top, top_s, pos, c
    ccols = np.sort(rng.choice(ni, 4, replace=False)).astype(np.int32)
    a = eng.catalogue_audience(ccols, K, exclude=(irowptr, iusers), targets=held[ccols], want_scores=True)
    wa = audience(a[4].cpu().numpy(), K, num_users=nu, excl_rowptr=irp, excl_users=iu, excl_ids=ccols,
                  targets=held.cpu().numpy()[ccols])
    if not (np.array_equal(a[0].cpu().numpy(), wa[0]) and np.array_equal(a[2].cpu().numpy(), wa[2])
            and np.array_equal(a[1].cpu().numpy().view(np.int32), wa[1].view(np.int32))):
        fail("catalogue_audience items {}".format(ccols.tolist()))
    del a
    if not args.no_audience:
        full = eng.catalogue_audience(all_items, K, exclude=(irowptr, iusers), targets=held)
        if not (np.array_equal(full[0].cpu().numpy()[ccols], wa[0])
                and np.array_equal(full[2].cpu().numpy()[ccols], wa[2])):
            fail("catalogue_audience over every item, items {}".format(ccols.tolist()))
        del full
    R, L = 1024, 5000
    lu = torch.from_numpy(rng.integers(0, nu, R).astype(np.int32)).to(dev)
    lrowptr = torch.arange(0, (R + 1) * L, L, dtype=torch.int64, device=dev)
    litems = torch.from_numpy(rng.integers(0, ni, R * L).astype(np.int32)).to(dev)
    ltargets = torch.from_numpy(rng.integers(0, L, R).astype(np.int32)).to(dev)
    r = eng.rank_lists(lu, (lrowptr, litems), K, targets=ltargets, want_probs=True)
    wl_ = topk_lists(r[5].cpu().numpy(), lrowptr.cpu().numpy(), K, targets=ltargets.cpu().numpy())
    if not (np.array_equal(r[2].cpu().numpy(), wl_[0]) and np.array_equal(r[3].cpu().numpy(), wl_[2])
            and np.array_equal(r[1].cpu().numpy().view(np.int32), wl_[1].view(np.int32))):
        fail("rank_lists")
    del r

    topk = alternated({"k{}".format(k): (lambda k=k: eng.catalogue_topk(users, k, exclude=(rowptr, lists),
                                                                        targets=targets)) for k in ks}, args.reps)
    for k in ks:
        topk["k{}".format(k)]["over_k10"] = round(topk["k{}".format(k)]["ms"] / topk["k10"]["ms"], 4) \
            if "k10" in topk else None
    out = {"tool": "topk_large_bench", "workload": args.workload, "users": nu, "items": ni, "layers": wl["layers"],
           "mf_dim": wl["mf_dim"], "reps": args.reps, "lib": os.path.relpath(nat.LIB_PATH, ROOT),
           "catalogue_topk": topk}
    if not args.no_audience:
        aud = alternated({"all_k{}".format(k): (lambda k=k: eng.catalogue_audience(all_items, k,
                                                                                   exclude=(irowptr, iusers),
                                                                                   targets=held)) for k in (10, K)},
                         args.reps)
        aud["all_k{}".format(K)]["over_k10"] = round(aud["all_k{}".format(K)]["ms"] / aud["all_k10"]["ms"], 4)
        aud.update(alternated({"new100_k{}".format(k): (lambda k=k: eng.catalogue_audience(
            new_items, k, exclude=(irowptr, iusers))) for k in (10, K)}, args.reps))
        out["catalogue_audience"] = aud
    out["rank_lists_1024x5000"] = alternated({"k{}".format(k): (lambda k=k: eng.rank_lists(
        lu, (lrowptr, litems), k, targets=ltargets)) for k in sorted({256, K})}, args.reps)
    name, power = gpu_info()
    out.update({"gpu": name, "power_limit": power, "oracle_check": "passed",
                "oracle_check_users": check.tolist(), "oracle_check_items": ccols.tolist()})
    print(json.dumps(out))


if __name__ == "__main__":
    main()
