"""Many held-out items per user ranked against the whole catalogue (mr_catalogue_targets), timed next to the
leave-one-out top-k call (mr_catalogue_topk, k = 10, each user's first held-out item) on the same seeded weights.
GPU only.

Ratings: bench.synth_ratings of the workload's shape; the last 20 % of each user's ratings (at least one) are held out
and the rest are the exclusion lists.  Cutoffs 1, 5, 10, 20, 50, 100.  CUDA events around each call after a warm-up
call; the phase split comes from one extra profiled call.  Before any number is printed, the positions of >= 8 sampled
users are checked bit for bit against the NumPy reference (tests/targets_oracle.py on the model's probabilities); a
failed check exits non-zero.  Prints one JSON line and writes it to --out.

    python tools/catalogue_targets_bench.py --workload ml-20m [--reps 3] [--out profiles/r05_catalogue_targets_ml20m.json]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "movierecommender-tf-trt_b200"), os.path.join(ROOT, "tests")]

import torch  # noqa: E402

import bench  # noqa: E402
from catalogue_topk_bench import gpu_info, timed  # noqa: E402
from movierec import _engine  # noqa: E402
from targets_oracle import target_positions  # noqa: E402

KS = (1, 5, 10, 20, 50, 100)


def split_last_fifth(users, n_users):
    """Boolean mask of the held-out ratings: per user (ratings grouped by user, in order), the last 20 %, at least one."""
    counts = np.bincount(users, minlength=n_users)
    start = np.concatenate([[0], np.cumsum(counts)[:-1]])
    held = np.maximum(1, counts // 5)
    place = np.arange(users.size) - start[users]
    return place >= (counts - held)[users]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="ml-20m", choices=["ml-20m", "ml-1m"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--check-users", type=int, default=8)
    ap.add_argument("--out", default=None, help="default: profiles/r05_catalogue_targets_<workload>.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("catalogue_targets_bench: needs a CUDA device")
    wl = bench.WORKLOADS[args.workload]
    nu, ni = wl["num_users"], wl["num_items"]
    dev = torch.device("cuda")
    eng = _engine.NeuMFEngine(nu, ni, wl["layers"], [0] * len(wl["layers"]), mf_dim=wl["mf_dim"], seed=1)
    ru, ri = bench.synth_ratings(wl, 0)
    held = split_last_fifth(ru, nu)
    ex_rowptr, ex_items = _engine.build_user_csr(ru[~held], ri[~held], nu, ni)
    t_rowptr, t_items = _engine.build_user_csr(ru[held], ri[held], nu, ni)
    users = torch.arange(nu, dtype=torch.int32, device=dev)
    assert bool((t_rowptr[1:] > t_rowptr[:-1]).all())  # every user holds out at least one item
    first = t_items[t_rowptr[:-1]].contiguous()

    def targets():
        return eng.catalogue_targets(users, (t_rowptr, t_items), KS, exclude=(ex_rowptr, ex_items))

    def topk():
        return eng.catalogue_topk(users, 10, exclude=(ex_rowptr, ex_items), targets=first)

    rng = np.random.default_rng(2)
    check = np.sort(rng.choice(nu, args.check_users, replace=False)).astype(np.int32)
    tpos, _ = targets()
    _, _, _, _, full = eng.catalogue_topk(check, 10, want_scores=True)
    rp, it = t_rowptr.cpu().numpy(), t_items.cpu().numpy()
    lists = [it[rp[u]:rp[u + 1]] for u in check]
    sub_rowptr = np.concatenate([[0], np.cumsum([x.size for x in lists])])
    want = target_positions(full.cpu().numpy(), sub_rowptr, np.concatenate(lists), ex_rowptr.cpu().numpy(),
                            ex_items.cpu().numpy(), excl_ids=check)
    got = np.concatenate([tpos.cpu().numpy()[rp[u]:rp[u + 1]] for u in check])
    if not np.array_equal(got, want):
        sys.exit("catalogue_targets_bench: oracle check FAILED on users {}".format(check.tolist()))

    tgt_ms, tgt_phases, tgt_launches = timed(targets, args.reps)
    topk_ms, topk_phases, _ = timed(topk, args.reps)
    _, sums = targets()
    s = sums.cpu().numpy().astype(np.float64)
    metrics = {"mrr": s[1] / s[0]}
    for c, k in enumerate(KS):
        for j, name in enumerate(("hr", "precision", "recall", "ndcg", "map")):
            metrics["{}@{}".format(name, k)] = s[2 + 5 * c + j] / s[0]
    name, power = gpu_info()
    pairs = nu * ni
    rank_ms = tgt_phases.get("rank", 0.0)
    out = {
        "tool": "catalogue_targets_bench", "workload": args.workload, "gpu": name, "power_limit": power,
        "users": nu, "items": ni, "layers": wl["layers"], "mf_dim": wl["mf_dim"], "cutoffs": list(KS),
        "held_out_items": int(it.size), "excluded_pairs": int(ex_items.numel()), "reps": args.reps,
        "max_held_out_per_user": int(np.diff(rp).max()),
        "targets_ms": round(tgt_ms, 3), "targets_users_per_s": nu / (tgt_ms / 1e3),
        "targets_gpairs_per_s": pairs / (tgt_ms / 1e3) / 1e9,
        "targets_phase_ms": tgt_phases, "targets_kernel_launches": tgt_launches,
        "positions_and_metrics_share": round(rank_ms / sum(tgt_phases.values()), 4) if tgt_phases else None,
        "catalogue_topk_k10_ms": round(topk_ms, 3), "catalogue_topk_phase_ms": topk_phases,
        "targets_over_topk": round(tgt_ms / topk_ms, 4),
        "metrics_at_seeded_weights": {k: round(v, 6) for k, v in metrics.items()},
        "oracle_check_users": check.tolist(), "oracle_check": "passed",
    }
    line = json.dumps(out)
    print(line)
    path = args.out or os.path.join(ROOT, "profiles", "r05_catalogue_targets_{}.json".format(
        args.workload.replace("-", "")))
    with open(path, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
