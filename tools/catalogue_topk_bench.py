"""Full-catalogue top-k and leave-one-out ranking against every unseen item (mr_catalogue_topk), timed next to the
sampled ranking eval (mr_rank_eval, 100 candidates per user) on the same seeded weights.  GPU only.

For every user of the workload's shape: k = 10, exclusion lists = the per-user CSR of the synthetic ratings
(bench.synth_ratings), one held-out target per user.  CUDA events around each call after a warm-up call.  Before any
number is printed, the top-k, positions and probabilities of >= 8 sampled users are checked against the NumPy
reference (tests/catalogue_oracle.py on the kernel's scores; the scores against oracle.forward); a failed check
exits non-zero.  Prints one JSON line.

    python tools/catalogue_topk_bench.py --workload ml-20m [--reps 3]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "movierecommender-tf-trt_b200"), os.path.join(ROOT, "tests")]

import torch  # noqa: E402

import bench  # noqa: E402
from catalogue_oracle import catalogue_topk  # noqa: E402
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


def timed(fn, reps):
    """(mean ms over reps, phase split of one extra profiled call)."""
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    ms = a.elapsed_time(b) / reps
    nat.profile_begin()
    fn()
    phases, launches = nat.profile_end()
    return ms, {k: round(v[0], 4) for k, v in phases.items() if v[1]}, launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="ml-20m", choices=["ml-20m", "ml-1m"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--check-users", type=int, default=8)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("catalogue_topk_bench: needs a CUDA device")
    wl = bench.WORKLOADS[args.workload]
    nu, ni, k = wl["num_users"], wl["num_items"], args.k
    dev = torch.device("cuda")
    eng = _engine.NeuMFEngine(nu, ni, wl["layers"], [0] * len(wl["layers"]), mf_dim=wl["mf_dim"], seed=1)
    ru, ri = bench.synth_ratings(wl, 0)
    rowptr, lists = _engine.build_user_csr(ru, ri, nu, ni)
    rng = np.random.default_rng(2)
    users = torch.arange(nu, dtype=torch.int32, device=dev)
    targets = torch.from_numpy(rng.integers(0, ni, nu).astype(np.int32)).to(dev)

    def catalogue():
        return eng.catalogue_topk(users, k, exclude=(rowptr, lists), targets=targets)

    ev_users, ev_items, group = bench.synth_eval(wl, nu, 3)
    d_eu, d_ei = torch.from_numpy(ev_users).to(dev), torch.from_numpy(ev_items).to(dev)

    def sampled():
        return eng.rank_eval(d_eu, d_ei, group, wl["k_eval"])

    # oracle check on sampled users (their scores through want_scores, the rest of the selection on the device)
    check = np.sort(rng.choice(nu, args.check_users, replace=False)).astype(np.int32)
    top, top_s, pos, _ = catalogue()[:4]
    c_items, c_scores, c_pos, _, full = eng.catalogue_topk(check, k, exclude=(rowptr, lists), targets=targets[check],
                                                           want_scores=True)
    p = full.cpu().numpy()
    rp, li = rowptr.cpu().numpy(), lists.cpu().numpy()
    t0 = time.perf_counter()
    w_items, w_scores, w_pos, _ = catalogue_topk(p, k, rp, li, excl_ids=check, targets=targets.cpu().numpy()[check])
    oracle_s = time.perf_counter() - t0
    w = eng.get_weights()
    p_or = o.forward({n: np.asarray(v, np.float64) for n, v in w.items()}, np.repeat(check, ni),
                     np.tile(np.arange(ni), check.size))["p"].reshape(check.size, ni)
    ok = (np.array_equal(c_items.cpu().numpy(), w_items) and np.array_equal(c_pos.cpu().numpy(), w_pos)
          and np.array_equal(top.cpu().numpy()[check], w_items) and np.array_equal(pos.cpu().numpy()[check], w_pos)
          and np.array_equal(top_s.cpu().numpy()[check], w_scores)
          and float(np.max(np.abs(p - p_or))) <= 1e-5 * float(np.max(np.abs(p_or))) + 1e-6)
    if not ok:
        sys.exit("catalogue_topk_bench: oracle check FAILED on users {}".format(check.tolist()))

    cat_ms, cat_phases, cat_launches = timed(catalogue, args.reps)
    ev_ms, ev_phases, _ = timed(sampled, args.reps)
    name, power = gpu_info()
    pairs = nu * ni
    sel_ms = cat_phases.get("rank", 0.0)
    out = {
        "tool": "catalogue_topk_bench", "workload": args.workload, "gpu": name, "power_limit": power,
        "users": nu, "items": ni, "k": k, "layers": wl["layers"], "mf_dim": wl["mf_dim"],
        "excluded_pairs": int(li.size), "reps": args.reps,
        "catalogue_ms": round(cat_ms, 3), "catalogue_users_per_s": nu / (cat_ms / 1e3),
        "catalogue_pairs_per_s": pairs / (cat_ms / 1e3),
        "catalogue_phase_ms": cat_phases, "catalogue_kernel_launches": cat_launches,
        "selection_share": round(sel_ms / sum(cat_phases.values()), 4) if cat_phases else None,
        "sampled_eval_ms": round(ev_ms, 3), "sampled_eval_rows_per_s": ev_users.size * group / (ev_ms / 1e3),
        "sampled_eval_phase_ms": ev_phases,
        "pairs_over_sampled_rows": round((pairs / cat_ms) / (ev_users.size * group / ev_ms), 4),
        "oracle_check_users": check.tolist(), "oracle_check": "passed",
        "cpu_oracle_selection_s_per_user": oracle_s / check.size,
    }
    print(json.dumps(out))


if __name__ == "__main__":
    main()
