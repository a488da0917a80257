"""Fold-in (mr_fold_in_users) timed on the GPU, and the planted-cluster quality sweep behind the defaults.

Speed (default): 10,000 users whose histories are the first 10,000 users of bench.synth_ratings of the workload's shape
(20 + a lognormal tail, Zipf items), folded in with the model's defaults (steps = FOLD_IN_STEPS, lr = FOLD_IN_LR,
negs = 4, Adam) into a model of the workload's tower.  Reports users/s, fold-in rows/s (steps x sum of n (negs + 1))
and the longest user's share of the call (that user folded in alone, over the whole call); then the request latency of
NeuMFModel.recommend_for_histories for one user with 50 ratings (host clock, results read back); then the float32 NumPy
reference (tests/fold_in_oracle.py) on the CPU for a few of the same users as the baseline.  CUDA events around each
call after a warm-up call.  Prints one JSON line and writes it to --out.

    python tools/fold_in_bench.py --workload ml-20m [--out profiles/r06_fold_in_ml20m.json]
    python tools/fold_in_bench.py --quality [--out profiles/r06_fold_in_quality.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "movierecommender-tf-trt_b200"), os.path.join(ROOT, "tests")]

import torch  # noqa: E402

import bench  # noqa: E402
from catalogue_topk_bench import gpu_info  # noqa: E402
from movierec import _engine  # noqa: E402
from movierec import model as mm  # noqa: E402

NEGS = 4


def histories(wl, users):
    ru, ri = bench.synth_ratings(wl, 0)
    keep = ru < users
    rp, it = _engine.build_user_csr(ru[keep], ri[keep], users, wl["num_items"])
    return rp.cpu().numpy(), it.cpu().numpy()


def event_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def speed(args):
    wl = bench.WORKLOADS[args.workload]
    nu, ni = wl["num_users"], wl["num_items"]
    eng = _engine.NeuMFEngine(nu, ni, wl["layers"], [0] * len(wl["layers"]), mf_dim=wl["mf_dim"], seed=1)
    rowptr, items = histories(wl, args.users)
    lens = np.diff(rowptr)
    steps, lr = mm.FOLD_IN_STEPS, mm.FOLD_IN_LR
    call = lambda h: eng.fold_in(h, steps, lr, NEGS, seed=1)
    ms = event_ms(lambda: call((rowptr, items)), args.reps)
    u = int(np.argmax(lens))
    one = (np.int64([0, lens[u]]), items[rowptr[u]:rowptr[u + 1]])
    ms_longest = event_ms(lambda: call(one), args.reps)
    rows = steps * int(lens.sum()) * (NEGS + 1)

    params = dict(num_users=nu, num_items=ni, layers_sizes=wl["layers"], layers_l2reg=[0] * len(wl["layers"]),
                  optimizer="adam", lr=0.001, batch_size=5, num_negs_per_pos=NEGS, batch_size_eval=100,
                  num_negs_per_pos_eval=99, k=5, mf_dim=wl["mf_dim"], seed=1)
    model = mm.MovierecModel(params, output_dir=os.path.join(args.tmp, "model"), verbose=0)
    model.model.engine = eng
    req = [np.sort(np.random.default_rng(2).choice(ni, 50, replace=False))]
    model.model.recommend_for_histories(req, 10)
    lat = []
    for _ in range(args.reps * 10):
        t0 = time.perf_counter()
        model.model.recommend_for_histories(req, 10)
        lat.append((time.perf_counter() - t0) * 1e3)

    from fold_in_oracle import fold_in
    w = eng.get_weights()
    sub = np.arange(args.cpu_users)
    c_rowptr = np.concatenate([[0], np.cumsum(lens[sub])]).astype(np.int64)
    c_items = np.concatenate([items[rowptr[i]:rowptr[i + 1]] for i in sub])
    t0 = time.perf_counter()
    fold_in(w, c_rowptr, c_items, steps, NEGS, 1, lr=lr)
    cpu_s = time.perf_counter() - t0

    name, power = gpu_info()
    return {
        "tool": "fold_in_bench", "workload": args.workload, "gpu": name, "power_limit": power,
        "items": ni, "layers": wl["layers"], "mf_dim": wl["mf_dim"], "users": args.users, "ratings": int(lens.sum()),
        "max_history": int(lens.max()), "steps": steps, "lr": lr, "negs": NEGS, "optimizer": "adam", "reps": args.reps,
        "fold_in_ms": round(ms, 3), "users_per_s": args.users / ms * 1e3, "fold_in_rows_per_s": rows / ms * 1e3,
        "longest_user_ms": round(ms_longest, 3), "longest_user_share": round(ms_longest / ms, 4),
        "request_50_ratings_ms_median": round(float(np.median(lat)), 3),
        "request_50_ratings_ms_p90": round(float(np.percentile(lat, 90)), 3),
        "cpu_oracle_fp32_users": args.cpu_users, "cpu_oracle_fp32_users_per_s": args.cpu_users / cpu_s,
    }


def quality(args):
    """Recall@10 on the held-out 20 % of planted-cluster users folded in from the other 80 %, over a grid of steps and
    lr (Adam, negs 4), next to the zero-row and popularity baselines (tests/test_gpu_fold_in.py's dataset and model)."""
    import test_gpu_fold_in as t
    uc, ic, hist = t.planted_dataset()
    n_train = 2500
    eng = t.train_planted(_engine, hist[:n_train], 480)
    keep, held = t.split_80_20(hist[n_train:])
    users = np.arange(len(keep), dtype=np.int32)
    excl = t._csr(keep)

    def recall(steps, lr):
        mlp, gmf, loss = eng.fold_in(keep, steps, lr, NEGS, seed=3)
        top = eng.user_view(mlp, gmf).catalogue_topk(users, 10, exclude=excl)[0].cpu().numpy()
        return t.recall_at(top, held), (float(np.nanmean(loss.cpu().numpy())) if steps else float("nan"))

    grid = []
    for steps in (5, 10, 20, 30, 50, 100):
        for lr in (0.001, 0.01, 0.03, 0.05, 0.1, 0.3):
            r, lo = recall(steps, lr)
            grid.append({"steps": steps, "lr": lr, "recall@10": round(r, 4), "mean_last_loss": round(lo, 4)})
    name, power = gpu_info()
    return {"tool": "fold_in_bench", "mode": "quality", "gpu": name, "power_limit": power,
            "dataset": "planted clusters: 3000 users (2500 trained, 500 folded in), 480 items, 8 clusters, 40 ratings "
                       "per user, 90 % inside the user's cluster",
            "model": "64-32-16-8 + GMF 8, Adam lr 0.005, 8 epochs, negs 4",
            "zero_rows_recall@10": round(recall(0, 0.0)[0], 4),
            "popularity_recall@10": round(t.popularity_recall(hist[:n_train], keep, held, 480), 4), "grid": grid}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="ml-20m", choices=["ml-20m", "ml-1m"])
    ap.add_argument("--users", type=int, default=10000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cpu-users", type=int, default=4)
    ap.add_argument("--quality", action="store_true")
    ap.add_argument("--tmp", default="/tmp/fold_in_bench")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("fold_in_bench: needs a CUDA device")
    res = quality(args) if args.quality else speed(args)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
