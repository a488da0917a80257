"""Item fold-in (mr_fold_in_items) timed on the GPU, and the planted-cluster quality grid behind its defaults.

Speed (default): a model of the workload's tower; the new items are the 2,000 least popular items of bench.synth_ratings
of the workload's shape, with their rater lists from the same data, folded in with the defaults (steps = FOLD_IN_STEPS,
lr = FOLD_IN_LR, negs = 4, Adam).  Reports items/s, fold-in rows/s (steps x sum of |R| (negs + 1)) and the longest
list's share of the call (that item folded in alone, over the whole call); the item at popularity rank 100 folded in
alone, which is the single-CTA floor (one CTA folds one item: a long list is not split); the latency of one new item
with 50 raters including the item view and one recommend_for_users for 1,024 users over the extended catalogue (host
clock, results read back); and the float32 NumPy reference (tests/fold_in_items_oracle.py) on the CPU for a few of the
items as the baseline.  CUDA events around each call after a warm-up call.  Prints one JSON line and writes it to
--out.

    python tools/fold_in_items_bench.py --workload ml-20m [--out profiles/r07_fold_in_items_ml20m.json]
    python tools/fold_in_items_bench.py --quality [--out profiles/r07_fold_in_items_quality.json]
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "movierecommender-tf-trt_b200"), os.path.join(ROOT, "tests"),
                os.path.join(ROOT, "tools")]

import torch  # noqa: E402

import bench  # noqa: E402
from catalogue_topk_bench import gpu_info  # noqa: E402
from fold_in_bench import event_ms  # noqa: E402
from movierec import _engine  # noqa: E402
from movierec import model as mm  # noqa: E402

NEGS = 4


def rater_lists(ru, ri, items):
    """Ascending unique raters of each of `items` -> (rowptr, users)."""
    sel = np.isin(ri, items)
    where = np.full(max(int(ri.max()), int(items.max())) + 1, -1, np.int64)
    where[items] = np.arange(items.size)
    key = np.unique(where[ri[sel]] * (1 << 32) + ru[sel].astype(np.int64))
    slot, users = key >> 32, (key & 0xFFFFFFFF).astype(np.int32)
    rowptr = np.zeros(items.size + 1, np.int64)
    rowptr[1:] = np.cumsum(np.bincount(slot, minlength=items.size))
    return rowptr, users


def speed(args):
    wl = bench.WORKLOADS[args.workload]
    nu, ni = wl["num_users"], wl["num_items"]
    eng = _engine.NeuMFEngine(nu, ni, wl["layers"], [0] * len(wl["layers"]), mf_dim=wl["mf_dim"], seed=1)
    ru, ri = bench.synth_ratings(wl, 0)
    counts = np.bincount(ri, minlength=ni)
    by_pop = np.argsort(-counts, kind="stable")
    new_items = by_pop[::-1][:args.items].copy()
    rowptr, users = rater_lists(ru, ri, new_items)
    lens = np.diff(rowptr)
    steps, lr = mm.FOLD_IN_STEPS, mm.FOLD_IN_LR
    call = lambda r: eng.fold_in_items(r, steps, lr, NEGS, seed=1)
    ms = event_ms(lambda: call((rowptr, users)), args.reps)
    j = int(np.argmax(lens))
    one = (np.int64([0, lens[j]]), users[rowptr[j]:rowptr[j + 1]])
    ms_longest = event_ms(lambda: call(one), args.reps)
    rows = steps * int(lens.sum()) * (NEGS + 1)
    rp100, us100 = rater_lists(ru, ri, by_pop[99:100].copy())
    ms_100 = event_ms(lambda: call((rp100, us100)), args.reps)
    rows_100 = steps * int(us100.size) * (NEGS + 1)

    params = dict(num_users=nu, num_items=ni, layers_sizes=wl["layers"], layers_l2reg=[0] * len(wl["layers"]),
                  optimizer="adam", lr=0.001, batch_size=5, num_negs_per_pos=NEGS, batch_size_eval=100,
                  num_negs_per_pos_eval=99, k=5, mf_dim=wl["mf_dim"], seed=1)
    with tempfile.TemporaryDirectory() as tmp:
        model = mm.MovierecModel(params, output_dir=tmp, verbose=0)
    model.model.engine = eng
    req = [np.sort(np.random.default_rng(2).choice(nu, 50, replace=False))]
    serve_users = np.arange(1024, dtype=np.int32)

    def request():
        folded = model.fold_in_items(req)
        return folded.model.recommend_for_users(serve_users, 10)

    request()
    lat = []
    for _ in range(args.reps * 10):
        t0 = time.perf_counter()
        request()
        lat.append((time.perf_counter() - t0) * 1e3)

    from fold_in_items_oracle import fold_in_item
    w = eng.get_weights()
    t0 = time.perf_counter()
    for i in range(args.cpu_items):
        fold_in_item(w, users[rowptr[i]:rowptr[i + 1]], steps, NEGS, 1, lr=lr)
    cpu_s = time.perf_counter() - t0

    name, power = gpu_info()
    return {
        "tool": "fold_in_items_bench", "workload": args.workload, "gpu": name, "power_limit": power,
        "users": nu, "catalogue_items": ni, "layers": wl["layers"], "mf_dim": wl["mf_dim"],
        "new_items": args.items, "new_items_from": "least popular of bench.synth_ratings(wl, 0)",
        "raters": int(lens.sum()), "mean_raters": round(float(lens.mean()), 2), "max_raters": int(lens.max()),
        "steps": steps, "lr": lr, "negs": NEGS, "optimizer": "adam", "reps": args.reps,
        "fold_in_ms": round(ms, 3), "items_per_s": args.items / ms * 1e3, "fold_in_rows_per_s": rows / ms * 1e3,
        "longest_item_ms": round(ms_longest, 3), "longest_item_share": round(ms_longest / ms, 4),
        "rank_100_item_raters": int(us100.size), "rank_100_item_ms": round(ms_100, 3),
        "rank_100_item_rows_per_s": rows_100 / ms_100 * 1e3,
        "request_50_raters_1024_users_ms_median": round(float(np.median(lat)), 3),
        "request_50_raters_1024_users_ms_p90": round(float(np.percentile(lat, 90)), 3),
        "cpu_oracle_fp32_items": args.cpu_items, "cpu_oracle_fp32_items_per_s": args.cpu_items / cpu_s,
    }


def quality(args):
    """Recall@10 of the held-out (user, new item) pairs of planted clusters, with 60 items kept out of training and
    folded in from 80 % of their raters, over a grid of steps and lr (Adam, negs 4), next to the zero-row and
    mean-row baselines (tests/test_gpu_fold_in_items.py's protocol)."""
    import test_gpu_fold_in_items as t
    eng, setup = t.planted_items_setup(_engine)
    with tempfile.TemporaryDirectory() as tmp:
        mr = t.planted_items_model(eng, setup, tmp)
    M = t.HELD_ITEMS

    def run(steps, lr):
        folded = mr.fold_in_items(setup["fold"], steps=steps, lr=lr, seed=3)
        return t.planted_items_recall(folded, setup), (float(np.nanmean(folded.loss)) if steps else float("nan"))

    grid = []
    for steps in (5, 10, 20, 30, 50, 100):
        for lr in (0.001, 0.01, 0.03, 0.05, 0.1, 0.3):
            r, lo = run(steps, lr)
            grid.append({"steps": steps, "lr": lr, "recall@10": round(r, 4), "mean_last_loss": round(lo, 4)})
    name, power = gpu_info()
    return {"tool": "fold_in_items_bench", "mode": "quality", "gpu": name, "power_limit": power,
            "dataset": "planted clusters: 3000 users, 480 items, 8 clusters, 40 ratings per user, 90 % inside the "
                       "user's cluster; 60 items held out of training, renumbered 420..479, folded in from 80 % of "
                       "their raters, recall@10 over the other 20 % of (user, new item) pairs",
            "model": "64-32-16-8 + GMF 8 on the 420 trained items, Adam lr 0.005, 8 epochs, negs 4",
            "zero_rows_recall@10": round(run(0, 0.0)[0], 4),
            "mean_rows_recall@10": round(t.planted_items_recall(t.mean_rows_model(mr, M), setup), 4), "grid": grid}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="ml-20m", choices=["ml-20m", "ml-1m"])
    ap.add_argument("--items", type=int, default=2000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--cpu-items", type=int, default=4)
    ap.add_argument("--quality", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("fold_in_items_bench: needs a CUDA device")
    res = quality(args) if args.quality else speed(args)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
