"""Similar items and users (mr_similar): exact k nearest neighbours of every item among all items, and of every user
among all users, on the workload shapes of bench.py with seeded weights.  GPU only.

ML-20M (tower 256-128-64 + GMF 64, D = 192): all items x all items at k = 10 / 100 / 1000, 1,000 query items, one
query item (median latency on the host clock, 50 calls), all users x all users at k = 10.  ML-1M (default tower + GMF 8,
D = 40): all items and all users at k = 10.  Each call: CUDA events after a warm-up call, `reps` runs, the median
reported, and a separate run with the library's phase profile (GEMM = tc_dense_fwd, selection = rank, representation
= misc).  Comparisons in the same process, all items x all items at k = 10: mr_topk_scores on the materialised score
matrix with each query's own id as its exclusion list (the selection alone), and torch fp32 matmul (TF32 off) plus a
masked torch.topk over the same representation.  Before any number is printed, sampled queries are checked: the
selection bit for bit against tests/similar_oracle.py on the call's own scores, the similarities against the float64
oracle; a failed check exits non-zero.  With --quality: neighbour precision@10 on the planted clusters of
tests/test_gpu_fold_in.py (the share of a row's 10 neighbours in its own cluster) for this representation, for the raw
[mlp | gmf] cosine (NumPy) and chance, items and users.  Prints one JSON line.

    python tools/similar_bench.py --workload ml-20m [--reps 3] [--quality]
"""
import argparse
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
from movierec import _engine, _native as nat  # noqa: E402
from similar_oracle import representation, side_parts, similar_select, similarity  # noqa: E402


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


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    runs = [event_ms(fn) for _ in range(reps)]
    nat.profile_begin()
    fn()
    ph, launches = nat.profile_end()
    ph = {k: round(v[0], 4) for k, v in ph.items() if v[1]}
    tot = sum(ph.values()) or 1.0
    return {"ms": round(float(np.median(runs)), 3), "ms_runs": [round(x, 3) for x in runs], "phase_ms": ph,
            "gemm_share": round(ph.get("tc_dense_fwd", 0.0) / tot, 4),
            "selection_share": round(ph.get("rank", 0.0) / tot, 4), "kernel_launches": launches}


def check(eng, side, mf, N, k, rng, n=8):
    """Sampled queries: the selection bit for bit on the call's own scores, the similarities against float64."""
    ids = np.sort(rng.choice(N, n, replace=False)).astype(np.int32)
    top, sims, full = eng.similar(ids, k, side=side, want_scores=True)
    S = full.cpu().numpy()
    w_top, w_sims = similar_select(S, ids, k)
    R64 = representation(*side_parts(eng.get_weights(), side, mf))
    err = float(np.max(np.abs(S - similarity(R64, ids))))
    ok = (np.array_equal(top.cpu().numpy(), w_top) and np.array_equal(sims.cpu().numpy().view(np.int32),
                                                                       w_sims.view(np.int32)) and err <= 1e-5)
    if not ok:
        sys.exit("similar_bench: oracle check FAILED ({} side, ids {}, max error {:.3e})".format(side, ids.tolist(), err))
    return err


def torch_reference(eng, mf, k, chunk=4096):
    """torch fp32 (TF32 off) matmul over the representation plus a masked torch.topk, all items x all items."""
    w = eng.get_weights()
    R = torch.from_numpy(representation(*side_parts(w, "items", mf), dtype=np.float32)).cuda()
    N = R.shape[0]
    torch.backends.cuda.matmul.allow_tf32 = False

    def run():
        for q0 in range(0, N, chunk):
            S = R[q0:q0 + chunk] @ R.T
            r = torch.arange(S.shape[0], device=S.device)
            S[r, r + q0] = float("-inf")
            torch.topk(S, k, dim=1)
    return run


def precision_at_10(top, cl_rows, cl_cands):
    return float(np.mean(cl_cands[top] == cl_rows[:, None]))


def quality():
    import test_gpu_fold_in as t
    uc, ic, hist = t.planted_dataset()
    eng = t.train_planted(_engine, hist, 480)
    w = eng.get_weights()
    out = {}
    for side, cl in (("items", ic), ("users", uc)):
        N = cl.size
        top = eng.similar(np.arange(N, dtype=np.int32), 10, side=side)[0].cpu().numpy()
        E, _, G, _ = side_parts(w, side, 8)
        raw = np.concatenate([E, G], axis=1).astype(np.float64)
        raw /= np.maximum(np.linalg.norm(raw, axis=1, keepdims=True), 1e-30)
        C = raw @ raw.T
        np.fill_diagonal(C, -np.inf)
        raw_top = np.argsort(-C, axis=1, kind="stable")[:, :10]
        out[side] = {"representation_precision@10": round(precision_at_10(top, cl, cl), 4),
                     "raw_cosine_precision@10": round(precision_at_10(raw_top, cl, cl), 4), "chance": 1 / 8}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="ml-20m", choices=["ml-20m", "ml-1m"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--quality", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("similar_bench: needs a CUDA device")
    wl = bench.WORKLOADS[args.workload]
    nu, ni, mf = wl["num_users"], wl["num_items"], wl["mf_dim"]
    dev = torch.device("cuda")
    eng = _engine.NeuMFEngine(nu, ni, wl["layers"], [0] * len(wl["layers"]), mf_dim=mf, seed=1)
    rng = np.random.default_rng(2)
    errs = {"items": check(eng, "items", mf, ni, 10, rng), "users": check(eng, "users", mf, nu, 10, rng)}
    all_items = torch.arange(ni, dtype=torch.int32, device=dev)
    all_users = torch.arange(nu, dtype=torch.int32, device=dev)
    L1 = wl["layers"][1]
    D = (L1 + mf + 31) // 32 * 32
    out = {"tool": "similar_bench", "workload": args.workload, "users": nu, "items": ni, "layers": wl["layers"],
           "mf_dim": mf, "D": D, "reps": args.reps, "oracle_check": "passed",
           "oracle_max_abs_error": {k: float("{:.3e}".format(v)) for k, v in errs.items()}}
    ks = (10, 100, 1000) if args.workload == "ml-20m" else (10,)
    for k in ks:
        r = timed(lambda: eng.similar(all_items, k), args.reps)
        r["pairs_per_s"] = ni * ni / (r["ms"] / 1e3)
        out["items_all_k{}".format(k)] = r
    r = timed(lambda: eng.similar(all_users, 10, side="users"), args.reps)
    r["pairs_per_s"] = nu * nu / (r["ms"] / 1e3)
    out["users_all_k10"] = r
    # GEMM bytes and FLOPs per pair: 3 TF32 MMAs per K step (6 D FLOPs), one fp32 score written and read back
    out["gemm_flops_per_pair"] = 6 * D
    out["score_bytes_per_pair"] = 8
    if args.workload == "ml-20m":
        q = torch.from_numpy(rng.choice(ni, 1000, replace=False).astype(np.int32)).to(dev)
        out["items_1000_queries_k10"] = timed(lambda: eng.similar(q, 10), args.reps)
        one = torch.from_numpy(np.int32([int(rng.integers(0, ni))])).to(dev)
        for _ in range(5):
            eng.similar(one, 10)
        torch.cuda.synchronize()
        lat = []
        for _ in range(50):
            t0 = time.perf_counter()
            top = eng.similar(one, 10)[0]
            torch.cuda.synchronize()
            lat.append((time.perf_counter() - t0) * 1e3)
        out["items_one_query_k10_ms_median"] = round(float(np.median(lat)), 4)
        del top
    # comparisons on all items x all items at k = 10
    full = eng.similar(all_items, 10, want_scores=True)[2]
    self_rp = torch.arange(ni + 1, dtype=torch.int64, device=dev)

    def sel():
        return _engine.topk_scores(full, 10, exclude=(self_rp, all_items))
    out["selection_alone_topk_scores_k10"] = timed(sel, args.reps)
    out["items_call_over_selection_alone"] = round(out["items_all_k10"]["ms"] / out["selection_alone_topk_scores_k10"]["ms"], 4)
    del full
    torch.cuda.empty_cache()
    ref = torch_reference(eng, mf, 10)
    ref()
    torch.cuda.synchronize()
    t_ref = [event_ms(ref) for _ in range(args.reps)]
    out["torch_fp32_matmul_topk_k10_ms"] = round(float(np.median(t_ref)), 3)
    out["torch_over_call"] = round(out["torch_fp32_matmul_topk_k10_ms"] / out["items_all_k10"]["ms"], 3)
    if args.quality:
        out["planted_quality"] = quality()
    name, power = gpu_info()
    out["gpu"], out["power_limit"] = name, power
    print(json.dumps(out))


if __name__ == "__main__":
    main()
