"""Ragged candidate lists (mr_rank_lists) on the ML-20M-shaped model (256-128-64, GMF 64, 138,493 x 26,744 seeded
weights), k = 10.  GPU only.  Three measurements, each a warm-up call and then at least a second of calls between CUDA
events (the library is called directly on preallocated device buffers, so the timings are the calls' device work):

  A  serving: 1024 lists of 1000 random candidates per call (users/s), the same 1024 requests through
     NeuMFModel.recommend one by one on the host wall clock, and a single 1 x 1000 call (with its per-call item
     projection);
  B  uniform eval: 138,493 lists of 100 with the positive last, mr_rank_lists against mr_rank_eval alternating in
     the same run; their positions must be identical;
  C  ragged eval: 20,000 lists with lengths log-uniform in [1, 26,744]: rows/s and the selection's (RANK phase)
     share of the call.

Before any timing, A's top-k is checked bit for bit against the NumPy reference selection (tests/lists_oracle.py) on
the call's own probabilities, and the probabilities of eight lists against oracle.forward in float64; a failed check
exits non-zero.  Prints one JSON line per measurement (and writes them under --out-dir when given).

    python tools/rank_lists_bench.py [--out-dir DIR] [--seconds 1.0]
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
from lists_oracle import topk_lists  # noqa: E402
from movierec import _engine, _native as nat, model as mm  # noqa: E402
from oracle import movierec_oracle as o  # noqa: E402


def gpu_info():
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


class ListsCall(object):
    """mr_rank_lists on device buffers allocated once."""

    def __init__(self, eng, users, rowptr, items, k, targets=None, want_probs=False):
        dev = eng.device
        self.eng, self.k = eng, k
        self.users = torch.from_numpy(np.asarray(users, np.int32)).to(dev)
        self.rowptr = torch.from_numpy(np.asarray(rowptr, np.int64)).to(dev)
        self.items = torch.from_numpy(np.asarray(items, np.int32)).to(dev)
        self.U, self.nnz = self.users.numel(), self.items.numel()
        self.t = torch.from_numpy(np.asarray(targets, np.int32)).to(dev) if targets is not None else None
        self.top_pos = torch.empty((self.U, k), dtype=torch.int32, device=dev)
        self.top_items = torch.empty((self.U, k), dtype=torch.int32, device=dev)
        self.top_scores = torch.empty((self.U, k), dtype=torch.float32, device=dev)
        self.pos = torch.empty(self.U, dtype=torch.int32, device=dev) if targets is not None else None
        self.sums = torch.zeros(2, dtype=torch.float32, device=dev) if targets is not None else None
        self.probs = torch.empty(self.nnz, dtype=torch.float32, device=dev) if want_probs else None
        nbytes = int(nat.lib.mr_rank_lists_workspace_bytes(C.byref(eng._model), self.U, self.nnz, k))
        self.ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        self.ws_bytes = nbytes
        self.stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def __call__(self):
        p = _engine._ptr
        nat.check(nat.lib.mr_rank_lists(C.byref(self.eng._model), p(self.users), self.U, p(self.rowptr), p(self.items),
                                        self.nnz, self.k, p(self.t), p(self.top_pos), p(self.top_items),
                                        p(self.top_scores), p(self.pos), p(self.sums), p(self.probs), p(self.ws),
                                        self.ws_bytes, self.stream), "mr_rank_lists")


def timed(fns, seconds):
    """Mean device ms per call of each fn: a warm-up call, then rounds of all fns (alternating) until each has run for
    `seconds`; plus the phase split of one extra profiled call of each."""
    for fn in fns:
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for fn in fns:
        fn()
    torch.cuda.synchronize()
    reps = max(3, int(seconds / max(time.perf_counter() - t0, 1e-6) * len(fns)) // len(fns) + 1)
    tot = [0.0] * len(fns)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in fns]
    for _ in range(reps):
        for i, fn in enumerate(fns):
            ev[i][0].record()
            fn()
            ev[i][1].record()
        torch.cuda.synchronize()
        for i in range(len(fns)):
            tot[i] += ev[i][0].elapsed_time(ev[i][1])
    out = []
    for i, fn in enumerate(fns):
        nat.profile_begin()
        fn()
        phases, launches = nat.profile_end()
        out.append((tot[i] / reps, {k: round(v[0], 4) for k, v in phases.items() if v[1]}, launches, reps))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", default=None)
    ap.add_argument("--seconds", type=float, default=1.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("rank_lists_bench: needs a CUDA device")
    wl = bench.WORKLOADS["ml-20m"]
    nu, ni, k = wl["num_users"], wl["num_items"], 10
    eng = _engine.NeuMFEngine(nu, ni, wl["layers"], [0] * len(wl["layers"]), mf_dim=wl["mf_dim"], seed=1)
    name, power = gpu_info()
    common = {"tool": "rank_lists_bench", "gpu": name, "power_limit": power, "layers": wl["layers"],
              "mf_dim": wl["mf_dim"], "users": nu, "items": ni, "k": k}
    rng = np.random.default_rng(3)
    results = {}

    # ---- A: serving --------------------------------------------------------------------------------------------
    U, L = 1024, 1000
    users = rng.integers(0, nu, U).astype(np.int32)
    items = rng.integers(0, ni, U * L).astype(np.int32)
    rowptr = np.arange(U + 1, dtype=np.int64) * L
    a = ListsCall(eng, users, rowptr, items, k, want_probs=True)
    a()
    p = a.probs.cpu().numpy()
    w_pos, w_scores, _, _ = topk_lists(p, rowptr, k)
    chk = rng.choice(U, 8, replace=False)
    wts = eng.get_weights()
    rows = np.concatenate([np.arange(rowptr[u], rowptr[u + 1]) for u in chk])
    p64 = o.forward({n: np.asarray(v, np.float64) for n, v in wts.items()}, np.repeat(users[chk], L), items[rows])["p"]
    ok = (np.array_equal(a.top_pos.cpu().numpy(), w_pos) and np.array_equal(a.top_scores.cpu().numpy(), w_scores)
          and float(np.max(np.abs(p[rows] - p64))) <= 1e-5 * float(np.max(np.abs(p64))) + 1e-6)
    if not ok:
        sys.exit("rank_lists_bench: oracle check FAILED")
    serve = ListsCall(eng, users, rowptr, items, k)
    single = ListsCall(eng, users[:1], rowptr[:2], items[:L], k)
    (ms_a, ph_a, la_a, reps_a), (ms_1, ph_1, _, reps_1) = timed([serve], args.seconds)[0], timed([single], args.seconds)[0]
    facade = mm.NeuMFModel.__new__(mm.NeuMFModel)
    facade.engine = eng
    facade.recommend(int(users[0]), items[:L], k)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for u in range(U):
        facade.recommend(int(users[u]), items[rowptr[u]:rowptr[u + 1]], k)
    loop_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    facade.recommend_batch(users, (rowptr, items), k)
    batch_s = time.perf_counter() - t0
    results["serving"] = dict(common, measurement="A serving", lists=U, candidates_per_list=L, reps=reps_a,
                              call_ms=round(ms_a, 4), users_per_s=U / (ms_a / 1e3), phase_ms=ph_a,
                              kernel_launches=la_a, recommend_loop_host_s=round(loop_s, 4),
                              recommend_loop_users_per_s=U / loop_s, recommend_batch_host_s=round(batch_s, 4),
                              single_1x1000_call_ms=round(ms_1, 4), single_phase_ms=ph_1, single_reps=reps_1,
                              oracle_check="passed")

    # ---- B: uniform eval against mr_rank_eval ----------------------------------------------------------------------
    ev_users, ev_items, group = bench.synth_eval(wl, nu, 3)
    G = ev_users.size
    lists_b = ListsCall(eng, ev_users, np.arange(G + 1, dtype=np.int64) * group, ev_items, k,
                        targets=np.full(G, group - 1, np.int32))
    d_eu, d_ei = torch.from_numpy(ev_users).cuda(), torch.from_numpy(ev_items).cuda()
    pos_e = torch.empty(G, dtype=torch.int32, device="cuda")
    sums_e = torch.zeros(2, dtype=torch.float32, device="cuda")
    nb = int(nat.lib.mr_rank_eval_workspace_bytes(C.byref(eng._model), G, group))
    ws_e = torch.empty(nb, dtype=torch.uint8, device="cuda")

    def rank_eval():
        nat.check(nat.lib.mr_rank_eval(C.byref(eng._model), _engine._ptr(d_eu), _engine._ptr(d_ei), G, group, k, None,
                                       _engine._ptr(pos_e), None, _engine._ptr(sums_e), _engine._ptr(ws_e), nb,
                                       lists_b.stream), "mr_rank_eval")

    (ms_l, ph_l, _, reps_b), (ms_e, ph_e, _, _) = timed([lists_b, rank_eval], args.seconds)
    same = bool(torch.equal(lists_b.pos, pos_e))
    if not same:
        sys.exit("rank_lists_bench: positions differ from mr_rank_eval")
    rows_b = G * group
    results["uniform_eval"] = dict(common, measurement="B uniform eval", lists=G, candidates_per_list=group,
                                   rows=rows_b, reps=reps_b, rank_lists_ms=round(ms_l, 4), rank_eval_ms=round(ms_e, 4),
                                   rank_lists_rows_per_s=rows_b / (ms_l / 1e3),
                                   rank_eval_rows_per_s=rows_b / (ms_e / 1e3),
                                   ratio_to_rank_eval=round(ms_e / ms_l, 4), bar=0.8, positions_identical=same,
                                   rank_lists_phase_ms=ph_l, rank_eval_phase_ms=ph_e)

    # ---- C: ragged eval ------------------------------------------------------------------------------------------
    Uc = 20000
    lens = np.floor(np.exp(rng.uniform(0.0, np.log(ni + 1), Uc))).astype(np.int64).clip(1, ni)
    rp_c = np.zeros(Uc + 1, np.int64)
    rp_c[1:] = np.cumsum(lens)
    it_c = rng.integers(0, ni, int(rp_c[-1])).astype(np.int32)
    lists_c = ListsCall(eng, rng.integers(0, nu, Uc).astype(np.int32), rp_c, it_c, k,
                        targets=(rng.random(Uc) * lens).astype(np.int32))
    ms_c, ph_c, la_c, reps_c = timed([lists_c], args.seconds)[0]
    results["ragged_eval"] = dict(common, measurement="C ragged eval", lists=Uc, rows=int(rp_c[-1]),
                                  min_len=int(lens.min()), max_len=int(lens.max()), reps=reps_c,
                                  call_ms=round(ms_c, 4), rows_per_s=int(rp_c[-1]) / (ms_c / 1e3), phase_ms=ph_c,
                                  rank_share=round(ph_c.get("rank", 0.0) / sum(ph_c.values()), 4),
                                  kernel_launches=la_c)
    for key, r in results.items():
        line = json.dumps(r)
        print(line)
        if args.out_dir:
            os.makedirs(args.out_dir, exist_ok=True)
            with open(os.path.join(args.out_dir, "r04_rank_lists_{}.json".format(key)), "w") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
