#!/usr/bin/env python
"""Benchmark of the NeuMF train step (BASELINE.json metric: NCF train samples/sec) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload ml-20m|ml-1m|large-sharded] [--impl reference]
                    [--dump-outputs DIR]

One "step" = the device negative sampler over the step's positives + one optimisation step (forward + BCE +
backward + deterministic embedding-gradient reduction + legacy-Keras dense Adam + train-batch HR/DCG).  `value`
includes the sampler, `value_excl_sampler` does not (SURVEY 8d).  N > 1 runs under torchrun, one rank per GPU, weak
scaling (every rank has its own batch of the same size), gradients summed over NCCL.  Prints ONE JSON line on rank 0.

`--dump-outputs DIR` (ml-20m / ml-1m) writes what the last headline step computed as DIR/<name>.npy, so that two builds
run with the same arguments (hence the same seeded inputs) can be compared output for output: the step outputs, the
batch the device sampler drew, and the weights after the step (tables larger than DUMP_TABLE_ROWS rows as a fixed,
seeded sample of rows, with the row ids beside them).

`--impl reference` times the CPU restatement of the reference's Keras path (oracle/, NumPy fp32, all host threads
BLAS will use) on a bounded sample of the same workload; TensorFlow is not installable here, so this is the "port"
kind of baseline (see DESIGN.md).
"""

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "movierecommender-tf-trt_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

WORKLOADS = {
    # BASELINE.json configs[2]: ML-20M shape, embed dim 64 (GMF), MLP 256-128-64 (SURVEY 8: C-20M)
    "ml-20m": dict(num_users=138493, num_items=26744, layers=[256, 128, 64], mf_dim=64, negs=4, ratings=20000263,
                   batch=5 * 2 ** 18, eval_negs=99, k_eval=10, cpu_batch=5 * 2 ** 13, cpu_eval_users=2048),
    # BASELINE.json configs[1]: ML-1M shape, reference default tower + GMF 8
    "ml-1m": dict(num_users=6040, num_items=3706, layers=[64, 32, 16, 8], mf_dim=8, negs=4, ratings=1000209,
                  batch=5 * 2 ** 16, eval_negs=99, k_eval=10, cpu_batch=5 * 2 ** 14, cpu_eval_users=6040),
    # BASELINE.json configs[4]: synthetic large NeuMF, embed dim 128, tables ROW-SHARDED over the GPUs (owner =
    # row % world), all-to-all of gathered rows and of their gradients; needs --gpus >= 2 (torchrun)
    "large-sharded": dict(num_users=10_000_000, num_items=1_000_000, layers=[256, 128, 64], mf_dim=128, negs=4,
                          batch=5 * 2 ** 18, eval_negs=99, k_eval=10, cpu_batch=5 * 2 ** 12, cpu_eval_users=256,
                          sharded=True),
}
METRIC = "ncf_train_samples_per_sec"
UNIT = "samples/s"

# stdout carries exactly ONE JSON line.  Libraries print there too (NCCL's "NCCL version ..." banner under torchrun),
# so file descriptor 1 is pointed at stderr for the whole run and the line goes out through the saved descriptor.
_REAL_STDOUT = None


def _claim_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def synth_batches(wl, n_batches, seed, rows=None):
    """MovieLens-shaped synthetic batches (SURVEY 8d): users with a lognormal activity tail, positive
    items Zipf-distributed over a fixed permutation, negatives uniform, generator layout
    (users repeated per group, negatives first, positive last, labels [0]*negs+[1])."""
    rng = np.random.default_rng(seed)
    nu, ni, negs = wl["num_users"], wl["num_items"], wl["negs"]
    rows = wl["batch"] if rows is None else rows
    groups = rows // (negs + 1)
    act = 20.0 + rng.lognormal(3.0, 1.0, nu)
    act_cdf = np.cumsum(act / act.sum())
    zipf = 1.0 / (np.arange(ni) + 1.0)
    zipf_cdf = np.cumsum(zipf / zipf.sum())
    perm = rng.permutation(ni)
    out = []
    for _ in range(n_batches):
        u = np.minimum(np.searchsorted(act_cdf, rng.random(groups)), nu - 1).astype(np.int32)
        pos = perm[np.minimum(np.searchsorted(zipf_cdf, rng.random(groups)), ni - 1)].astype(np.int32)
        items = rng.integers(0, ni, (groups, negs + 1), dtype=np.int32)
        items[:, -1] = pos
        users = np.repeat(u, negs + 1)
        y = np.tile(np.array([0] * negs + [1], np.float32), groups)
        out.append((users, items.reshape(-1), y))
    return out


def synth_ratings(wl, seed):
    """MovieLens-shaped (user, item) pairs for the negative sampler's per-user item lists (SURVEY 8d): per-user
    counts 20 + a lognormal tail scaled to the shape's number of ratings, items Zipf(~1) over a fixed permutation
    (repeats inside a user are dropped by the CSR build).  Returns int32 arrays."""
    rng = np.random.default_rng(seed)
    nu, ni, n = wl["num_users"], wl["num_items"], wl["ratings"]
    tail = rng.lognormal(3.0, 1.0, nu)
    extra = max(n - 20 * nu, 0)
    counts = 20 + np.floor(tail * (extra / tail.sum())).astype(np.int64)
    counts = np.minimum(counts, ni // 2)
    users = np.repeat(np.arange(nu, dtype=np.int32), counts)
    zipf = 1.0 / (np.arange(ni) + 1.0)
    cdf = np.cumsum(zipf / zipf.sum())
    perm = rng.permutation(ni).astype(np.int32)
    items = perm[np.minimum(np.searchsorted(cdf, rng.random(users.size)), ni - 1)]
    return users, items


def synth_eval(wl, n_users, seed):
    rng = np.random.default_rng(seed)
    group = wl["eval_negs"] + 1
    users = np.arange(n_users, dtype=np.int32) % wl["num_users"]
    items = rng.integers(0, wl["num_items"], n_users * group, dtype=np.int32)
    return users, items, group


def model_params(wl, rows):
    n = len(wl["layers"])
    return {"num_users": wl["num_users"], "num_items": wl["num_items"], "layers_sizes": wl["layers"],
            "layers_l2reg": [0] * n, "optimizer": "adam", "lr": 0.001, "beta_1": 0.9, "beta_2": 0.999,
            "batch_size": rows, "num_negs_per_pos": wl["negs"],
            "batch_size_eval": (wl["eval_negs"] + 1) * 2, "num_negs_per_pos_eval": wl["eval_negs"],
            "k": wl["negs"] + 1, "mf_dim": wl["mf_dim"], "adam_mode": "dense", "seed": 1}


def algorithmic_bytes(wl, rows):
    """SURVEY 8(d): A_train = B*(4*(d_U+d_I)+12) + 24*(rows of both tables, dense-Adam form) + 24*P_d;
    the fused tile kernel alone moves the first term."""
    L, f = wl["layers"], wl["mf_dim"]
    d_u = L[0] // 2
    d_i = L[0] - d_u
    dU, dI = d_u + f, d_i + f
    p_dense = sum(L[i - 1] * L[i] + L[i] for i in range(1, len(L))) + f + L[-1] + 1
    tile = rows * (4 * (dU + dI) + 12)
    step = tile + 24 * (wl["num_users"] * dU + wl["num_items"] * dI) + 24 * p_dense
    f_fwd = 2 * (sum(L[i - 1] * L[i] for i in range(1, len(L))) + L[-1] + f) + f
    eval_per_user = 4 * dU + (wl["eval_negs"] + 1) * (4 * dI + 4) + 4
    return dict(tile=tile, step=step, flops_step=3 * rows * f_fwd, f_fwd=f_fwd, eval_per_user=eval_per_user)


PHASE_KERNELS = {
    "fused_tile": "neumf_fused_train_kernel (tcgen05, 3 x bf16: H1 gather, layer-2 forward, head + BCE, dW2, backward, staged rows)",
    "sampler": "sample_negatives_kernel (Philox4x32-10, uniform without replacement over the complement of the user's items)",
    "tile_train": "neumf_tile_kernel<TM,true> (SIMT fused gather+tower+head+BCE+backward)",
    "tile_forward": "neumf_tile_kernel<TM,false> (SIMT fused forward)",
    "tc_dense_fwd": "tc_dense_kernel<A_GATHER|A_DENSE|A_PROJ,EPI_BIAS_RELU|EPI_HEAD_DOT> (tcgen05 3xTF32 forward layers)",
    "h1_gather": "h1_from_projection_kernel (item-projected first layer: gather + add + ReLU of the projected rows)",
    "tc_dense_bwd": "tc_dense_kernel<A_DENSE,EPI_MASK|EPI_STAGE> (tcgen05 3xTF32 backward-activation layers)",
    "tc_wgrad": "tc_wgrad_kernel (tcgen05 3xTF32 weight gradients, MN-major operands)",
    "head": "head_kernel (GMF + output unit + sigmoid + BCE + their gradients)",
    "segreduce": "segreduce_level_kernel (deterministic segmented reduction of row gradients)",
    "sort": "radix_hist/rowscan/scatter kernels",
    "optimizer": "optimizer_flat_kernel (legacy-Keras Adam sweep)",
}


def phase_interface_bytes(wl, rows, grouped=False, projected=False, user_projected=False):
    """Bytes each phase must move per step GIVEN its interface (inputs read once, outputs written once) --
    the per-kernel roofline numerator.  The SURVEY 8(d) whole-step algorithmic figure (which charges no
    intermediate) is reported separately as step_roofline.  grouped: the launch sequence for grouped batches
    (user half of the first layer once per group of negs+1 rows)."""
    L, f, n = wl["layers"], wl["mf_dim"], len(wl["layers"])
    d_u = L[0] // 2
    d_i = L[0] - d_u
    dU, dI = d_u + f, d_i + f
    pairs = [(L[l - 1], L[l]) for l in range(1, n)]
    tables = wl["num_users"] * dU + wl["num_items"] * dI
    if grouped:
        G = rows // (wl["negs"] + 1)
        L1 = L[1]
        later = [(L[l - 1], L[l]) for l in range(2, n)]
        if projected:
            # item half of the first layer once per ITEM: Pi = E_item . W1i over the item table, per row a gather of
            # the (L2-resident) Pi row + the group's Zu row -> H1 and its ReLU bits; backward on per-item sums of dZ1
            ni = wl["num_items"]
            nu = wl["num_users"] if user_projected else G  # rows of the user-half GEMMs: users, or groups
            return {
                "tc_dense_fwd": ni * 4 * (d_i + L1) + nu * 4 * (d_u + L1) + rows * sum(4 * (a + b) for a, b in later),
                # ids in, H1 + its ReLU bits out; the projected rows are L2-resident, one user-side row per group
                "h1_gather": rows * (4 + 4 * L1 + L1 // 8) + G * (4 * L1 + (4 if user_projected else 0)),
                "head": rows * (8 * L[-1] + 8 * f + 16) + G * (8 * f + 4),
                "tc_wgrad": ni * 4 * (d_i + L1) + nu * (4 + 4 * (d_u + L1)) + rows * sum(4 * (a + b) for a, b in later),
                "tc_dense_bwd": rows * sum(4 * (a + b) + 4 * a for a, b in later) + ni * 4 * (L1 + d_i) + nu * 4 * (L1 + d_u),
                "misc": rows * 4 * L1 + G * 4 * L1,
                # (user-projected steps reduce the user side on the side stream, under the item side: not counted here)
                "segreduce": (0 if user_projected else G * 2 * (4 * dU + 8)) + rows * 2 * (4 * dI + 8),
                "optimizer": 28 * tables,
            }
        return {
            # Zu (G rows: user row in, L1 out) + first layer on the item row (+ one Zu row per group) + later layers
            "tc_dense_fwd": G * 4 * (d_u + L1) + rows * (8 + 4 * (d_i + L1)) + G * 4 * L1 + rows * sum(4 * (a + b) for a, b in later),
            # GMF user row once per group, its gradient once per group
            "head": rows * (8 * L[-1] + 8 * f + 16) + G * (8 * f + 4),
            "tc_wgrad": rows * (4 + 4 * (d_i + L1)) + G * (4 + 4 * (d_u + L1)) + rows * sum(4 * (a + b) for a, b in later),
            # later layers as before; first layer: item half per row, user half per group on the group sums
            "tc_dense_bwd": rows * sum(4 * (a + b) + 4 * a for a, b in later) + rows * 4 * (L1 + d_i) + G * 4 * (L1 + d_u),
            "misc": rows * 4 * L1 + G * 4 * L1,  # group sums of dZ1
            "segreduce": G * 2 * (4 * dU + 8) + rows * 2 * (4 * dI + 8),
            "sort": (G + rows) * 2 * 16,
            "optimizer": 28 * tables,
        }
    return {
        "tile_train": rows * (4 * (dU + dI) + 12),
        "tc_dense_fwd": rows * (8 + sum(4 * (a + b) for a, b in pairs)),
        "head": rows * (8 * L[-1] + 16 * f + 20),
        "tc_wgrad": rows * (8 + sum(4 * (a + b) for a, b in pairs)),
        "tc_dense_bwd": rows * sum(4 * (a + b) + (4 * a if i > 0 else 0) for i, (a, b) in enumerate(pairs)),
        "segreduce": rows * 2 * (4 * (dU + dI) + 8),
        "sort": rows * 2 * 16,
        "optimizer": 28 * tables,
    }


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def measured_tensor_peak():
    """Dense bf16 TFLOP/s sustained inside a long step (MEASURED_PEAKS.json), else the profiling guide's fallback."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f).get("bf16_tflops_sustained", 1400.0))
    return 1400.0


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.path = gpu_index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(prefix="clocks_", suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                parts = [x.strip() for x in line.split(",")]
                if len(parts) < 7:
                    continue
                try:
                    sm.append(float(parts[0]))
                    mx.append(float(parts[1]))
                except ValueError:
                    continue
                for name, val in zip(names, parts[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


# ---------------------------------------------------------------------------------------------------
# CPU restatement (oracle) timing: cpu_baseline leg and --impl reference
# ---------------------------------------------------------------------------------------------------

def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        n = [i.get("num_threads", 1) for i in threadpool_info() if i.get("user_api") == "blas"]
        return int(max(n)) if n else 1
    except Exception:
        return int(os.cpu_count() or 1)


def time_oracle_train(wl, steps, warmup):
    """Oracle train steps (NumPy fp32: forward, BCE, backward with batch-order scatter, legacy-Keras
    dense Adam over the full tables, train-batch HR/DCG) on `cpu_batch` rows per step."""
    from oracle import movierec_oracle as o
    rows = wl["cpu_batch"]
    params = model_params(wl, rows)
    w = o.init_weights(wl["num_users"], wl["num_items"], wl["layers"], wl["mf_dim"], np.random.default_rng(1))
    st = o.new_opt_state(w)
    batches = synth_batches(wl, 2, seed=0, rows=rows)
    for i in range(warmup):
        o.train_step(w, st, *batches[i % 2], params)
    t0 = time.perf_counter()
    for i in range(steps):
        o.train_step(w, st, *batches[i % 2], params)
    dt = time.perf_counter() - t0
    return rows * steps / dt, dt / steps * 1e3, rows


def time_oracle_eval(wl, reps=2):
    from oracle import movierec_oracle as o
    w = o.init_weights(wl["num_users"], wl["num_items"], wl["layers"], wl["mf_dim"], np.random.default_rng(1))
    users, items, group = synth_eval(wl, wl["cpu_eval_users"], seed=2)
    o.evaluate_groups(w, users, items, group, wl["k_eval"])
    t0 = time.perf_counter()
    for _ in range(reps):
        o.evaluate_groups(w, users, items, group, wl["k_eval"])
    dt = (time.perf_counter() - t0) / reps
    return len(users) / dt


def run_reference(args, wl):
    """The reference arm: the CPU restatement of the reference's Keras train_on_batch (oracle/, NumPy fp32, every host
    thread BLAS uses) on the SAME workload -- same tables, tower, optimizer, batch layout -- each step a bounded
    sample of the GPU arm's rows per step (the full 1,310,720-row step takes ~15 s of NumPy), throughput in the same
    unit.  `config` is the GPU arm's; the sample size is stated in `cpu_baseline.sample` / `sample_rows_per_step`."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    value, ms, rows = time_oracle_train(wl, args.steps, args.warmup)
    threads = blas_threads()
    sample = ("oracle (NumPy fp32 restatement of the reference's Keras train_on_batch, dense Adam over the full "
              "tables) on {} of the workload's {} rows per step, {} steps".format(rows, wl["batch"], args.steps))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(args, wl), "sample_rows_per_step": rows,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "host_cores": os.cpu_count()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def config_dict(args, wl, rows_override=None):
    return {"workload": "{} shape: {} users x {} items, NeuMF layers {} mf_dim {}, {} negatives/positive, "
                        "Adam (legacy Keras, dense over tables)".format(args.workload, wl["num_users"], wl["num_items"],
                                                                       wl["layers"], wl["mf_dim"], wl["negs"]),
            "baseline_config": "BASELINE.json configs[{}]".format({"ml-20m": 2, "ml-1m": 1}.get(args.workload, 4)),
            "rows_per_step_per_gpu": wl["batch"] if rows_override is None else rows_override,
            "global_rows_per_step": (wl["batch"] if rows_override is None else rows_override) * args.gpus,
            "parallelism": "single GPU" if args.gpus == 1 else
                           "dp{} replicated tables; gradient sum + Adam + weight distribution in one kernel over NVLink "
                           "peer pointers (mr_dp_reduce_apply), optimizer state sharded by owner".format(args.gpus)
                           if args.dp_exchange != "nccl" else
                           "dp{} replicated tables, NCCL all-reduce of dense+table gradients, full Adam sweep per rank".format(args.gpus),
            "l2_policy": "working set larger than L2: 4 rotating batches; staged row gradients (~{:.1f} GB/step) and "
                         "tables+Adam state exceed the 126 MB L2".format(wl["batch"] * 4 * (sum(wl["layers"][:1]) + 2 * wl["mf_dim"]) / 1e9)}


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------

DUMP_TABLE_ROWS = 16384
DUMP_MAX_BYTES = 64 * 10 ** 6


def dump_outputs(path, step_out, batch, weights):
    """--dump-outputs: the step outputs [loss_sum, hit_sum, dcg_sum, l2_penalty, bad_ids, ...] of the last headline
    step, the (users, items, labels) batch the sampler drew for it, and the weights after it.  Ids are written as
    float64 (exact).  Rows of a table taller than DUMP_TABLE_ROWS are a sample drawn with a generator seeded by the
    table's height, so the user-side (and item-side) tables share one set of rows, stored as <table>.rows."""
    arrays = {"step_out": np.asarray(step_out, np.float64)}
    for name, t in zip(("batch_users", "batch_items", "batch_labels"), batch):
        a = t.cpu().numpy()
        arrays[name] = a.astype(np.float64 if a.dtype.kind in "iu" else np.float32)
    for name, w in weights.items():
        key = "weights." + name.replace("/", ".")
        if w.ndim == 2 and w.shape[0] > DUMP_TABLE_ROWS:
            rows = np.sort(np.random.default_rng(w.shape[0]).choice(w.shape[0], DUMP_TABLE_ROWS, replace=False))
            arrays[key + ".rows"] = rows.astype(np.float64)
            w = w[rows]
        arrays[key] = np.ascontiguousarray(w, np.float32)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit("--dump-outputs: {} bytes exceed the {}-byte limit".format(total, DUMP_MAX_BYTES))
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)

def refuse_diagnostics(args):
    """A bench value must come from the product build with no diagnostic switch: any MR_* environment variable
    (variant libraries via MR_LIB_PATH, MR_DP_OVERLAP, ...) makes the run a profiling run, allowed only with --lean."""
    found = sorted(k for k in os.environ if k.startswith("MR_"))
    if found and not args.lean:
        raise SystemExit("refusing to emit a bench value with diagnostic variables set: {} (use --lean for profiling "
                         "runs; their line is marked and carries no e2e / baseline)".format(", ".join(found)))
    return found


def time_reference_faithful():
    """BASELINE.md C1: the reference's own operating point (trainer.py:8-27: tower 64-32-16-8, batch 100, 4 negatives,
    Adam) on ML-100k-shaped data, ONE process as Keras' fit_generator default (workers=1): the oracle's NumPy train
    step fed by the restated generator (data_pipeline.py:99-150: a scan of the ratings and a setdiff per positive)."""
    from oracle import movierec_oracle as o
    nu, ni, n, negs, batch = 943, 1682, 100000, 4, 100
    rng = np.random.default_rng(0)
    users = rng.integers(0, nu, n)
    items = rng.integers(0, ni, n)
    L = [64, 32, 16, 8]
    params = {"layers_sizes": L, "layers_l2reg": [0, 0, 0, 0], "optimizer": "adam", "lr": 0.001, "beta_1": 0.9,
              "beta_2": 0.999, "num_negs_per_pos": negs, "k": 5}
    w = o.init_weights(nu, ni, L, 0, np.random.default_rng(1))
    st = o.new_opt_state(w)
    idx = rng.permutation(n)
    steps, t_gen, t_step = 60, 0.0, 0.0
    for i in range(steps + 3):
        t0 = time.perf_counter()
        (xu, xi), y = o.reference_batch(users, items, idx, i, batch, negs, ni, rng)
        t1 = time.perf_counter()
        o.train_step(w, st, xu, xi, y.astype(np.float32), params)
        t2 = time.perf_counter()
        if i >= 3:
            t_gen += t1 - t0
            t_step += t2 - t1
    return {"samples_per_sec": batch * steps / (t_gen + t_step), "samples_per_sec_excl_generation": batch * steps / t_step,
            "batch": batch, "cores": 1, "steps": steps,
            "config": "reference defaults (trainer.py:8-27): layers [64,32,16,8], batch 100, 4 negatives, Adam; ML-100k "
                      "shape (943 x 1682, 100,000 ratings); oracle NumPy step + restated generator, one process"}


def run_gpu(args, wl):
    import torch
    import torch.distributed as dist
    from movierec import _engine as eng_mod
    from movierec import _native as nat
    from movierec.model import MovierecModel

    diag_env = refuse_diagnostics(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus {} needs torchrun (one process per GPU); see the module docstring".format(args.gpus))
        args.gpus = world
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dp = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    rows = wl["batch"]
    negs = wl["negs"]
    group = negs + 1
    out_dir = tempfile.mkdtemp(prefix="movierec_bench_")
    model = MovierecModel(model_params(wl, rows), "bench", out_dir, verbose=0)
    eng = model.model.engine
    if world > 1:
        from movierec._distributed import DataParallelNeuMF
        dp = DataParallelNeuMF(eng, exchange=None if args.dp_exchange == "auto" else args.dp_exchange)
        args.dp_exchange = dp.exchange  # what the wrapper took ("auto" falls back to NCCL without symmetric memory)
        dp.broadcast_parameters(0)

    # ---- synthetic ratings -> per-user item lists on the device (what the sampler excludes); positives of a step
    # are drawn from the ratings (activity-weighted users, Zipf items), a different stream per rank
    ru, ri = synth_ratings(wl, seed=0)
    rowptr, csr = eng_mod.build_user_csr(ru, ri, wl["num_users"], wl["num_items"])
    P = rows // group
    n_batches = 4
    rng = np.random.default_rng(1000 + rank)
    positives = []
    for _ in range(n_batches):
        sel = rng.integers(0, ru.size, P)
        positives.append((torch.from_numpy(ru[sel]).to(dev), torch.from_numpy(ri[sel]).to(dev)))
    global_rows = rows * world
    draw = [0]

    def sample(i):
        pu, pi = positives[i % n_batches]
        draw[0] += 1
        return eng_mod.sample_negatives(rowptr, csr, wl["num_items"], pu, pi, 0, negs, 2 + rank, draw[0])

    def train(u, it, y):
        if dp is None:
            return eng.train_step(u, it, y, group=group, k=group, grouped=True)
        return dp.train_step(u, it, y, global_rows, group=group, k=group, grouped=True)

    resident = [sample(b) for b in range(n_batches)]                       # pre-sampled: the sampler-excluded loop
    pinned = [tuple(t.cpu().pin_memory() for t in b) for b in resident]     # ... and the end-to-end loop's host batches

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def timed(step_fn, steps, profile=False):
        sync_all()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if profile:
            nat.profile_begin()
        sync_all()
        ev0.record()
        last = None
        for i in range(steps):
            last = step_fn(i)
        ev1.record()
        sync_all()
        prof = nat.profile_end() if profile else None
        t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), last, prof

    last_batch = [None]

    def headline_step(i):
        last_batch[0] = sample(args.warmup + i)
        return train(*last_batch[0])

    for i in range(args.warmup):
        train(*sample(i))
    # ---- timed region 1 (the headline): sampler + train step, positives resident in HBM ---------------------------
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    ms_total, last, (phases, launches) = timed(headline_step, args.steps, profile=True)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:  # before region 2 trains the weights further
        dump_outputs(args.dump_outputs, last.cpu().numpy(), last_batch[0], eng.get_weights())
    # ---- timed region 2: the train step alone on pre-sampled batches -----------------------------------------------
    ms_nosampler, _, _ = timed(lambda i: train(*resident[i % n_batches]), args.steps)
    value = global_rows * args.steps / (ms_total / 1e3)
    value_nosampler = global_rows * args.steps / (ms_nosampler / 1e3)
    final = last.cpu().numpy()
    if final[4] != 0 or not np.isfinite(final[0]):
        raise SystemExit("bench produced invalid step outputs: {}".format(final))

    # ---- the weights the timed steps produced must still score like the oracle says (rank 0) -----------------------
    check = None
    if rank == 0:
        from oracle import movierec_oracle as o
        w_now = eng.get_weights()
        u0, i0, _ = resident[0]
        pick = np.random.default_rng(7).choice(rows, 4096, replace=False)
        pick_t = torch.from_numpy(pick).to(dev)
        logits = eng.forward(u0[pick_t], i0[pick_t])[0].cpu().numpy().astype(np.float64)
        want = o.forward(w_now, u0.cpu().numpy()[pick], i0.cpu().numpy()[pick])["z"].astype(np.float64)
        err, scale = float(np.max(np.abs(logits - want))), float(np.max(np.abs(want)))
        check = {"rows": 4096, "max_abs_err": err, "max_abs_logit": scale, "tolerance": 1e-5 * scale}
        if not np.isfinite(err) or err > 1e-5 * scale:
            raise SystemExit("bench weights fail the oracle check: logits differ by {:.3e} (scale {:.3e})".format(err, scale))

    # ---- end to end through the public API: host buffers in, loss out, every step ----------------------------------
    def step_e2e(i):
        u, it, y = pinned[i % n_batches]
        if dp is None:  # uploads, steps, reads the loss back; the next batch's upload runs under this step
            nxt = pinned[(i + 1) % n_batches]
            return model.model.train_on_batch([u, it], y, prefetch=([nxt[0], nxt[1]], nxt[2]))
        return dp.train_step(u, it, y, global_rows, group=group, k=group, grouped=True,
                             prefetch=pinned[(i + 1) % n_batches]).cpu()

    e2e_steps = 0 if args.lean else max(3, min(args.steps, 20))
    if not args.lean:
        step_e2e(0)
    sync_all()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        step_e2e(i + 1)
    sync_all()
    e2e_s = max(time.perf_counter() - t0, 1e-9)
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = global_rows * e2e_steps / float(t.item())

    # ---- ranking eval: HR@10 users/sec (second half of the BASELINE metric), rank 0's replica ----------------------
    eval_obj = None
    if rank == 0 and not args.lean:
        n_eval = wl["num_users"]
        eu, ei, egroup = synth_eval(wl, n_eval, seed=2)
        eu_d, ei_d = torch.from_numpy(eu).to(dev), torch.from_numpy(ei).to(dev)
        for _ in range(2):
            eng.rank_eval(eu_d, ei_d, egroup, wl["k_eval"])
        torch.cuda.synchronize(dev)
        nat.profile_begin()
        reps = 7
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a, b in evs:  # one event pair per sweep; the median is reported (host hiccups show in single sweeps)
            a.record()
            pos, sums, _, _ = eng.rank_eval(eu_d, ei_d, egroup, wl["k_eval"])
            b.record()
        torch.cuda.synchronize(dev)
        eph, _ = nat.profile_end()
        ems = float(np.median([a.elapsed_time(b) for a, b in evs]))
        # end to end: pinned host ids in, HR / NDCG back on the host
        eu_p, ei_p = torch.from_numpy(eu).pin_memory(), torch.from_numpy(ei).pin_memory()
        e2e_t = []
        for _ in range(4):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            pos2, sums2, _, _ = eng.rank_eval(eu_p, ei_p, egroup, wl["k_eval"])
            hr_host = float(sums2.cpu()[0])
            e2e_t.append(time.perf_counter() - t0)
        ab = algorithmic_bytes(wl, rows)
        peak, peak_kind = measured_peaks()
        fwd_ms = sum(eph[k][0] for k in ("tile_forward", "tc_dense_fwd", "h1_gather", "head") if k in eph) / reps
        ach = ab["eval_per_user"] * n_eval / (max(fwd_ms, 1e-9) / 1e3) / 1e9
        eval_obj = {"metric": "hr10_eval_users_per_sec", "value": n_eval / (ems / 1e3), "unit": "users/s",
                    "users": n_eval, "candidates_per_user": egroup, "k": wl["k_eval"], "ms": ems,
                    "hr_at_k": float(sums[0].item()) / n_eval, "ndcg_at_k": float(sums[1].item()) / n_eval,
                    "e2e": {"value": n_eval / float(np.median(e2e_t[1:])), "unit": "users/s",
                            "h2d_bytes_per_sweep": int(eu.nbytes + ei.nbytes), "d2h_bytes_per_sweep": 8,
                            "api": "NeuMFEngine.rank_eval on pinned host ids (MovierecModel.evaluate), sums read back"},
                    "phase_ms": {k: v[0] / reps for k, v in eph.items() if v[1]},
                    "roofline": {"bound": "hbm", "kernel": "forward kernels (tcgen05 layers + head, or the SIMT tile kernel)",
                                 "forward_ms": fwd_ms, "achieved": ach, "peak": peak,
                                 "unit": "GB/s", "frac": ach / peak, "peak_kind": peak_kind, "traffic": None}}
        assert abs(hr_host - float(sums[0].item())) < 0.5

    # ---- N >= 2: the row-sharded configuration (BASELINE.json configs[4]) rides on the same line, the way the ranking
    # eval rides on the N = 1 line, so that the scaling record sees it at every N
    sharded_obj = None
    if world > 1 and not args.lean:
        resident = pinned = positives = None  # (free the replicated run's batches)
        torch.cuda.empty_cache()
        sharded_obj = sharded_measure(WORKLOADS["large-sharded"], steps=max(5, min(args.steps, 10)), warmup=3, dev=dev,
                                      rank=rank, world=world, e2e=False)
    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    ab = algorithmic_bytes(wl, rows)
    peak, peak_kind = measured_peaks()
    tensor_peak = measured_tensor_peak()
    step_ms = ms_total / args.steps
    grouped_seq = bool(eng.uses_tensor_cores()) and wl["mf_dim"] + wl["layers"][-1] <= 128
    projected_seq = grouped_seq and bool(eng.uses_item_projection(rows))
    uprojected_seq = projected_seq and bool(eng.uses_user_projection(rows, group))
    pbytes = phase_interface_bytes(wl, rows, grouped=grouped_seq, projected=projected_seq, user_projected=uprojected_seq)
    pbytes["fused_tile"] = ab["tile"]  # SURVEY 8(d): B * (4 * (d_U + d_I) + 12), the per-row term of A_train
    phase_table = {}
    for name, (ms, cnt) in phases.items():
        if not cnt:
            continue
        per_step = ms / args.steps
        row = {"ms_per_step": per_step, "launch_groups_per_step": cnt / args.steps, "share_of_step": per_step / step_ms}
        if name in pbytes:
            row["interface_bytes_per_step"] = pbytes[name]
            row["gbs"] = pbytes[name] / (per_step / 1e3) / 1e9
            row["frac_of_hbm_peak"] = row["gbs"] / peak
        phase_table[name] = row
    dom = max(phase_table, key=lambda k: phase_table[k]["ms_per_step"])
    dom_groups = max(phases[dom][1], 1)
    dom_avg_ms = phases[dom][0] / dom_groups            # one launch group = the kernel(s) of one phase interval
    small_tower = bool(eng.uses_small_tower(rows, group))
    kernels = dict(PHASE_KERNELS)
    if small_tower:  # the default tower's step reuses the phase slots of the tensor-core sequence
        kernels.update(fused_tile="small_tower_train_kernel<5> (fp32 CUDA cores, thread per group: projected first layer, "
                                  "layers 2-3, head + BCE, backward, weight gradients, staged rows) + wait for the id sorts",
                       tc_dense_fwd="small_rows_gemm_kernel (Pi, Pu over the tables)",
                       tc_dense_bwd="small_rows_gemm_kernel (dE = S . W1^T over the tables)",
                       tc_wgrad="small_table_wgrad_kernel (dW1 = E^T . S)")
    dominant = {"phase": dom, "kernel": kernels.get(dom, dom), "avg_launch_ms": dom_avg_ms,
                "launches_timed": dom_groups, "share_of_step": phase_table[dom]["share_of_step"]}
    if dom in pbytes:
        dom_bytes = pbytes[dom] * args.steps / dom_groups
        dominant.update(algorithmic_bytes_per_launch=dom_bytes, achieved_gbs=dom_bytes / (dom_avg_ms / 1e3) / 1e9,
                        frac_of_hbm_peak=dom_bytes / (dom_avg_ms / 1e3) / 1e9 / peak)
    if dom == "fused_tile" and small_tower:
        # per row: 656 multiply-adds forward, the same again for the data gradients and for the weight gradients
        dominant.update(bound="instruction issue / launch latency (fp32 CUDA cores); HBM traffic is ~0.1 GB per step",
                        fp32_tflops=3 * 2 * 656.0 * rows * args.steps / dom_groups / (dom_avg_ms / 1e3) / 1e12)
    elif dom == "fused_tile":
        # three GEMMs of 2 * 128 * 64 flops per row, each fp32 product = six bf16 part products on the tensor cores
        tflops = 6.0 * 3 * 2 * 128 * 64 * rows * args.steps / dom_groups / (dom_avg_ms / 1e3) / 1e12
        dominant.update(bound="hbm (per-row gather + staged gradient rows); tensor time is ~3/4 of the HBM time",
                        tensor_tflops_bf16=tflops, frac_of_tensor_peak=tflops / tensor_peak)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get(args.workload, {}).get("step_dram_bytes")
    if args.lean:
        cpu_value, cpu_ms, cpu_rows, cpu_eval, faithful = None, None, 0, None, None
    else:
        cpu_value, cpu_ms, cpu_rows = time_oracle_train(wl, steps=4, warmup=1)
        cpu_eval = time_oracle_eval(wl)
        faithful = time_reference_faithful()
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": config_dict(args, wl),
        "value_excl_sampler": value_nosampler, "ms_per_step_excl_sampler": ms_nosampler / args.steps,
        "clocks": clk,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": rows * 12, "d2h_bytes_per_step": 32,
                "steps": e2e_steps,
                "api": "MovierecModel.model.train_on_batch([x_users, x_items], y, prefetch=next batch) on pinned host arrays: "
                       "the next batch's upload runs under the current step; the loss is read back every step"
                if dp is None else "DataParallelNeuMF.train_step on pinned host arrays"},
        "gpu_launches": launches,
        "launch_sequence": {"grouped": grouped_seq, "item_projection": projected_seq, "user_projection": uprojected_seq,
                            "fused_tile_kernel": "fused_tile" in phase_table and not small_tower,
                            "small_tower_kernel": small_tower},
        # SURVEY 8(d): the whole step's algorithmic bytes over the step time, against the measured copy bandwidth
        "roofline": {"bound": "hbm", "scope": "whole train step (sampler included), SURVEY 8(d) A_train",
                     "kernel": kernels.get(dom, dom), "achieved": ab["step"] / (step_ms / 1e3) / 1e9, "peak": peak,
                     "unit": "GB/s", "frac": ab["step"] / (step_ms / 1e3) / 1e9 / peak, "traffic": traffic,
                     "peak_kind": peak_kind, "algorithmic_bytes_per_step": ab["step"],
                     "fp32_tflops": ab["flops_step"] / (step_ms / 1e3) / 1e12, "dominant_kernel": dominant},
        "phases": phase_table,
        "phase_ms_per_step": {k: v[0] / args.steps for k, v in phases.items() if v[1]},
        "oracle_check": check,
        "cpu_baseline": {"value": cpu_value, "unit": UNIT, "cores": blas_threads(), "kind": "port",
                         "host_cores": os.cpu_count(),
                         "sample": "oracle NumPy fp32 train step (dense Adam over the full tables) on {} rows/step of the "
                                   "same workload, 4 steps after 1 warm-up; eval: {} users x {} candidates".format(
                                       cpu_rows, wl["cpu_eval_users"], wl["eval_negs"] + 1),
                         "eval_users_per_sec": cpu_eval, "reference_faithful": faithful},
        "eval": eval_obj,
        "sharded": sharded_obj,
        "final_loss": float(final[0]) / rows,
    }
    if args.lean:
        line["lean"] = True
        line["diagnostic_env"] = diag_env
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def sharded_measure(wl, steps, warmup, dev, rank, world, e2e=True):
    """The row-sharded step (BASELINE.json configs[4]) on an initialised process group: returns rank 0's summary
    (all ranks must call).  Tables row-sharded over the ranks (owner = row % world), every rank trains on its own
    batch of `batch` rows (weak scaling)."""
    import torch
    import torch.distributed as dist
    from movierec import _native as nat
    from movierec._distributed import ShardedNeuMF

    rows, group = wl["batch"], wl["negs"] + 1
    groups = rows // group
    global_rows = rows * world
    sh = ShardedNeuMF(wl["num_users"], wl["num_items"], wl["layers"], mf_dim=wl["mf_dim"], optimizer="adam", lr=1e-3,
                      max_local_rows=1 << 21, seed=None)
    n_batches = 4
    rng = np.random.default_rng(1000 + rank)  # SURVEY 8(d): ids drawn uniformly per step (no CSR at this size)
    host = []
    for _ in range(n_batches):
        u = np.repeat(rng.integers(0, wl["num_users"], groups, dtype=np.int32), group)
        it = rng.integers(0, wl["num_items"], rows, dtype=np.int32)
        y = np.tile(np.array([0] * wl["negs"] + [1], np.float32), groups)
        host.append((u, it, y))
    pinned = [tuple(torch.from_numpy(a).pin_memory() for a in b) for b in host]
    resident = [tuple(t.to(dev) for t in b) for b in pinned]

    def step(bufs, i):
        u, it, y = bufs[i % n_batches]
        return sh.train_step(u, it, y, global_rows, group=group, k=group, grouped=True)

    def sync_all():
        torch.cuda.synchronize(dev)
        dist.barrier()
        torch.cuda.synchronize(dev)

    for i in range(warmup):
        step(resident, i)
    sync_all()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nat.profile_begin()
    sync_all()
    ev0.record()
    last = None
    for i in range(steps):
        last = step(resident, warmup + i)
    ev1.record()
    sync_all()
    phases, launches = nat.profile_end()
    t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    final = last.cpu().numpy()
    if int(final[4]) != 0 or not np.isfinite(final[0]):
        raise SystemExit("sharded bench produced invalid step outputs: {}".format(final))
    e2e_value, e2e_steps = None, 0
    if e2e:  # end to end: pinned host arrays in, step outputs back, every step
        e2e_steps = max(3, min(steps, 10))
        step(pinned, 0).cpu()
        sync_all()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            step(pinned, i + 1).cpu()
        sync_all()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_value = global_rows * e2e_steps / float(t.item())
    dist.barrier()
    del sh
    torch.cuda.empty_cache()
    step_ms = ms_total / steps
    L, f = wl["layers"], wl["mf_dim"]
    row_bytes = 4 * (L[0] + 2 * f)  # one user row + one item row (MLP + GMF parts)
    kernel_ms = sum(ms / steps for ms, cnt in phases.values() if cnt)
    return {"value": global_rows * steps / (ms_total / 1e3), "unit": UNIT, "ms_per_step": step_ms, "steps": steps,
            "warmup": warmup, "n_gpus": world, "rows_per_step_per_gpu": rows, "global_rows_per_step": global_rows,
            "workload": "large-sharded: {} users x {} items, NeuMF layers {} mf_dim {}, {} negatives/positive, sparse-row "
                        "Adam at the owners (BASELINE.json configs[4])".format(wl["num_users"], wl["num_items"], L, f, wl["negs"]),
            "parallelism": "tables row-sharded over {} ranks (owner = row % world)".format(world),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": rows * 12, "d2h_bytes_per_step": 32,
                    "steps": e2e_steps, "api": "ShardedNeuMF.train_step on pinned host arrays"},
            "gpu_launches": launches, "final_loss": float(final[0]) / rows,
            "exchange": {"bytes_per_step_per_rank_upper_bound": 2 * 2 * rows * row_bytes // 2,
                         "library_kernel_ms_per_step": kernel_ms,
                         "routing_and_collectives_ms_per_step": step_ms - kernel_ms},
            "phase_ms_per_step": {k: v[0] / steps for k, v in phases.items() if v[1]}}


def run_sharded(args, wl):
    """BASELINE.json configs[4] as the headline of the line (`--workload large-sharded`, torchrun, --gpus >= 2)."""
    import torch
    import torch.distributed as dist

    refuse_diagnostics(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world < 2:
        raise SystemExit("--workload large-sharded shards the tables over the ranks: run it under torchrun with "
                         "--gpus >= 2 (python -m torch.distributed.run --nproc-per-node N bench.py --gpus N --workload large-sharded)")
    args.gpus = world
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", device_id=dev)
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    r = sharded_measure(wl, args.steps, args.warmup, dev, rank, world)
    clk = clocks.stop() if rank == 0 else None
    if rank != 0:
        dist.destroy_process_group()
        return
    peak, peak_kind = measured_peaks()
    L, f = wl["layers"], wl["mf_dim"]
    # SURVEY 8(d), sparse-row form: per-row gathers + Adam on the touched rows (every id distinct at this table size)
    a_step = wl["batch"] * (4 * (L[0] + 2 * f) + 12) + 24 * (wl["batch"] // (wl["negs"] + 1) + wl["batch"]) * (L[0] // 2 + f)
    line = {
        "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": r["workload"], "baseline_config": "BASELINE.json configs[4]",
                   "rows_per_step_per_gpu": r["rows_per_step_per_gpu"], "global_rows_per_step": r["global_rows_per_step"],
                   "parallelism": r["parallelism"] + "; per step and side: ids to the owners, rows gathered over peer "
                                  "pointers (NVLink), gradient rows back to the owners, all-reduce of the dense tower",
                   "table_bytes_total": 4 * (wl["num_users"] + wl["num_items"]) * (L[0] // 2 + f) * 3,
                   "l2_policy": "working set larger than L2: 4 rotating batches of uniformly drawn ids over 11 GB of tables"},
        "clocks": clk, "e2e": r["e2e"], "gpu_launches": r["gpu_launches"],
        "roofline": {"bound": "hbm", "scope": "whole step per GPU, SURVEY 8(d) A_train in sparse-row form",
                     "kernel": "row-sharded step (exchange + cache-slot train step + owner-side sparse-row Adam)",
                     "achieved": a_step / (r["ms_per_step"] / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": a_step / (r["ms_per_step"] / 1e3) / 1e9 / peak, "traffic": None, "peak_kind": peak_kind,
                     "algorithmic_bytes_per_step": a_step},
        "exchange": r["exchange"], "phase_ms_per_step": r["phase_ms_per_step"],
        "cpu_baseline": {"value": None, "unit": UNIT, "cores": 0, "kind": "port",
                         "sample": "not timed: the CPU baseline leg runs at N=1 only and this workload needs N >= 2"},
        "final_loss": r["final_loss"],
    }
    emit(line)
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)   # ~0.3 s timed at N=1: several nvidia-smi clock samples
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dp-exchange", default="auto", choices=["auto", "peer", "nccl"],
                    help="N > 1: fused peer-memory reduce + optimizer kernel (auto: wherever torch symmetric memory works) "
                         "or NCCL all-reduce + full sweep")
    ap.add_argument("--workload", default="ml-20m", choices=sorted(WORKLOADS))
    ap.add_argument("--lean", action="store_true",
                    help="profiling runs (ncu): skip the e2e, eval and CPU-baseline legs; not a bench value")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the step outputs, sampled batch and weights of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or WORKLOADS[args.workload].get("sharded")):
        ap.error("--dump-outputs covers the replicated-table GPU workloads (ml-20m, ml-1m)")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3  # timing rule: at least 3 warm-up steps
    wl = WORKLOADS[args.workload]
    _claim_stdout()
    if args.impl == "reference":
        run_reference(args, wl)
    elif wl.get("sharded"):
        run_sharded(args, wl)
    else:
        run_gpu(args, wl)


if __name__ == "__main__":
    main()
