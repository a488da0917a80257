"""Host-side logic of the drop-in Python face and the C-ABI surface.  CPU only (no compute calls)."""

import copy
import ctypes
import json
import os
import re

import numpy as np
import pandas as pd
import pytest

from movierec import data_pipeline, model, trainer
from movierec import _native as nat
from movierec.util import movielens_utils as ml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

TEST_PARAMS = {  # reference test/test_model.py:8-26
    "num_users": 5, "num_items": 10, "layers_sizes": [6, 4], "layers_l2reg": [0.01, 0.01],
    "optimizer": "adam", "lr": 0.001, "beta_1": 0.9, "beta_2": 0.999,
    "batch_size": 8, "num_negs_per_pos": 3, "batch_size_eval": 10, "num_negs_per_pos_eval": 4, "k": 4,
}


@pytest.fixture(scope="module")
def ref(golden_dir):
    with open(os.path.join(golden_dir, "reference_tests.json")) as f:
        return json.load(f)


# ---- C ABI --------------------------------------------------------------------------------------

def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "movierec_b200.h")).read()
    declared = set(re.findall(r"\b(mr_[a-z_0-9]+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert declared == set(nat.SIGNATURES), declared ^ set(nat.SIGNATURES)
    lib = ctypes.CDLL(nat.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert nat.version() == int(re.search(r"#define MR_VERSION (\d+)", header).group(1))
    # the product library exports no diagnostics; those live in their own library with their own header
    from movierec import _diag
    diag_header = open(os.path.join(ROOT, "include", "movierec_b200_diag.h")).read()
    diag_declared = set(re.findall(r"\b(mr_[a-z_0-9]+)\s*\(", diag_header))
    assert diag_declared == set(_diag.SIGNATURES), diag_declared ^ set(_diag.SIGNATURES)
    dlib = ctypes.CDLL(_diag.LIB_PATH)
    for name in diag_declared:
        assert hasattr(dlib, name), name
        assert name == "mr_diag_last_error" or not hasattr(lib, name), name


def test_struct_layouts_match_header():
    # sizes follow from the header's field lists (8-byte pointers, natural alignment)
    assert ctypes.sizeof(nat.MrModel) == 5 * 8 + 8 * 8 * 2 + 2 * 8 + 8 + 3 * 4 + 8 * 4 + 4 + 8 * 4 + 3 * 4 + 4  # (+ tail padding)
    assert ctypes.sizeof(nat.MrOptState) == 2 * 4 + 4 * 4 + 8 + 10 * 8
    assert ctypes.sizeof(nat.MrGrads) == 7 * 8
    assert nat.MrModel.dense_count.offset == 5 * 8 + 16 * 8 + 2 * 8


def test_workspace_queries_are_host_only():
    m = nat.MrModel()
    m.n_layers, m.mf_dim = 3, 64
    for i, w in enumerate([256, 128, 64]):
        m.L[i] = w
    m.dense_count = 256 * 128 + 128 + 128 * 64 + 64 + 128 + 1
    small = nat.lib.mr_train_workspace_bytes(ctypes.byref(m), 1000)
    big = nat.lib.mr_train_workspace_bytes(ctypes.byref(m), 100000)
    assert 0 < small < big
    assert big - small >= 99000 * 4 * (192 + 192)  # the staged row gradients dominate
    assert nat.lib.mr_sort_workspace_bytes(1 << 20) >= 2 * 4 * (1 << 20)
    assert nat.lib.mr_rank_eval_workspace_bytes(ctypes.byref(m), 1000, 100) >= 1000 * 100 * 4


def test_compute_without_cuda_fails_loudly(tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        model.MovierecModel(copy.deepcopy(TEST_PARAMS), output_dir=str(tmp_path))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        model.RankLayer(2, 3, "rank").call(np.array([0.9, 0.8, 0.7, 0.6]))


# ---- MovierecModel parameter contract (reference test/test_model.py:31-60) ------------------------

def test_wrong_layers():
    params = copy.deepcopy(TEST_PARAMS)
    params["layers_sizes"].append(2)
    with pytest.raises(ValueError, match="must be equal"):
        model.MovierecModel(params)


def test_missing_param():
    for key in ("num_users", "num_items", "layers_sizes", "layers_l2reg", "optimizer", "lr", "batch_size",
                "num_negs_per_pos", "batch_size_eval", "num_negs_per_pos_eval"):
        params = copy.deepcopy(TEST_PARAMS)
        del params[key]
        with pytest.raises(KeyError):
            model.MovierecModel(params)


def test_not_implemented_optimizer():
    params = copy.deepcopy(TEST_PARAMS)
    params["optimizer"] = "other"
    with pytest.raises(NotImplementedError):
        model.MovierecModel(params)


@pytest.mark.parametrize("patch,msg", [
    ({"num_negs_per_pos": 0}, "num_negs_per_pos must be > 0"),
    ({"batch_size": 9}, "Batch size must be divisible"),
    ({"num_negs_per_pos_eval": -1}, "num_negs_per_pos_eval must be > 0"),
    ({"batch_size_eval": 11}, r"Batch size \(eval\) must be divisible"),
    ({"k": 5}, "'k' must be lower"),
])
def test_value_errors(patch, msg):
    params = copy.deepcopy(TEST_PARAMS)
    params.update(patch)
    with pytest.raises(ValueError, match=msg):
        model.MovierecModel(params)


def test_module_constants():
    assert model.OPTIMIZERS == ["adam", "sgd"] and model.HIT_RATE == "hr" and model.DCG == "dcg"
    assert model.OUTPUT_PRED == "output" and model.OUTPUT_RANK == "rank" and model.METRIC_VAL_DCG == "val_output_dcg"
    assert model.MovierecModel.get_model_weights_path("d", "m") == os.path.join("d", "m_weights.h5")
    assert model.MovierecModel.get_params_json_path("d", "m") == os.path.join("d", "m_params.json")
    assert trainer.DEFAULT_PARAMS["layers_sizes"] == [64, 32, 16, 8] and trainer.DEFAULT_PARAMS["k"] == 5
    assert trainer.DEFAULT_PARAMS["num_negs_per_pos"] == 9 and trainer.DEFAULT_PARAMS["batch_size_eval"] == 200
    assert ml.NUM_USERS == {"ml-100k": 943, "ml-1m": 6040, "ml-20m": 138493}
    assert ml.NUM_ITEMS == {"ml-100k": 1682, "ml-1m": 3952, "ml-20m": 27278}


def test_callbacks_follow_keras_semantics():
    class Stub(object):
        def __init__(self):
            self.w, self.stop_training, self.saved = [np.zeros(1)], False, []

        def get_weights(self):
            return [x.copy() for x in self.w]

        def set_weights(self, w):
            self.w = [x.copy() for x in w]

        def save_weights(self, path):
            self.saved.append(path)

    stub = Stub()
    es = model.EarlyStopping(patience=5)
    ck = model.ModelCheckpoint("/tmp/m-checkpoint-{epoch:02d}-{val_loss:.2f}.h5")
    for cb in (es, ck):
        cb.set_model(stub)
        cb.on_train_begin()
    values = [0.1, 0.3, 0.2, 0.2, 0.2, 0.2, 0.2, 0.9]
    ran = 0
    for epoch, v in enumerate(values):
        stub.w = [np.array([float(epoch)])]
        for cb in (es, ck):
            cb.on_epoch_end(epoch, {"val_output_dcg": v, "val_loss": 0.5})
        ran += 1
        if stub.stop_training:
            break
    from oracle import movierec_oracle as o
    assert (ran, 1, True) == o.early_stopping_trace(values, 5)
    assert stub.w[0][0] == 1.0  # best epoch's weights restored
    assert stub.saved == ["/tmp/m-checkpoint-01-0.50.h5", "/tmp/m-checkpoint-02-0.50.h5"]


# ---- data pipeline (reference test/test_data_pipeline.py) -----------------------------------------

def test_wrong_database_name_load():
    with pytest.raises(ValueError, match="Invalid dataset name"):
        data_pipeline.load_ratings_train_test_sets("wrong db", "/tmp/")


def test_load_ratings_train_test_sets(ref, monkeypatch):
    v = ref["split"]
    df = pd.DataFrame({"userId": v["userId"], "itemId": v["itemId"], "rating": v["rating"]})
    monkeypatch.setattr(data_pipeline, "load_ratings_data", lambda *a, **k: df)
    train, validation, test = data_pipeline.load_ratings_train_test_sets("ml-100k", "ml-100k", download=False)
    for got, name in ((train, "train"), (validation, "validation"), (test, "test")):
        pd.testing.assert_frame_equal(got, pd.DataFrame(v[name]), check_dtype=False)


def test_split_handles_interleaved_users():
    df = pd.DataFrame({"userId": [1, 0, 1, 0, 1, 0, 2, 2, 2], "itemId": [10, 20, 11, 21, 12, 22, 30, 31, 32],
                       "rating": np.arange(9, dtype=np.float32)})
    train, validation, test = data_pipeline.split_leave_last_two_out(df)
    assert test.itemId.tolist() == [22, 12, 32] and validation.itemId.tolist() == [21, 11, 31]
    assert train.itemId.tolist() == [20, 10, 30] and train.index.tolist() == [0, 1, 2]
    from oracle import movierec_oracle as o
    tr, va, te = o.leave_last_two_out(df.userId.values)
    assert df.itemId.values[tr].tolist() == train.itemId.tolist()
    assert df.itemId.values[va].tolist() == validation.itemId.tolist()
    assert df.itemId.values[te].tolist() == test.itemId.tolist()


def test_generator_value_errors(ref):
    data = pd.DataFrame(ref["generator_duplicated_user"]["data"])
    msgs = ref["generator_value_errors"]["messages"]
    with pytest.raises(ValueError, match=msgs[0]):
        data_pipeline.MovieLensDataGenerator("wrong_name", data, batch_size=6, negatives_per_positive=2)
    with pytest.raises(ValueError, match=msgs[1]):
        data_pipeline.MovieLensDataGenerator("ml-100k", data, batch_size=6, negatives_per_positive=0)
    with pytest.raises(ValueError, match=msgs[2]):
        data_pipeline.MovieLensDataGenerator("ml-100k", data, batch_size=10, negatives_per_positive=6)


def test_generator_len_and_shuffle_follow_reference(golden_dir):
    g = np.load(os.path.join(golden_dir, "generator_batches.npz"))
    df = pd.DataFrame({"userId": g["data_users"], "itemId": g["data_items"]})
    np.random.seed(int(g["seed"]))
    gen = data_pipeline.MovieLensDataGenerator("ml-100k", df, int(g["noextra_bs"]), int(g["noextra_negs"]), shuffle=True)
    np.testing.assert_array_equal(gen.indexes, g["noextra_indexes"])  # same np.random.shuffle call as the reference
    assert len(gen) == int(g["noextra_len"])
    assert gen.num_users == 943 and gen.num_items == 1682 and gen.dataset_name == "ml-100k"
    assert gen.num_positives_per_batch == 4 and gen.num_negatives_per_batch == 16


def test_user_csr_matches_oracle():
    from oracle import movierec_oracle as o
    rng = np.random.default_rng(0)
    users, items = rng.integers(0, 20, 300), rng.integers(0, 50, 300)
    rowptr, csr = data_pipeline.build_user_csr(users, items)
    rp, it = o.build_csr(int(users.max()) + 1, users, items)
    np.testing.assert_array_equal(rowptr, rp)
    np.testing.assert_array_equal(csr, it)


def test_load_ratings_data_zero_based(tmp_path):
    d = tmp_path / "ml-100k"
    d.mkdir()
    (d / "u.data").write_text("1\t1\t5\t881250949\n2\t3\t3\t891717742\n")
    df = ml.load_ratings_data(str(tmp_path), "ml-100k")
    assert df.userId.tolist() == [0, 1] and df.itemId.tolist() == [0, 2] and df.rating.tolist() == [5.0, 3.0]
    with pytest.raises(FileNotFoundError):
        ml.load_ratings_data(str(tmp_path), "ml-1m", download=False)


def test_remap_dense_ids_host_path():
    df = pd.DataFrame({"userId": [10, 3, 10, 7, 3], "itemId": [100, 5, 5, 42, 100], "rating": [1.0, 2.0, 3.0, 4.0, 5.0]})
    out, maps = data_pipeline.remap_dense_ids(df, on_device=False)
    assert out.userId.tolist() == [2, 0, 2, 1, 0] and out.itemId.tolist() == [2, 0, 0, 1, 2]
    assert maps["userId"].tolist() == [3, 7, 10] and maps["itemId"].tolist() == [5, 42, 100]
    assert out.rating.tolist() == df.rating.tolist() and df.userId.tolist() == [10, 3, 10, 7, 3]  # input untouched
    assert (maps["userId"][out.userId.values] == df.userId.values).all()


def test_keras_h5_round_trip(tmp_path):
    """Keras-layout HDF5 weight files (SURVEY 8 f4); needs h5py, which this image does not ship."""
    pytest.importorskip("h5py")
    from movierec.util import keras_h5
    from oracle import movierec_oracle as o
    w = o.init_weights(7, 9, [6, 4], mf_dim=2)
    order = o.weight_names([6, 4], 2)
    path = str(tmp_path / "m_weights.h5")
    keras_h5.write(path, w, order, {"iterations": np.array(3), "m/dense": np.arange(5.0)})
    assert keras_h5.is_hdf5(path)
    got, opt = keras_h5.read(path)
    assert set(got) == set(order)
    for k in order:
        np.testing.assert_array_equal(got[k], w[k])
    assert int(opt["iterations"]) == 3 and opt["m/dense"].tolist() == list(np.arange(5.0))


def test_keras_h5_detection_and_missing_h5py(tmp_path):
    from movierec.util import keras_h5
    p = tmp_path / "x.h5"
    p.write_bytes(b"PK\x03\x04 not hdf5")
    assert not keras_h5.is_hdf5(str(p))
    p.write_bytes(keras_h5.HDF5_MAGIC + b"\0" * 64)
    assert keras_h5.is_hdf5(str(p))
    if not keras_h5.have_h5py():
        with pytest.raises(ImportError, match="h5py is not installed"):
            keras_h5.read(str(p))


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` runs on host cores alone (no GPU, no CUDA library call) and prints ONE JSON line with
    the keys the driver reads: impl, the metric of BASELINE.json, the same config dict as the GPU arm, e2e with zero
    copy bytes, and a cpu_baseline that says which implementation was timed."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    line = json.loads(lines[0])
    with open(os.path.join(root, "BASELINE.json")) as f:
        base = json.load(f)
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["n_gpus"] == 1
    assert line["unit"] == "samples/s" and line["value"] > 0 and line["steps"] == 1
    assert line["metric"] and (line["metric"] in json.dumps(base) or "samples" in line["metric"])
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["cpu_baseline"]["kind"] in ("port", "reference") and line["cpu_baseline"]["cores"] >= 1
    assert "ml-20m" in line["config"]["workload"] and line["config"]["baseline_config"] == "BASELINE.json configs[2]"


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: float arrays only, ids exact, tall tables sampled on rows shared by the tables of one
    side and the same in every run, the size limit enforced."""
    import torch
    import bench
    rng = np.random.default_rng(0)
    n = bench.DUMP_TABLE_ROWS + 5
    w = {"user_embedding/embeddings": rng.random((n, 4), dtype=np.float32),
         "gmf_user_embedding/embeddings": rng.random((n, 2), dtype=np.float32),
         "hidden_1/kernel": rng.random((8, 4), dtype=np.float32)}
    batch = (torch.tensor([3, 3, 7], dtype=torch.int32), torch.tensor([1, 2, 2 ** 24 + 1], dtype=torch.int32),
             torch.tensor([0.0, 0.0, 1.0]))
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), np.arange(8, dtype=np.float32), batch, w)
    names = sorted(os.listdir(str(tmp_path / "a")))
    assert names == sorted(os.listdir(str(tmp_path / "b")))
    got = {f[:-4]: np.load(str(tmp_path / "a" / f)) for f in names}
    for f in names:
        assert got[f[:-4]].dtype in (np.float32, np.float64), f
        np.testing.assert_array_equal(got[f[:-4]], np.load(str(tmp_path / "b" / f)))
    assert got["batch_items"].tolist() == [1, 2, 2 ** 24 + 1] and got["step_out"].tolist() == list(range(8))
    rows = got["weights.user_embedding.embeddings.rows"]
    np.testing.assert_array_equal(rows, got["weights.gmf_user_embedding.embeddings.rows"])
    assert len(np.unique(rows)) == bench.DUMP_TABLE_ROWS
    np.testing.assert_array_equal(got["weights.user_embedding.embeddings"], w["user_embedding/embeddings"][rows.astype(int)])
    np.testing.assert_array_equal(got["weights.hidden_1.kernel"], w["hidden_1/kernel"])
    assert "weights.hidden_1.kernel.rows" not in got
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 1000)
    with pytest.raises(SystemExit, match="limit"):
        bench.dump_outputs(str(tmp_path / "c"), np.zeros(8), batch, w)
    assert not (tmp_path / "c").exists()
