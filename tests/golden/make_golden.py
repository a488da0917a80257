"""Generate golden vectors by executing the REFERENCE's own Python source for the rank layer,
ranking metrics and batch generator.

Needs a checkout of the reference (carlamb/MovieRecommender-TF-TRT) and pandas; no GPU:

    python tests/golden/make_golden.py <reference checkout>

TensorFlow is not installed, so the reference's `movierec/model.py` and `data_pipeline.py` are
imported with a NumPy stand-in for the dozen `tf.python.keras.backend` calls they make
(model.py:345-351, 414-454).  Everything else that runs -- reshape/argmax/where/equal/less logic
of `_get_hits_per_user`, the DCG formula, the generator's batch layout and sampling calls -- is
the reference's own code.  The stand-in fixes one TF semantic that cannot be re-verified here:
`nn.top_k(sorted=True)` returns the lower index first among equal values (documented TF
behaviour, pinned by the reference's test/test_model.py:168-190, which these stand-ins pass).
pandas 3 removed `Series.append` (data_pipeline.py:105); it is restored as `pd.concat`.

Outputs (committed): rank_metrics.npz, generator_batches.npz.
"""

import importlib.util
import os
import sys
import types

import numpy as np
import pandas as pd

HERE = os.path.dirname(os.path.abspath(__file__))


class _NumpyBackend(object):
    """NumPy stand-in for tensorflow.python.keras.backend, limited to what the reference calls."""

    learning_phase = 0

    class ops(object):
        convert_to_tensor = staticmethod(np.asarray)

    class nn(object):
        @staticmethod
        def top_k(x, k, sorted=True):
            idx = np.argsort(-np.asarray(x), axis=-1, kind="stable")[..., :k]
            return np.take_along_axis(np.asarray(x), idx, axis=-1), idx.astype(np.int32)

    class math_ops(object):
        log = staticmethod(lambda x: np.log(np.asarray(x, dtype=np.float32)))

        @staticmethod
        def argmax(x, axis=-1, output_type="int64"):
            return np.argmax(x, axis=axis).astype(output_type)

    class array_ops(object):
        where = staticmethod(lambda c: np.argwhere(c))

    @classmethod
    def in_train_phase(cls, a, b):
        return a if cls.learning_phase else b

    @classmethod
    def set_learning_phase(cls, v):
        cls.learning_phase = v

    reshape = staticmethod(lambda x, s: np.reshape(x, s))
    shape = staticmethod(lambda x: np.shape(x))
    equal = staticmethod(lambda a, b: np.equal(a, b))
    less = staticmethod(lambda a, b: np.less(a, b))
    cast = staticmethod(lambda x, d: np.asarray(x).astype(d))
    mean = staticmethod(lambda x, axis=None: np.mean(x, axis=axis))


def _install_fake_tf():
    class Layer(object):
        def __init__(self, name=None, **kwargs):
            self.name = name

    class Sequence(object):
        pass

    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    stub = lambda *a, **k: None
    mod("tensorflow")
    mod("tensorflow.python")
    keras = mod("tensorflow.python.keras", backend=_NumpyBackend)
    mod("tensorflow.python.keras.backend")
    sys.modules["tensorflow.python.keras.backend"] = _NumpyBackend
    mod("tensorflow.python.keras.callbacks", EarlyStopping=stub, ModelCheckpoint=stub)
    mod("tensorflow.python.keras.layers", concatenate=stub, Dense=stub, Embedding=stub, Input=stub,
        Flatten=stub, Layer=Layer)
    mod("tensorflow.python.keras.models", Model=stub)
    mod("tensorflow.python.keras.optimizers", Adam=stub, SGD=stub)
    mod("tensorflow.python.keras.regularizers", l2=stub)
    mod("tensorflow.python.keras.utils", Sequence=Sequence)
    return keras


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    sys.modules[name] = m
    spec.loader.exec_module(m)
    return m


def main(ref_root):
    _install_fake_tf()
    ref = os.path.abspath(ref_root)
    sys.path.insert(0, os.path.join(ref, "movierec"))  # the reference imports `util.*` top-level
    ref_model = _load("ref_model", os.path.join(ref, "movierec", "model.py"))
    if not hasattr(pd.Series, "append"):
        pd.Series.append = lambda self, other: pd.concat([self, other])
    ref_dp = _load("ref_data_pipeline", os.path.join(ref, "movierec", "data_pipeline.py"))
    K = _NumpyBackend

    # -- the stand-in must itself pass the reference's rank-layer test (test_model.py:168-190)
    layer = ref_model.RankLayer(num_negs_per_pos_train=2, num_negs_per_pos_eval=3, name="rank")
    K.set_learning_phase(1)
    assert np.array_equal(layer.call(np.array([0.9, 0.8, 0.7, 0.7, 0.8, 0.9])), [[0, 1, 2], [2, 1, 0]])
    K.set_learning_phase(0)
    assert np.array_equal(layer.call(np.array([0.9, 0.8, 0.7, 0.6, 0.5, 0.9, 0.9, 0.9])),
                          [[0, 1, 2, 3], [1, 2, 3, 0]])

    # -- rank + metrics on seeded scores, with heavy ties and saturated values mixed in
    rng = np.random.default_rng(20261018)
    out = {}
    case = 0
    for group in (2, 3, 5, 10, 33, 100, 128):
        for quant in (0, 4, 1):  # 0: continuous scores, 4: 4 distinct levels, 1: all equal
            G = 64 if group < 100 else 16
            s = rng.random((G, group), dtype=np.float32)
            if quant == 4:
                s = np.floor(s * 4).astype(np.float32) / 4
            elif quant == 1:
                s = np.full((G, group), 0.5, np.float32)
            y = np.zeros((G, group), np.int64)
            y[:, -1] = 1  # generator layout: the positive is last (data_pipeline.py:113,148)
            lay = ref_model.RankLayer(group - 1, group - 1, name="rank")
            rank = lay.call(s.reshape(-1))
            ks = sorted({1, 2, min(5, group), min(10, group), group})
            hr = [float(ref_model.hit_rate(y, None, k=k, pred_rank_idx=rank)) for k in ks]
            dcg = [float(ref_model.discounted_cumulative_gain(y, None, k, rank)) for k in ks]
            _, pos = ref_model._get_hits_per_user(y, rank, group)
            pre = "c{}_".format(case)
            out[pre + "scores"], out[pre + "rank"] = s, np.asarray(rank, np.int32)
            out[pre + "ks"], out[pre + "hr"], out[pre + "dcg"] = np.array(ks), np.array(hr), np.array(dcg)
            out[pre + "pos"] = np.asarray(pos, np.int32)
            case += 1
    out["num_cases"] = np.array(case)
    np.savez_compressed(os.path.join(HERE, "rank_metrics.npz"), **out)

    # -- generator batches from the reference's own __getitem__, global NumPy RNG seeded
    rng = np.random.default_rng(7)
    num_users, num_items, per_user = 12, 40, 9
    users = np.repeat(np.arange(num_users), per_user)
    items = np.concatenate([rng.choice(num_items, per_user, replace=False) for _ in range(num_users)])
    df = pd.DataFrame({"userId": users.astype(np.int32), "itemId": items.astype(np.int32),
                       "rating": np.ones(len(users), np.float32)})
    # hold out 2 per user as "extra" the way trainer.py:63-69 passes train_df to the val generator
    is_extra = np.zeros(len(df), bool)
    is_extra[per_user - 2::per_user] = True
    data_df = df[~is_extra].reset_index(drop=True)
    extra_df = df[is_extra].reset_index(drop=True)
    gen_out = {"data_users": data_df.userId.values, "data_items": data_df.itemId.values,
               "extra_users": extra_df.userId.values, "extra_items": extra_df.itemId.values,
               "num_items": np.array(1682), "seed": np.array(1234)}
    for tag, extra, negs, bs in (("noextra", None, 4, 20), ("extra", extra_df, 9, 30)):
        np.random.seed(1234)
        gen = ref_dp.MovieLensDataGenerator("ml-100k", data_df, bs, negs, extra_data_df=extra, shuffle=True)
        gen_out[tag + "_indexes"] = gen.indexes.copy()
        gen_out[tag + "_len"] = np.array(len(gen))
        gen_out[tag + "_negs"], gen_out[tag + "_bs"] = np.array(negs), np.array(bs)
        for b in range(3):
            (xu, xi), y = gen[b]
            gen_out["{}_b{}_users".format(tag, b)] = np.asarray(xu)
            gen_out["{}_b{}_items".format(tag, b)] = np.asarray(xi)
            gen_out["{}_b{}_y".format(tag, b)] = np.asarray(y)
    np.savez_compressed(os.path.join(HERE, "generator_batches.npz"), **gen_out)
    print("wrote rank_metrics.npz ({} cases) and generator_batches.npz".format(case))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit("usage: python tests/golden/make_golden.py <reference checkout>")
    main(sys.argv[1])
