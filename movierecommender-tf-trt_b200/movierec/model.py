"""Recommender model: the `movierec.model` surface of carlamb/MovieRecommender-TF-TRT
(reference movierec/model.py) on top of the B200 kernels.

Same constructor contract, parameter dict, exceptions, method names and constants as the
reference; the Keras graph (model.py:135-215) is replaced by `_engine.NeuMFEngine`, which owns
the device tensors and calls libmovierec_b200.so.  Optional new parameters keep the reference
behaviour by default: `mf_dim` (0 = the reference's MLP-only model), `adam_mode` ("dense" =
legacy-Keras Adam over every table row, "sparse" = touched rows only), `seed`.
Deviations, each deliberate: weights are saved under the reference's `.h5` file names in the Keras
HDF5 layout when h5py is installed (util/keras_h5.py) and as NumPy `.npz` payloads under the same
names otherwise (this image has no h5py; `load_weights` tells the two apart by the file signature),
and `load_from_files` passes name and directory in the declared order (the reference swaps them,
model.py:301).
"""

import json
import logging
import os
import random

import numpy as np

DEFAULT_PARAMS = {  # the reference's toy defaults (model.py:15-34)
    "num_users": 5,
    "num_items": 10,
    "layers_sizes": [5, 4],
    "layers_l2reg": [0.01, 0.01],
    "optimizer": "adam",
    "lr": 0.001,
    "beta_1": 0.9,
    "beta_2": 0.999,
    "batch_size": 6,
    "num_negs_per_pos": 2,
    "batch_size_eval": 12,
    "num_negs_per_pos_eval": 5,
    "k": 3,
}

ADAM_NAME = "adam"
SGD_NAME = "sgd"
OPTIMIZERS = [ADAM_NAME, SGD_NAME]

HIT_RATE = "hr"
DCG = "dcg"

OUTPUT_PRED = "output"
OUTPUT_RANK = "rank"

METRIC_VAL_DCG = "val_{}_{}".format(OUTPUT_PRED, DCG)

EARLY_STOPPING_PATIENCE = 5  # model.py:324

# Fold-in defaults (MovierecModel.fold_in), from the planted-cluster grid of tools/fold_in_bench.py --quality
# (profiles/r06_fold_in_quality.json, Adam, 4 negatives): recall@10 of the folded-in users is flat at 0.28-0.30 for lr
# 0.03-0.3 at 5-100 steps, and the mean loss still falls up to about 30 steps; lr 0.01 needs >= 20 steps, and the
# training lr 0.001 reaches the plateau only at 100 steps (0.04 at 30).  30 steps at 0.05 sits inside the plateau on
# both axes.
FOLD_IN_STEPS = 30
FOLD_IN_LR = 0.05


def _engine_module():
    # imported lazily so that parameter validation (pure host logic) works without a GPU;
    # anything that computes goes through the CUDA library and fails loudly without it
    from . import _engine
    return _engine


class History(object):
    """What Keras' fit_generator returns: `.history` maps metric name -> list of epoch values."""

    def __init__(self):
        self.history = {}
        self.epoch = []

    def _append(self, epoch, logs):
        self.epoch.append(epoch)
        for k, v in logs.items():
            self.history.setdefault(k, []).append(v)


class NeuMFModel(object):
    """Stands where the Keras `Model` stood (`MovierecModel.model`): batch-level entry points with
    Keras' names, backed by the CUDA engine."""

    def __init__(self, owner, engine):
        self._owner = owner
        self.engine = engine
        self.name = owner.name
        self.stop_training = False
        self.output_names = [OUTPUT_PRED, OUTPUT_RANK]
        self.metrics_names = ["loss", OUTPUT_PRED + "_loss", OUTPUT_PRED + "_" + HIT_RATE, OUTPUT_PRED + "_" + DCG]

    # ---- weights ---------------------------------------------------------------------------------
    @property
    def weight_names(self):
        return self.engine.weight_names()

    def get_weights(self):
        w = self.engine.get_weights()
        return [w[k] for k in self.engine.weight_names()]

    def set_weights(self, weights):
        self.engine.set_weights(weights)

    def save_weights(self, path):
        """Keras-layout HDF5 when h5py is installed (the reference's format, model.py:245), else an .npz payload
        under the same file name."""
        from .util import keras_h5
        if keras_h5.have_h5py():
            keras_h5.write(path, self.engine.get_weights(), self.engine.weight_names(),
                           self.engine.get_optimizer_state())
            return
        arrays = dict(self.engine.get_weights())
        arrays.update({"optimizer/" + k: np.asarray(v) for k, v in self.engine.get_optimizer_state().items()})
        with open(path, "wb") as f:  # keep the caller's file name (np.savez would append .npz)
            np.savez(f, **arrays)

    def load_weights(self, path):
        from .util import keras_h5
        if keras_h5.is_hdf5(path):  # written by Keras (the reference) or by save_weights above
            weights, opt = keras_h5.read(path)
            missing = [k for k in self.engine.weight_names() if k not in weights]
            if missing:
                raise ValueError("weight file {} lacks {}".format(path, ", ".join(missing)))
            self.engine.set_weights({k: weights[k] for k in self.engine.weight_names()})
            if opt:
                self.engine.set_optimizer_state(opt)
            return
        with np.load(path) as z:
            self.engine.set_weights({k: z[k] for k in self.engine.weight_names()})
            opt = {k[len("optimizer/"):]: z[k] for k in z.files if k.startswith("optimizer/")}
        if opt:
            self.engine.set_optimizer_state(opt)

    def summary(self, print_fn=print):
        e = self.engine
        print_fn("Model: {}".format(self.name))
        total = 0
        for k in e.weight_names():
            shape = tuple(e._view(k).shape)
            total += int(np.prod(shape))
            print_fn("  {:<36s} {}".format(k, shape))
        print_fn("Total params: {}".format(total))

    # ---- batch entry points ------------------------------------------------------------------------
    def predict_on_batch(self, x):
        """[x_users, x_items] -> [output (B,1) float32, rank (G, negs_eval+1) int32]
        (reference test/test_model.py:161-166; the rank layer is in eval phase, model.py:347)."""
        x_users, x_items = x
        o = self._owner
        group = o._num_negs_per_pos_eval + 1
        _, probs, _ = self.engine.forward(x_users, x_items, want_logits=False)
        if probs.numel() % group:
            raise ValueError("batch of {} rows is not divisible by (num_negs_per_pos_eval + 1) = {}".format(
                probs.numel(), group))
        rank, _, _ = _engine_module().rank_scores(probs, group, o._k, want_rank=True, device=self.engine.device)
        out = probs.cpu().numpy().reshape(-1, 1)
        self._raise_on_bad_ids(bool(np.isnan(out).any()))  # the kernels mark rows with an out-of-range id with NaN
        return [out, rank.cpu().numpy()]

    def recommend(self, user_id, candidate_items, top_k=10):
        """Serving-shaped scoring (reference client, trt_client.py:47-57: one user, N candidate items, the K best):
        returns (items (K,), scores (K,)) ordered as the RankLayer orders them (descending score, the earlier
        candidate first among ties).  One forward of N rows that share the user (the user row is read once per
        launch tile) and one rank pass, both on the device."""
        items = np.asarray(candidate_items, dtype=np.int32).reshape(-1)
        n = int(items.size)
        if n == 0:
            return items, np.zeros(0, np.float32)
        eng = self.engine
        _, probs, _ = eng.forward(np.asarray([user_id], dtype=np.int32), items, user_div=n, want_logits=False)
        rank, _, _ = _engine_module().rank_scores(probs, n, min(int(top_k), n), want_rank=True, device=eng.device)
        order = rank.cpu().numpy().reshape(-1)[:min(int(top_k), n)]
        p = probs.cpu().numpy()
        return items[order], p[order]

    def recommend_for_users(self, users, top_k=10, exclude=None):
        """The top_k best items of the WHOLE catalogue for each of `users` (RankLayer order: descending score, the
        lower item id first among ties), leaving out each user's exclusion list.  exclude: None, a
        MovieLensDataGenerator (the items its sampler never draws for the user: data ∪ extra_data) or a
        (rowptr, items) pair of ascending per-user lists.  Returns NumPy (items (U, top_k) int32, scores (U, top_k)
        float32); slots beyond the number of candidates hold -1 / NaN.  One device call for all users."""
        eng = self.engine
        items, scores, _, _, _ = eng.catalogue_topk(users, top_k, exclude=_exclusion_lists(exclude))
        self._raise_on_bad_ids(float(eng.last_catalogue_bad.item()))
        return items.cpu().numpy(), scores.cpu().numpy()

    def recommend_batch(self, users, candidate_lists, top_k=10):
        """recommend() for many requests at once: user users[u] against its own candidate list, of any length.
        candidate_lists: a list (or other sequence) of 1-D item arrays, one per user, or a tuple (rowptr, items) of
        CSR offsets (U + 1) and concatenated items.  Returns NumPy (items (U, top_k) int32, scores (U, top_k) float32)
        in the RankLayer order (descending score, the earlier candidate first among ties); slots beyond a list's
        length hold -1 / NaN.  Raises IndexError on an out-of-range user or item.  Host offsets are cut into device
        calls of whole lists of at most 2^22 candidates (a longer list is a call of its own)."""
        users = np.asarray(users, dtype=np.int32).reshape(-1)
        rowptr, items = _candidate_csr(candidate_lists, users.size)
        eng = self.engine
        self._raise_on_bad_ids(_ids_outside(users, eng.num_users) or _ids_outside(items, eng.num_items))
        k = int(top_k)
        out_items = np.full((users.size, k), -1, np.int32)
        out_scores = np.full((users.size, k), np.nan, np.float32)
        for lo, hi in _list_chunks(rowptr):
            r0, r1 = int(rowptr[lo]), int(rowptr[hi])
            top, sc, _, _, _, _ = eng.rank_lists(users[lo:hi], (rowptr[lo:hi + 1] - r0, items[r0:r1]), k)
            out_items[lo:hi] = top.cpu().numpy()
            out_scores[lo:hi] = sc.cpu().numpy()
        return out_items, out_scores

    def recommend_for_histories(self, histories, top_k=10, **fold_in_args):
        """Top-k for users the model has not seen, from their rating histories alone: one fold-in of every history
        (MovierecModel.fold_in, whose keyword arguments fold_in_args takes) and one full-catalogue top-k call on the
        folded rows, with each history as that user's exclusion list.  histories as MovierecModel.fold_in.  Returns
        NumPy (items (U, top_k) int32, scores (U, top_k) float32) like recommend_for_users."""
        eng = self.engine
        rowptr, items = _engine_module().fold_in_histories(histories, eng.num_items)
        view = self._owner.fold_in((rowptr, items), **fold_in_args)
        return view.model.recommend_for_users(np.arange(rowptr.size - 1, dtype=np.int32), top_k,
                                              exclude=(rowptr, items))

    def _step_logs(self, out, rows, group):
        loss = out[0] / rows + out[3]
        return {"loss": loss, OUTPUT_PRED + "_loss": out[0] / rows,
                OUTPUT_PRED + "_" + HIT_RATE: out[1] / (rows // group), OUTPUT_PRED + "_" + DCG: out[2] / (rows // group)}

    def train_on_batch(self, x, y, prefetch=None):
        """One optimisation step; returns [loss, output_loss, output_hr, output_dcg] like Keras.

        prefetch=([x_users, x_items], y) (optional, not in Keras): the NEXT batch.  Its host-to-device copies are
        issued on a copy stream before this step's loss is read back, so they run under this step; the next call
        finds them by the identity of the host arrays and skips its own upload.  Pinned host tensors make the
        copies asynchronous."""
        x_users, x_items = x
        o = self._owner
        group = o._num_negs_per_pos + 1
        # the reference accepts any users per row; the once-per-group fast path is taken only when the batch
        # really has the generator's layout (checked on the device before the step: one tiny kernel)
        eng = self.engine
        mod = _engine_module()
        rows = int(np.asarray(y).size if not hasattr(y, "numel") else y.numel())
        staged = getattr(self, "_prefetched", None)
        if staged is not None and staged[0] == (id(x_users), id(x_items), id(y)):
            _, d_users, d_items, d_y, ready = staged
            import torch
            torch.cuda.current_stream(eng.device).wait_event(ready)
        else:
            d_users = mod.as_device_i32(x_users, eng.device)
            d_items, d_y = x_items, y
        self._prefetched = None
        grouped = eng.users_grouped(d_users, group)
        out_dev = eng.train_step(d_users, d_items, d_y, group=group, k=o._k, grouped=grouped)
        if prefetch is not None:
            import torch
            (n_users, n_items), n_y = prefetch
            if getattr(self, "_copy_stream", None) is None:
                self._copy_stream = torch.cuda.Stream(device=eng.device)
            with torch.cuda.stream(self._copy_stream):
                staged = (mod.as_device_i32(n_users, eng.device), mod.as_device_i32(n_items, eng.device),
                          mod.as_device_f32(n_y, eng.device))
                ready = torch.cuda.Event()
                ready.record(self._copy_stream)
            self._prefetched = ((id(n_users), id(n_items), id(n_y)),) + staged + (ready,)
        out = out_dev.cpu().numpy().astype(np.float64)
        if int(out[4]) & 1:
            raise IndexError("user/item id out of range in batch (num_users={}, num_items={})".format(
                o._num_users, o._num_items))
        logs = self._step_logs(out, rows, group)
        return [logs[n] for n in self.metrics_names]

    def test_on_batch(self, x, y):
        """Loss and ranking metrics of one validation batch (eval phase: groups of negs_eval+1)."""
        sums, rows = self._eval_batch_sums(x, y)
        o = self._owner
        out = sums.cpu().numpy().astype(np.float64)
        self._raise_on_bad_ids(out[3])
        group = o._num_negs_per_pos_eval + 1
        logs = self._step_logs([out[0], out[1], out[2], 0.0], rows, group)
        return [logs[n] for n in self.metrics_names]

    def _eval_batch_sums(self, x, y):
        import torch
        x_users, x_items = x
        o = self._owner
        eng = self.engine
        group = o._num_negs_per_pos_eval + 1
        _, probs, loss = eng.forward(x_users, x_items, labels=y, want_logits=False)
        rows = probs.numel()
        # the label column is the argmax of y_true per group (model.py:447-448), wherever the batch puts its positive
        _, _, sums = _engine_module().rank_scores(probs, group, o._k, want_rank=False, device=eng.device, labels=y)
        # an out-of-range id makes its row's probability NaN (and is left out of the loss): reported with the sums so
        # that callers raise instead of returning metrics of a partly invalid batch
        bad = torch.isnan(probs).any().to(loss.dtype).reshape(1)
        return torch.cat([loss, sums, bad]), rows

    def evaluate_generator(self, generator, steps=None):
        """Keras `evaluate_generator`: batch-size-weighted mean of the per-batch values over
        `len(generator)` batches (SURVEY 3.4)."""
        import torch
        steps = len(generator) if steps is None else steps
        o = self._owner
        group = o._num_negs_per_pos_eval + 1
        acc = torch.zeros(4, dtype=torch.float64, device=self.engine.device)
        rows = 0
        for b in range(steps):
            x, y = _device_batch(generator, b)
            s, r = self._eval_batch_sums(x, y)
            acc += s.double()
            rows += r
        if rows == 0:
            return [float("nan")] * 4
        out = acc.cpu().numpy()
        self._raise_on_bad_ids(out[3])
        logs = self._step_logs([out[0], out[1], out[2], self._l2_penalty()], rows, group)
        return [logs[n] for n in self.metrics_names]

    def _raise_on_bad_ids(self, flag):
        if flag:
            o = self._owner
            raise IndexError("user/item id out of range in an evaluation batch (num_users={}, num_items={})".format(
                o._num_users, o._num_items))

    def _l2_penalty(self):
        o = self._owner
        if not any(o._layers_l2reg):
            return 0.0
        # the regulariser term of the reported loss (model.py:163,168,178); off the hot path and only
        # for non-default l2: computed from a host copy of the weights
        w = self.engine.get_weights()
        tot = 0.0
        for k, v in w.items():
            if k.endswith("embeddings"):
                tot += o._layers_l2reg[0] * float(np.sum(np.square(v, dtype=np.float64)))
            elif k.startswith("hidden_") and k.endswith("kernel"):
                tot += o._layers_l2reg[int(k.split("/")[0].split("_")[1])] * float(np.sum(np.square(v, dtype=np.float64)))
        return tot

    def fit_generator(self, generator, validation_data=None, epochs=1, callbacks=None, verbose=1, shuffle=True):
        """The Keras training loop the reference relies on (model.py:329-333): `epochs` x
        `len(generator)` train_on_batch steps (batch order shuffled per epoch as Keras does for a
        Sequence), validation after every epoch, callbacks, `generator.on_epoch_end()`.
        Step outputs stay on the device and are read back once per epoch."""
        import torch
        o = self._owner
        eng = self.engine
        history = History()
        callbacks = callbacks or []
        for cb in callbacks:
            cb.set_model(self)
            cb.on_train_begin()
        self.stop_training = False
        group = o._num_negs_per_pos + 1
        for epoch in range(epochs):
            steps = len(generator)
            order = list(range(steps))
            if shuffle:
                random.shuffle(order)
            acc = torch.zeros(5, dtype=torch.float64, device=eng.device)
            rows = 0
            for b in order:
                x, y = _device_batch(generator, b)
                out = eng.train_step(x[0], x[1], y, group=group, k=o._k, grouped=_is_grouped(generator, eng, x[0], group))
                acc[:3] += out[:3].double()
                acc[3] += out[3].double() * y.numel()
                acc[4] += out[4].double()
                rows += int(y.numel())
            logs = {}
            if rows:
                a = acc.cpu().numpy()
                if a[4] != 0:  # sum over steps of the per-step flag word (bit 0 bad id, bit 1 group layout broken)
                    raise IndexError("user/item id out of range (or a generator that declares grouped batches "
                                     "produced a group with more than one user) during training")
                logs = self._step_logs([a[0], a[1], a[2], a[3] / rows], rows, group)
            if validation_data is not None:
                vals = self.evaluate_generator(validation_data)
                for n, v in zip(self.metrics_names, vals):
                    logs["val_" + n] = v
            history._append(epoch, logs)
            if verbose:
                logging.info("Epoch %d/%d - %s", epoch + 1, epochs,
                             " - ".join("{}: {:.4f}".format(k, v) for k, v in logs.items()))
            for cb in callbacks:
                cb.on_epoch_end(epoch, logs)
            if hasattr(generator, "on_epoch_end"):
                generator.on_epoch_end()
            if self.stop_training:
                break
        for cb in callbacks:
            cb.on_train_end()
        return history


def _is_grouped(generator, engine, x_users, group):
    """Whether a training batch has one user per group.  Generators of this package say so themselves
    (`grouped_batches`: MovieLensDataGenerator always builds groups of one user, data_pipeline.py:99-150, and
    the device verifies it during the step); batches of any other Sequence are checked on the device first."""
    if getattr(generator, "grouped_batches", False):
        return True
    return engine.users_grouped(x_users, group)


def _device_batch(generator, b):
    """Batch `b` of a generator as device-ready arrays.  Our generator hands out device tensors
    (no host round trip); any other Sequence gives NumPy arrays that the engine uploads."""
    if hasattr(generator, "device_batch"):
        return generator.device_batch(b)
    import torch
    x, y = generator[b]
    return [x[0], x[1]], torch.as_tensor(np.asarray(y, dtype=np.float32))


class EarlyStopping(object):
    """Keras EarlyStopping as the reference configures it (model.py:324-325): monitor a metric to
    maximise, stop after `patience` epochs without improvement, restore the best weights when
    stopping."""

    def __init__(self, monitor=METRIC_VAL_DCG, mode="max", restore_best_weights=True, patience=5, verbose=0):
        if mode != "max":
            raise NotImplementedError("only mode='max' is used by the reference")
        self.monitor, self.patience, self.restore_best_weights, self.verbose = monitor, patience, restore_best_weights, verbose
        self.model = None

    def set_model(self, model):
        self.model = model

    def on_train_begin(self):
        self.wait, self.stopped_epoch, self.best, self.best_weights = 0, 0, -np.inf, None

    def on_epoch_end(self, epoch, logs):
        current = logs.get(self.monitor)
        if current is None:
            return
        if current > self.best:
            self.best, self.wait = current, 0
            if self.restore_best_weights:
                self.best_weights = self.model.get_weights()
        else:
            self.wait += 1
            if self.wait >= self.patience:
                self.stopped_epoch = epoch
                self.model.stop_training = True
                if self.restore_best_weights and self.best_weights is not None:
                    self.model.set_weights(self.best_weights)

    def on_train_end(self):
        if self.stopped_epoch > 0 and self.verbose:
            logging.info("Epoch %05d: early stopping", self.stopped_epoch + 1)


class ModelCheckpoint(object):
    """Keras ModelCheckpoint(save_best_only=True, mode='max') (model.py:326-327); the file name
    pattern is the reference's, the payload is `.npz` weights + optimizer state."""

    def __init__(self, filepath, monitor=METRIC_VAL_DCG, save_best_only=True, mode="max", verbose=0):
        self.filepath, self.monitor, self.save_best_only, self.verbose = filepath, monitor, save_best_only, verbose
        self.model = None

    def set_model(self, model):
        self.model = model

    def on_train_begin(self):
        self.best = -np.inf

    def on_epoch_end(self, epoch, logs):
        current = logs.get(self.monitor)
        if current is None:
            return
        if self.save_best_only and not current > self.best:
            return
        self.best = max(self.best, current)
        path = self.filepath.format(epoch=epoch + 1, **logs)
        self.model.save_weights(path)
        if self.verbose:
            logging.info("Epoch %05d: %s improved to %.5f, saving model to %s", epoch + 1, self.monitor, current, path)

    def on_train_end(self):
        pass


class MovierecModel(object):
    """
    Movie Recommendation Model (reference movierec/model.py:49-333).
    """

    def __init__(self, params=DEFAULT_PARAMS, model_name='movierec', output_dir="models/", verbose=1):
        # Same order of reads and checks as the reference (model.py:73-112) so that a missing key or
        # a bad value raises the same exception type at the same point.
        self._num_users = params["num_users"]
        self._num_items = params["num_items"]
        self._layers_sizes = params["layers_sizes"]
        self._layers_l2reg = params["layers_l2reg"]
        if len(self._layers_sizes) != len(self._layers_l2reg):
            raise ValueError("'layers_sizes' length = {}, 'layers_l2reg' length = {}, but must be equal."
                             .format(len(self._layers_sizes), len(self._layers_l2reg)))
        self._num_layers = len(self._layers_sizes)

        self._optimizer = params["optimizer"]
        if self._optimizer not in OPTIMIZERS:
            raise NotImplementedError("Optimizer {} is not implemented.".format(params["optimizer"]))
        self._lr = params["lr"]
        self._beta_1 = params.get("beta_1", 0.9)
        self._beta_2 = params.get("beta_2", 0.999)
        self._batch_size = params["batch_size"]
        self._num_negs_per_pos = params["num_negs_per_pos"]
        if self._num_negs_per_pos <= 0:
            raise ValueError("num_negs_per_pos must be > 0, found {}".format(self._num_negs_per_pos))
        if self._batch_size % (self._num_negs_per_pos + 1):
            raise ValueError("Batch size must be divisible by (num_negs_per_pos + 1). Found: batch_size={}, "
                             "num_negs_per_pos={}".format(self._batch_size, self._num_negs_per_pos))

        self._batch_size_eval = params["batch_size_eval"]
        self._num_negs_per_pos_eval = params["num_negs_per_pos_eval"]
        if self._num_negs_per_pos_eval <= 0:
            raise ValueError("num_negs_per_pos_eval must be > 0, found {}".format(self._num_negs_per_pos_eval))
        if self._batch_size_eval % (self._num_negs_per_pos_eval + 1):
            raise ValueError("Batch size (eval) must be divisible by (num_negs_per_pos_eval + 1). Found: "
                             "batch_size_eval={}, num_negs_per_pos_eval={}".format(self._batch_size_eval,
                                                                                   self._num_negs_per_pos_eval))

        self._k = params.get("k", self._num_negs_per_pos + 1)
        if self._k > (self._num_negs_per_pos + 1):  # the reference checks the TRAIN negatives only (model.py:108-112)
            raise ValueError("'k' must be lower than (num_negs_per_pos + 1) and lower than (num_negs_per_pos_eval + 1)."
                             "Found: k={}, num_negs_per_pos={}, num_negs_per_pos_eval={}"
                             .format(self._k, self._num_negs_per_pos, self._num_negs_per_pos_eval))

        # optional extensions; defaults reproduce the reference model exactly
        self._mf_dim = params.get("mf_dim", 0)
        self._adam_mode = params.get("adam_mode", "dense")
        self._seed = params.get("seed", None)

        os.makedirs(output_dir, exist_ok=True)
        self.name = model_name
        self._model_weights_path = self.get_model_weights_path(output_dir, model_name)
        self._params_path = self.get_params_json_path(output_dir, model_name)
        self._serialized_params = json.dumps(params)
        self._output_model_checkpoints = os.path.join(
            output_dir, "{}-checkpoint-{{epoch:02d}}-{{val_loss:.2f}}.h5".format(model_name))
        self.verbose = verbose

        self.model = self.build_mlp_model()
        self.compile_model()

    def build_mlp_model(self):
        """
        [ User Embedding ][ Item Embedding ] -> N x [ Hidden Dense ReLU ] -> [ Prediction (sigmoid) ]
        (+ GMF branch when mf_dim > 0) -- reference model.py:135-195, built as device tensors.
        """
        eng = _engine_module().NeuMFEngine(
            self._num_users, self._num_items, self._layers_sizes, self._layers_l2reg, mf_dim=self._mf_dim,
            optimizer=self._optimizer, lr=self._lr, beta_1=self._beta_1, beta_2=self._beta_2,
            table_mode=self._adam_mode, seed=self._seed)
        return NeuMFModel(self, eng)

    def compile_model(self):
        # optimizer, BCE loss and the hr/dcg metrics are part of the fused train step
        # (reference model.py:197-215); nothing to build here beyond a consistency check.
        if self._optimizer not in OPTIMIZERS:
            raise NotImplementedError("Optimizer {} is not implemented.".format(self._optimizer))

    @staticmethod
    def get_model_weights_path(output_dir, model_name):
        return os.path.join(output_dir, "{}_weights.h5".format(model_name))

    @staticmethod
    def get_params_json_path(output_dir, model_name):
        return os.path.join(output_dir, "{}_params.json".format(model_name))

    def get_pred_rank(self):
        """Callable standing in for the rank layer's output tensor (model.py:225-234)."""
        return RankLayer(self._num_negs_per_pos, self._num_negs_per_pos_eval, name=OUTPUT_RANK)

    def log_summary(self):
        self.model.summary(print_fn=logging.info)

    def save(self):
        """Save params and weights to files (model.py:239-249)."""
        self.model.save_weights(self._model_weights_path)
        logging.info('Model weights saved to: {}'.format(self._model_weights_path))
        with open(self._params_path, 'w') as f_out:
            f_out.write(self._serialized_params)
        logging.info('Model params saved to: {}'.format(self._params_path))

    @staticmethod
    def load_from_dir(model_dir, model_name, verbose=1):
        params_path = MovierecModel.get_params_json_path(model_dir, model_name)
        weights_path = MovierecModel.get_model_weights_path(model_dir, model_name)
        return MovierecModel.load_from_files(params_path, weights_path, model_dir, model_name, verbose)

    @staticmethod
    def load_from_files(params_path, weights_path, output_model_dir, output_model_name, verbose=1):
        with open(params_path, 'r') as f_in:
            params = json.load(f_in)
        movierec = MovierecModel(params, output_model_name, output_model_dir, verbose)
        movierec.model.load_weights(weights_path)
        return movierec

    def fit_generator(self, train_data_generator, validation_data_generator, epochs):
        """Training loop with the reference's callbacks (model.py:305-333): early stopping on
        `val_output_dcg` (patience 5, best weights restored) and best-only checkpoints."""
        callbacks = [
            EarlyStopping(monitor=METRIC_VAL_DCG, mode='max', restore_best_weights=True,
                          patience=EARLY_STOPPING_PATIENCE, verbose=self.verbose),
            ModelCheckpoint(self._output_model_checkpoints, monitor=METRIC_VAL_DCG, save_best_only=True,
                            mode='max', verbose=self.verbose),
        ]
        return self.model.fit_generator(generator=train_data_generator,
                                        validation_data=validation_data_generator,
                                        epochs=epochs, callbacks=callbacks, verbose=self.verbose)

    def fold_in(self, histories, steps=None, lr=None, negs=None, seed=0, init_users=None):
        """Fold-in of users the model was not trained on (or of known users whose history has grown): the item tables
        and the dense block stay frozen and only each user's two embedding rows are optimised, on the device, against
        the user's history and sampled negatives.  histories: a list of item arrays (one per user, any order) or a
        (rowptr, items) CSR of ascending lists.  steps / lr default to FOLD_IN_STEPS / FOLD_IN_LR, negs to the model's
        num_negs_per_pos; the optimiser is the model's.  init_users: per user, the model row to start from (-1 = zero
        rows, the default).  Returns a FoldedModel whose user id u is new user u: recommend_for_users, recommend_batch,
        evaluate_full_catalogue and evaluate_full_catalogue_sets work on it unchanged; .user_weights() gives the rows
        and .loss each user's last-step loss.  Raises IndexError on an out-of-range item or init user and ValueError on
        a malformed CSR or a history that covers every item."""
        eng = self.model.engine
        mlp, gmf, loss = eng.fold_in(histories, FOLD_IN_STEPS if steps is None else steps,
                                     FOLD_IN_LR if lr is None else lr,
                                     self._num_negs_per_pos if negs is None else negs, seed=seed, init_users=init_users)
        return FoldedModel(self, mlp, gmf, loss)

    def evaluate(self, users, items, k=None):
        """Full-sweep ranking evaluation (BASELINE config 4): one user id per group and
        (negs_eval+1) candidate items per user with the positive last.  Returns (hr, dcg)."""
        group = self._num_negs_per_pos_eval + 1
        k = self._k if k is None else k
        import torch
        eng = self.model.engine
        # (the fused eval kernels rank a candidate with an out-of-range id last and say nothing: the engine checks the
        # ids on the device -- four reductions next to a sweep of millions of rows -- and the verdict is read back
        # with the sums; host arrays are uploaded in chunks under the sweep, see NeuMFEngine.rank_eval)
        pos, sums, _, _ = eng.rank_eval(users, items, group, k, check_ids=True)
        bad = eng.last_eval_bad.to(sums.dtype)
        s = torch.cat([sums.reshape(-1), bad]).cpu().numpy().astype(np.float64)
        self.model._raise_on_bad_ids(s[2])
        G = max(int(pos.numel()), 1)
        return s[0] / G, s[1] / G

    def evaluate_full_catalogue(self, users, items, exclude=None, k=None):
        """Leave-one-out ranking evaluation against ALL items (no sampled negatives): for user users[g], the held-out
        item items[g] is ranked among every item not in the user's exclusion list (the held-out item itself always
        counts).  exclude: as NeuMFModel.recommend_for_users -- typically the training generator, whose lists hold
        every item the user has already rated.  Returns (hr, ndcg) at k (default: the model's k), like evaluate()."""
        k = self._k if k is None else k
        import torch
        eng = self.model.engine
        _, _, pos, sums, _ = eng.catalogue_topk(users, k, exclude=_exclusion_lists(exclude), targets=items)
        s = torch.cat([sums.reshape(-1), eng.last_catalogue_bad.to(sums.dtype)]).cpu().numpy().astype(np.float64)
        self.model._raise_on_bad_ids(s[2])
        G = max(int(pos.numel()), 1)
        return s[0] / G, s[1] / G

    def evaluate_candidate_lists(self, users, candidate_lists, targets, k=None):
        """Ranking evaluation with a candidate list of its own size per user (e.g. users with fewer unseen items than
        the negative count, or candidates from a retrieval stage): for user users[u], the candidate at position
        targets[u] of its list is ranked among the whole list.  candidate_lists as NeuMFModel.recommend_batch.
        Returns (hr, ndcg) at k (default: the model's k), like evaluate().  Raises IndexError on an out-of-range user,
        item or target position."""
        k = self._k if k is None else k
        import torch
        users = np.asarray(users, dtype=np.int32).reshape(-1)
        targets = np.asarray(targets, dtype=np.int32).reshape(-1)
        if targets.size != users.size:
            raise ValueError("targets ({}) and users ({}) differ in length".format(targets.size, users.size))
        rowptr, items = _candidate_csr(candidate_lists, users.size)
        eng = self.model.engine
        self.model._raise_on_bad_ids(_ids_outside(users, eng.num_users) or _ids_outside(items, eng.num_items) or
                                     bool(np.any((targets < 0) | (targets >= rowptr[1:] - rowptr[:-1]))))
        sums = []
        for lo, hi in _list_chunks(rowptr):
            r0, r1 = int(rowptr[lo]), int(rowptr[hi])
            sums.append(eng.rank_lists(users[lo:hi], (rowptr[lo:hi + 1] - r0, items[r0:r1]), k,
                                       targets=targets[lo:hi])[4])
        total = torch.stack(sums).cpu().numpy().astype(np.float64).sum(axis=0)  # chunk order
        G = max(int(users.size), 1)
        return total[0] / G, total[1] / G

    def evaluate_full_catalogue_sets(self, test, exclude=None, ks=None):
        """All-items ranking evaluation with several held-out items per user (a per-user last-20 % or temporal split,
        all of a user's future ratings): each held-out item is ranked among every item not on the user's exclusion list
        plus the user's held-out items (which are never excluded).  test: a ratings DataFrame (user / item columns) or
        a (rowptr, items) CSR indexed by user id with ascending lists; the users evaluated are those with a non-empty
        list.  exclude: as evaluate_full_catalogue -- typically the training generator.  ks: cutoffs (default: the
        model's k).  Returns the means over the users evaluated: {"mrr", "hr@k", "precision@k", "recall@k", "ndcg@k",
        "map@k"} for every cutoff k.  Raises IndexError on an out-of-range user or item."""
        ks = (self._k,) if ks is None else tuple(int(k) for k in np.asarray(ks).reshape(-1))
        import torch
        eng = self.model.engine
        nu, ni = eng.num_users, eng.num_items
        if hasattr(test, "columns"):
            from . import data_pipeline as dp
            u = np.asarray(test[dp.COL_USER_ID], dtype=np.int64)
            i = np.asarray(test[dp.COL_ITEM_ID], dtype=np.int64)
            self.model._raise_on_bad_ids(_ids_outside(u, nu) or _ids_outside(i, ni))
            rowptr, items = np.zeros(nu + 1, np.int64), np.zeros(0, np.int32)
            if u.size:
                rp, it = _engine_module().build_user_csr(u.astype(np.int32), i.astype(np.int32), nu, ni)
                rowptr, items = rp.cpu().numpy(), it.cpu().numpy()
        else:
            rp, it = test
            rowptr = np.asarray(rp.cpu() if hasattr(rp, "cpu") else rp, dtype=np.int64).reshape(-1)
            items = np.asarray(it.cpu() if hasattr(it, "cpu") else it, dtype=np.int64).reshape(-1)
            if rowptr.size < 1 or rowptr[0] != 0 or rowptr[-1] != items.size or np.any(rowptr[1:] < rowptr[:-1]):
                raise ValueError("test lists: offsets must start at 0, never decrease and end at {}".format(items.size))
            self.model._raise_on_bad_ids(_ids_outside(items, ni) or bool(np.any(rowptr[nu + 1:] > rowptr[nu])))
            inner = np.ones(max(items.size - 1, 0), bool)
            inner[rowptr[1:-1][(rowptr[1:-1] > 0) & (rowptr[1:-1] < items.size)] - 1] = False
            if np.any((items[1:] <= items[:-1]) & inner):
                raise ValueError("test lists: every user's items must be strictly ascending")
            items = items.astype(np.int32)
        users = np.flatnonzero(rowptr[1:] > rowptr[:-1]).astype(np.int32)
        total = np.zeros(2 + 5 * len(ks), np.float64)  # [users, mrr] + 5 per cutoff: MR_TGT_* of movierec_b200.h
        if users.size:
            r0, r1 = int(rowptr[users[0]]), int(rowptr[users[-1] + 1])
            sub_rowptr = np.append(rowptr[users], r1) - r0
            sub_items = items[r0:r1]
            excl = _exclusion_lists(exclude)
            sums = []
            for lo, hi in _list_chunks(sub_rowptr, TARGETS_CALL_ROWS):
                a, b = int(sub_rowptr[lo]), int(sub_rowptr[hi])
                sums.append(eng.catalogue_targets(users[lo:hi], (sub_rowptr[lo:hi + 1] - a, sub_items[a:b]), ks,
                                                  exclude=excl)[1])
            total = torch.stack(sums).cpu().numpy().astype(np.float64).sum(axis=0)  # call order
        G = max(total[0], 1.0)
        out = {"mrr": total[1] / G}
        for c, k in enumerate(ks):
            for m, name in enumerate(("hr", "precision", "recall", "ndcg", "map")):
                out["{}@{}".format(name, k)] = total[2 + 5 * c + m] / G
        return out


class FoldedModel(MovierecModel):
    """MovierecModel.fold_in's result: user id u is new user u, items and dense block are the model's (shared).
    Scoring and evaluation work as on the model; training and saving raise."""

    def __init__(self, base, user_mlp, user_gmf, loss):
        self.__dict__.update(base.__dict__)
        view = base.model.engine.user_view(user_mlp, user_gmf)
        self._num_users = view.num_users
        self.model = _FoldedNeuMF(self, view)
        self.loss = loss.cpu().numpy()

    def user_weights(self):
        """The folded rows as NumPy: (user_mlp (U, L[0]/2), user_gmf (U, mf_dim) or None)."""
        e = self.model.engine
        return e.user_mlp.cpu().numpy(), (e.user_gmf.cpu().numpy() if e.user_gmf is not None else None)

    def _no_training(self, *args, **kwargs):
        raise RuntimeError("a folded-in model only scores: train or save the model it was folded into")

    fit_generator = save = _no_training


class _FoldedNeuMF(NeuMFModel):
    def _no_training(self, *args, **kwargs):
        raise RuntimeError("a folded-in model only scores: train or save the model it was folded into")

    train_on_batch = fit_generator = save_weights = load_weights = set_weights = _no_training


LISTS_CALL_ROWS = 1 << 22  # candidates per device call of recommend_batch / evaluate_candidate_lists
TARGETS_CALL_ROWS = (1 << 31) - 1  # held-out items per device call of evaluate_full_catalogue_sets (int32 counts)


def _candidate_csr(candidate_lists, U):
    """A (rowptr, items) tuple or a sequence of 1-D item arrays -> host (rowptr int64 (U + 1,), items int32)."""
    if isinstance(candidate_lists, tuple) and len(candidate_lists) == 2:
        rp, it = candidate_lists
        rowptr = np.asarray(rp.cpu() if hasattr(rp, "cpu") else rp, dtype=np.int64).reshape(-1)
        items = np.asarray(it.cpu() if hasattr(it, "cpu") else it, dtype=np.int32).reshape(-1)
    else:
        parts = [np.asarray(x, dtype=np.int32).reshape(-1) for x in candidate_lists]
        rowptr = np.zeros(len(parts) + 1, np.int64)
        rowptr[1:] = np.cumsum([p.size for p in parts])
        items = np.concatenate(parts) if parts else np.zeros(0, np.int32)
    if rowptr.size != U + 1 or rowptr[0] != 0 or rowptr[-1] != items.size or np.any(rowptr[1:] < rowptr[:-1]):
        raise ValueError("candidate lists: expected {} lists with offsets starting at 0, never decreasing and ending at "
                         "{}".format(U, items.size))
    return rowptr, items


def _ids_outside(ids, limit):
    return bool(ids.size) and bool(ids.min() < 0 or ids.max() >= limit)


def _list_chunks(rowptr, max_rows=None):
    """[lo, hi) ranges of whole lists of at most max_rows candidates each (a longer list alone)."""
    max_rows = LISTS_CALL_ROWS if max_rows is None else max_rows
    U = rowptr.size - 1
    out, lo = [], 0
    while lo < U:
        hi = int(np.searchsorted(rowptr, rowptr[lo] + max_rows, side="right")) - 1
        hi = min(max(hi, lo + 1), U)
        out.append((lo, hi))
        lo = hi
    return out or [(0, 0)]


def _exclusion_lists(exclude):
    """None | MovieLensDataGenerator | (rowptr, items) -> None | (rowptr, items)."""
    if exclude is None:
        return None
    if hasattr(exclude, "user_item_lists"):
        return exclude.user_item_lists()
    rowptr, items = exclude
    return rowptr, items


class RankLayer(object):
    """Rank of every item inside its (negs+1)-wide group, descending score, lower index first among
    equal scores (reference model.py:336-358).  `call` accepts array-likes or device tensors and
    returns an int32 NumPy array of shape (groups, negs+1)."""

    learning_phase = 0  # 1 = training phase: group width uses the train negatives (model.py:347)

    def __init__(self, num_negs_per_pos_train, num_negs_per_pos_eval, name, **kwargs):
        self.name = name
        self.num_negs_per_pos_train = num_negs_per_pos_train
        self.num_negs_per_pos_eval = num_negs_per_pos_eval

    def call(self, inputs, training=None, **kwargs):
        training = bool(RankLayer.learning_phase) if training is None else training
        negs = self.num_negs_per_pos_train if training else self.num_negs_per_pos_eval
        rank, _, _ = _engine_module().rank_scores(_flat_scores(inputs), negs + 1, negs + 1, want_rank=True)
        return rank.cpu().numpy()

    __call__ = call

    def get_config(self):
        return {'name': self.name, 'num_negs_per_pos_train': self.num_negs_per_pos_train,
                'num_negs_per_pos_eval': self.num_negs_per_pos_eval}


def set_learning_phase(value):
    """Stand-in for K.set_learning_phase used by the reference's rank-layer test."""
    RankLayer.learning_phase = int(value)


def _flat_scores(x):
    if hasattr(x, "detach"):
        return x.detach().reshape(-1)
    return np.asarray(x, dtype=np.float32).reshape(-1)


def _positions_from_rank(y_true, pred_rank_idx, k):
    """(hit_sum, dcg_sum, groups) for a given rank permutation, on device: item j of a group gets the
    pseudo-score -(its place in the rank), so the kernel's position of the label column is exactly
    `where(rank == argmax(y_true))` of model.py:447-451."""
    import torch
    eng = _engine_module()
    eng.require_cuda()
    dev = torch.device("cuda:{}".format(torch.cuda.current_device()))
    rank = torch.as_tensor(np.asarray(pred_rank_idx), device=dev).long()
    G, group = rank.shape
    y = torch.as_tensor(np.asarray(y_true), device=dev).reshape(G, group)
    label_col = torch.argmax(y, dim=1).to(torch.int32)
    place = torch.arange(group, device=dev, dtype=torch.float32).expand(G, group)
    scores = torch.empty((G, group), dtype=torch.float32, device=dev)
    scores.scatter_(1, rank, -place)
    _, _, sums = eng.rank_scores(scores, group, k, label_col=label_col, want_rank=False, device=dev)
    s = sums.cpu().numpy().astype(np.float64)
    return s[0], s[1], G


def hit_rate(y_true, _, k, pred_rank_idx):
    """HR@k of a batch (reference model.py:361-385)."""
    hits, _, G = _positions_from_rank(y_true, pred_rank_idx, k)
    return np.float32(hits / G)


def discounted_cumulative_gain(y_true, _, k, pred_rank_idx):
    """DCG@k of a batch, ln2/ln(pos+2) on hits (reference model.py:388-417)."""
    _, dcg, G = _positions_from_rank(y_true, pred_rank_idx, k)
    return np.float32(dcg / G)
