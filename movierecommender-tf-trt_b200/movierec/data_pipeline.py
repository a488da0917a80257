""" Batches of MovieLens positives with freshly sampled negatives (reference movierec/data_pipeline.py).

`MovieLensDataGenerator` keeps the reference's constructor, `len()`, `[idx]`, `on_epoch_end()` and
properties; the per-positive pandas scan + `np.setdiff1d` + `np.random.choice` of
`_get_random_negatives_and_positive` (reference :99-113) is replaced by the on-device counter-based
sampler (`mr_sample_negatives`): the user's interactions live in a sorted CSR in HBM and a whole
batch is sampled by one kernel.  `gen[idx]` returns NumPy arrays like the reference; the training
loop uses `device_batch(idx)` and never leaves the GPU.
"""

import logging

import numpy as np
import pandas as pd

try:  # package import (movierec.data_pipeline) and the reference's script-style import both work
    from .util import movielens_utils as ml
    from .util.movielens_utils import load_ratings_data
except ImportError:  # pragma: no cover
    import util.movielens_utils as ml
    from util.movielens_utils import load_ratings_data

COL_USER_ID = 'userId'
COL_ITEM_ID = 'itemId'
COL_RATING = 'rating'
COL_LABEL = 'label'


class MovieLensDataGenerator(object):
    # every batch is made of groups of one user: negatives first, the positive last (reference
    # data_pipeline.py:99-150); the trainer passes this on so the kernels can share the user-only work
    grouped_batches = True

    def __init__(self, dataset_name, data_df, batch_size, negatives_per_positive, extra_data_df=None, shuffle=True,
                 seed=None):
        """
        Same parameters as the reference (data_pipeline.py:19-46).  `seed` (optional, new) fixes the
        sampler's key; by default it is drawn from NumPy's global RNG so `np.random.seed` governs it.
        """
        if dataset_name not in ml.MOVIELENS_DATASET_NAMES:
            raise ValueError('Invalid dataset name {}. Must be one of {}'
                             .format(dataset_name, ', '.join(ml.MOVIELENS_DATASET_NAMES)))
        if negatives_per_positive <= 0:
            raise ValueError("negatives_per_positive must be > 0, found {}".format(negatives_per_positive))
        if batch_size % (negatives_per_positive + 1):
            raise ValueError("Batch size must be divisible by (negatives_per_positive + 1). Found: batch_size={}, "
                             "negatives_per_positive={}".format(batch_size, negatives_per_positive))

        self._dataset_name = dataset_name
        self._num_users = ml.NUM_USERS[dataset_name]
        self._num_items = ml.NUM_ITEMS[dataset_name]
        self.data = data_df
        self.extra_data = extra_data_df
        self.batch_size = batch_size
        self.negatives_per_positive = negatives_per_positive
        self.num_positives_per_batch = self.batch_size // (negatives_per_positive + 1)
        self.num_negatives_per_batch = self.batch_size - self.num_positives_per_batch
        self.shuffle = shuffle
        self.indexes = np.arange(len(self.data))
        self._draw = 0          # bumps on every batch request: repeated gen[idx] calls differ (reference :111-112)
        self._device = None     # CSR and positives are uploaded on first use

        self.on_epoch_end()  # first shuffle consumes NumPy's global RNG exactly as the reference (:71)
        self._seed = int(np.random.randint(0, 2 ** 31 - 1)) if seed is None else int(seed)
        logging.info('Created generator for {}. Num users={}, num items={}, num_batches={}, batch size={}, '
                     'positives per batch={}, negatives per batch={}'
                     .format(dataset_name, self._num_users, self._num_items, len(self), batch_size,
                             self.num_positives_per_batch, self.num_negatives_per_batch))

    @property
    def num_users(self):
        return self._num_users

    @property
    def num_items(self):
        return self._num_items

    @property
    def dataset_name(self):
        return self._dataset_name

    def __len__(self):
        """Number of batches: floor(len(data) / batch_size), as the reference (data_pipeline.py:97)."""
        return int(np.floor(len(self.indexes) / self.batch_size))

    # ---- device state ------------------------------------------------------------------------------
    def _all_pairs(self):
        """(users, items) int64 of data ∪ extra_data, with their id bounds (max + 1, at least 1)."""
        users = np.asarray(self.data[COL_USER_ID].values, dtype=np.int64)
        items = np.asarray(self.data[COL_ITEM_ID].values, dtype=np.int64)
        all_u, all_i = users, items
        if self.extra_data is not None:
            all_u = np.concatenate([users, np.asarray(self.extra_data[COL_USER_ID].values, dtype=np.int64)])
            all_i = np.concatenate([items, np.asarray(self.extra_data[COL_ITEM_ID].values, dtype=np.int64)])
        if len(all_u) and (all_u.min() < 0 or all_i.min() < 0):
            raise ValueError("negative user / item ids")
        n_u = int(all_u.max()) + 1 if len(all_u) else 1
        n_i = int(all_i.max()) + 1 if len(all_i) else 1
        return all_u, all_i, n_u, n_i

    def _upload(self):
        import torch
        from . import _engine
        _engine.require_cuda()
        dev = torch.device("cuda:{}".format(torch.cuda.current_device()))
        users = np.asarray(self.data[COL_USER_ID].values, dtype=np.int64)
        items = np.asarray(self.data[COL_ITEM_ID].values, dtype=np.int64)
        # per-user sorted item lists built on the device (mr_build_user_csr: two stable radix sorts + compaction);
        # build_user_csr below is the same table in NumPy, kept for host-side use and as the tests' cross-check
        all_u, all_i, n_u, n_i = self._all_pairs()
        rowptr, csr = _engine.build_user_csr(all_u.astype(np.int32), all_i.astype(np.int32), n_u, n_i)
        self._device = {
            "dev": dev,
            "rowptr": rowptr,
            "csr": csr,
            "users": torch.from_numpy(users.astype(np.int32)).to(dev),
            "items": torch.from_numpy(items.astype(np.int32)).to(dev),
            "min_candidates_checked": False,
            "degree_max": int((rowptr[1:] - rowptr[:-1]).max().item()) if rowptr.numel() > 1 else 0,
        }

    def _max_seen_below(self, num_items):
        """Largest number of DISTINCT seen items below `num_items` any user has (only those take candidates away)."""
        import torch
        d = self._device
        key = ("seen_below", int(num_items))
        if key not in d:
            below = torch.cat([torch.zeros(1, dtype=torch.int64, device=d["dev"]),
                               (d["csr"] < num_items).to(torch.int64).cumsum(0)])
            rp = d["rowptr"].to(torch.int64)
            d[key] = int((below[rp[1:]] - below[rp[:-1]]).max().item()) if rp.numel() > 1 else 0
        return d[key]

    def user_item_lists(self):
        """(rowptr int64, items int32) device tensors: per user, the ascending distinct items of data ∪ extra_data --
        the items the sampler never draws as negatives, and the exclusion lists of a full-catalogue evaluation."""
        if self._device is None:
            self._upload()
        return self._device["rowptr"], self._device["csr"]

    def item_user_lists(self):
        """(rowptr int64, users int32) device tensors: per item, the ascending distinct users of data ∪ extra_data --
        user_item_lists transposed (the same device build with the roles swapped), the exclusion lists of an
        audience: who has already rated the item."""
        if self._device is None:
            self._upload()
        d = self._device
        if "item_rowptr" not in d:
            from . import _engine
            all_u, all_i, n_u, n_i = self._all_pairs()
            d["item_rowptr"], d["item_csr"] = _engine.build_user_csr(all_i.astype(np.int32), all_u.astype(np.int32), n_i,
                                                                     n_u)
        return d["item_rowptr"], d["item_csr"]

    def device_batch(self, idx):
        """Batch `idx` as device tensors ([x_user int32, x_item int32], y float32), layout of the
        reference's __getitem__ (:136-150): users repeated, negatives first, positive last."""
        import torch
        from . import _engine
        if self._device is None:
            self._upload()
        d = self._device
        num_items = self.num_items  # read through the property: the reference's tests patch it
        if d["degree_max"] >= num_items and self._max_seen_below(num_items) >= num_items:
            raise ValueError("a user has interacted with every item: no candidate negatives "
                             "(np.random.choice would raise 'a cannot be empty' in the reference)")
        P = self.num_positives_per_batch
        sel = torch.from_numpy(self.indexes[idx * P:(idx + 1) * P]).to(d["dev"])
        pos_u, pos_i = d["users"][sel], d["items"][sel]
        self._draw += 1
        xu, xi, y = _engine.sample_negatives(d["rowptr"], d["csr"], num_items, pos_u, pos_i, idx * P,
                                             self.negatives_per_positive, self._seed, self._draw)
        return [xu, xi], y

    def __getitem__(self, idx):
        """([x_user, x_item], y) NumPy arrays of length batch_size (reference :115-150)."""
        (xu, xi), y = self.device_batch(idx)
        return [xu.cpu().numpy(), xi.cpu().numpy()], y.cpu().numpy().astype(np.int64)

    def on_epoch_end(self):
        if self.shuffle:
            np.random.shuffle(self.indexes)


def build_user_csr(users, items):
    """Per-user sorted, de-duplicated item lists: (rowptr int64 (max_user+2,), items int32)."""
    users = np.asarray(users, dtype=np.int64)
    items = np.asarray(items, dtype=np.int64)
    if users.size == 0:
        return np.zeros(1, np.int64), np.zeros(0, np.int32)
    key = np.unique((users << 32) | items)
    u = key >> 32
    counts = np.bincount(u, minlength=int(u.max()) + 1)
    rowptr = np.zeros(len(counts) + 1, np.int64)
    np.cumsum(counts, out=rowptr[1:])
    return rowptr, (key & 0xFFFFFFFF).astype(np.int32)


def _cuda_available():
    try:
        import torch
        return bool(torch.cuda.is_available())
    except ImportError:  # pragma: no cover
        return False


def split_leave_last_two_out(ratings_df, col_user=COL_USER_ID, on_device=None):
    """Per user, in file order: last rating -> test, second last -> validation, the rest -> train
    (reference data_pipeline.py:190-198); each part ordered by user then file order, index reset.
    on_device: None = on the GPU when there is one (20 M ratings: milliseconds instead of seconds of pandas /
    NumPy), False = the NumPy statement of the same rule (host-only environments), True = require the GPU."""
    users = np.asarray(ratings_df[col_user].values)
    order = is_last = is_second_last = None
    if on_device is None:
        on_device = _cuda_available() and len(users) > 0 and users.min() >= 0 and users.max() < 2 ** 31 - 1
    if on_device:  # mr_split_last_two: stable radix sort by user + one pass over the sorted users
        from . import _engine
        d_order, d_part = _engine.split_last_two(users.astype(np.int32), int(users.max()) + 1)
        order, part = d_order.cpu().numpy().astype(np.int64), d_part.cpu().numpy()
        is_last, is_second_last = part == 2, part == 1
    else:
        order = np.argsort(users, kind="stable")
        su = users[order]
        n = len(su)
        is_last = np.ones(n, bool)
        is_last[:-1] = su[1:] != su[:-1]
        is_second_last = np.zeros(n, bool)
        is_second_last[:-1] = is_last[1:] & (su[:-1] == su[1:])
    test = ratings_df.iloc[order[is_last]].reset_index(drop=True)
    validation = ratings_df.iloc[order[is_second_last]].reset_index(drop=True)
    train = ratings_df.iloc[order[~(is_last | is_second_last)]].reset_index(drop=True)
    return train, validation, test


def remap_dense_ids(ratings_df, columns=(COL_USER_ID, COL_ITEM_ID), on_device=None):
    """New in this package (the reference keeps the raw, 1-based, sparse MovieLens ids and sizes its tables by
    constants, movielens_utils.py:51-55): replace the ids of each column by their rank among the distinct ids.
    Returns (DataFrame with dense ids, {column: array of the original id of every dense id}).  On the GPU when there
    is one (mr_remap_ids), else np.unique."""
    out = ratings_df.copy()
    maps = {}
    if on_device is None:
        on_device = _cuda_available()
    for col in columns:
        ids = np.asarray(ratings_df[col].values)
        if on_device and len(ids) and ids.min() >= 0 and ids.max() < 2 ** 31 - 1:
            from . import _engine
            dense, unique = _engine.remap_ids(ids.astype(np.int32))
            out[col] = dense.cpu().numpy().astype(ids.dtype)
            maps[col] = unique.cpu().numpy().astype(ids.dtype)
        else:
            unique, dense = np.unique(ids, return_inverse=True)
            out[col] = dense.reshape(-1).astype(ids.dtype)
            maps[col] = unique
    return out, maps


def load_ratings_train_test_sets(dataset_name, data_dir, download=True):
    """
    Load a Movielens ratings file and split it into (train, validation, test) DataFrames with columns
    COL_USER_ID, COL_ITEM_ID, COL_RATING (reference data_pipeline.py:157-200).
    """
    if dataset_name not in ml.MOVIELENS_DATASET_NAMES:
        raise ValueError('Invalid dataset name {}. Must be one of {}'
                         .format(dataset_name, ', '.join(ml.MOVIELENS_DATASET_NAMES)))
    ratings_df = load_ratings_data(data_dir, dataset_name, COL_USER_ID, COL_ITEM_ID, COL_RATING, download)
    return split_leave_last_two_out(ratings_df)
