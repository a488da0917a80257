"""Data-parallel training of one NeuMF model over the GPUs of a box (SURVEY 8e).

One process per GPU (`torch.distributed`, NCCL over NVLink 5 / NVSwitch on GPUs, gloo in CPU
tests).  Tables are replicated.  A global batch is split across ranks BY WHOLE GROUPS (a group = one
positive and its negatives, so the ranking metrics stay rank-local); every rank runs the fused
forward/backward on its groups with the gradient scale 1/B_global, the ranks' flat gradient buffers
(dense-layer gradients + the embedding gradient tables) are summed, and every replica receives the
identical optimizer update.  The result equals the single-GPU step on the global batch up to summation
order.  The reference is single-process (SURVEY 2.1): there is no reference collective to mirror; this
is the exchange step the data-parallel path needs and nothing more.

Two exchanges:
  "peer" (default on the GPUs of one box): parameters and gradients live in symmetric memory; the sum of the
      gradients, the optimizer step and the distribution of the new weights are ONE kernel over NVLink peer pointers
      (`mr_dp_reduce_apply`, csrc/dp_exchange.cu): every rank owns 1/world of every region, adds the ranks' gradient
      values in rank order, steps its slice with its own slice of the Adam state and stores the result into every
      replica.  The user tables' part (five sixths of the bytes at the ML-20M shape) runs on a communication stream
      as soon as every rank's user-side gradients are final (MrGrads.user_tables_ready), under the item-side half
      of the step; cross-rank barriers (symmetric-memory signal pads) order it.
  "nccl": all-reduce of the flat gradient buffer (the user part early, as above), then the full optimizer sweep on
      every rank.  Used with gloo on CPUs and when symmetric memory is not available.
"""

import os

import torch
import torch.distributed as dist


def split_groups(num_groups, world_size, rank):
    """[lo, hi) of the groups rank `rank` owns: contiguous, sizes differ by at most one."""
    base, rem = divmod(int(num_groups), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_batch(users, items, labels, group, world_size, rank):
    """Rank-local slice of a global batch laid out as the generator does (groups contiguous)."""
    n = len(labels)
    if n % group:
        raise ValueError("batch of {} rows is not divisible by the group width {}".format(n, group))
    lo, hi = split_groups(n // group, world_size, rank)
    sl = slice(lo * group, hi * group)
    return users[sl], items[sl], labels[sl]


def owner_slices(regions, world_size, rank, stage_of):
    """The elements of the flat parameter layout rank `rank` owns in the peer exchange: for every region
    (name, offset, padded count, l2) a contiguous [lo, hi) whose bounds are multiples of four elements (the kernel works
    on 16-byte pieces); over the ranks the slices of a region tile it exactly.  -> [(lo, hi, l2, stage_of(name))]."""
    out = []
    for name, off, count, l2 in regions:
        per = ((count // 4 + world_size - 1) // world_size) * 4
        lo, hi = off + min(count, per * rank), off + min(count, per * (rank + 1))
        out.append((lo, hi, l2, stage_of(name)))
    return out


class DataParallelNeuMF(object):
    """Wraps a NeuMFEngine replica; `train_step` takes the RANK-LOCAL rows of a global batch."""

    def __init__(self, engine, process_group=None, exchange=None, multicast=None):
        """exchange: "peer" | "nccl" | None (= "peer" on CUDA devices with the NCCL backend and more than one rank;
        MR_DP_EXCHANGE overrides the default for A/B runs).  multicast (peer exchange): None = NVSwitch multicast on
        more than four ranks when the buffers have a multicast address, False = peer loads / stores, True = insist."""
        if not dist.is_initialized():
            raise RuntimeError("torch.distributed is not initialised")
        if engine.table_mode != "dense":
            raise NotImplementedError("replicated data parallelism sums dense gradient tables; use table_mode='dense'")
        self.engine = engine
        self.group = process_group
        self.world_size = dist.get_world_size(process_group)
        self.rank = dist.get_rank(process_group)
        on_gpu = str(getattr(engine, "device", "cpu")).startswith("cuda")
        # MR_DP_OVERLAP=1 (nccl exchange): all-reduce region by region with the Adam sweep of one region under the
        # all-reduce of the next.  Parity-checked (tools/dp_gpu_check.py); not faster than the default on 2 GPUs.
        self.overlap = os.environ.get("MR_DP_OVERLAP") is not None
        # nccl exchange on GPUs: the all-reduce of the user tables' gradients starts as soon as they are final
        self.early_user = os.environ.get("MR_DP_NO_EARLY_USER") is None and on_gpu
        explicit = exchange is not None
        if exchange is None:
            exchange = os.environ.get("MR_DP_EXCHANGE") or (
                "peer" if on_gpu and self.world_size > 1 and dist.get_backend(process_group) == "nccl"
                and hasattr(engine, "rebind_flat") else "nccl")
        if exchange not in ("peer", "nccl"):
            raise ValueError("exchange must be 'peer' or 'nccl', found {!r}".format(exchange))
        self.exchange = exchange
        if exchange == "peer" and not self._symmetric_memory_available(explicit):
            self.exchange = exchange = "nccl"
        if os.environ.get("MR_DP_MULTICAST") is not None:  # A/B runs: 0 = peer loads / stores, 1 = insist
            multicast = os.environ["MR_DP_MULTICAST"] not in ("0", "")
        self.multicast = multicast
        self._comm = None
        self._ready = None
        if exchange == "peer":
            self._setup_peer()

    def _symmetric_memory_available(self, explicit):
        """True when EVERY rank can allocate symmetric memory on its device (the decision must be the same everywhere:
        the rendezvous that follows is a collective).  An explicit exchange="peer" raises instead of falling back."""
        ok = 1
        try:
            import torch.distributed._symmetric_memory as symm
            probe = symm.empty(1024, dtype=torch.float32, device=self.engine.device)
            del probe
        except Exception as err:  # noqa: BLE001 -- any failure means "not on this box"
            ok, why = 0, err
        flag = torch.tensor([ok], dtype=torch.int32, device=self.engine.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
        if int(flag.item()) == 1:
            return True
        if explicit:
            raise RuntimeError("exchange='peer' needs torch symmetric memory on every rank" +
                               ("" if ok else ": {}".format(why)))
        import sys
        print("movierec: symmetric memory is not available on every rank; data-parallel exchange falls back to NCCL",
              file=sys.stderr)
        return False

    def _setup_peer(self):
        """Parameters and gradients into symmetric memory (values kept), peer pointers, this rank's slices."""
        import ctypes as C
        import torch.distributed._symmetric_memory as symm
        e = self.engine
        pg = self.group if self.group is not None else dist.group.WORLD
        e.rebind_flat(lambda count: symm.empty(count, dtype=torch.float32, device=e.device))
        self._hp = symm.rendezvous(e.p_flat, pg.group_name)
        self._hg = symm.rendezvous(e.g_flat, pg.group_name)
        w = self.world_size
        self._p_peers = (C.c_void_p * w)(*[int(x) for x in self._hp.buffer_ptrs])
        self._g_peers = (C.c_void_p * w)(*[int(x) for x in self._hg.buffer_ptrs])
        # NVSwitch multicast addresses of the two buffers, when the box has them (NVLS): the switch then does the sum
        # and the replication (csrc/dp_exchange.cu); MR_DP_NO_MULTICAST keeps the peer loads / stores for A/B runs
        mc_g, mc_p = int(getattr(self._hg, "multicast_ptr", 0) or 0), int(getattr(self._hp, "multicast_ptr", 0) or 0)
        # measured (ML-20M shape, ms per step, multicast / peer): 2 GPUs 2.06 / 1.90, 4 GPUs 2.02 / 2.00, 8 GPUs
        # 2.02 / 2.09 -- the switch's reduction pays once the peer form would fetch more than four copies
        use_mc = bool(mc_g and mc_p) and (self.multicast is True or (self.multicast is None and w > 4))
        if self.multicast is True and not use_mc:
            raise RuntimeError("multicast=True, but the symmetric-memory buffers have no multicast address on this box")
        self.multicast = use_mc
        self._mc_g = C.c_void_p(mc_g) if use_mc else None
        self._mc_p = C.c_void_p(mc_p) if use_mc else None
        # (lo, hi, l2, stage) of the elements this rank owns; stage 0: the user GMF table (final first), 1: the user MLP
        # table, 2: dense block and item tables (after the step)
        from . import _engine
        one_early = os.environ.get("MR_DP_NO_GMF_SPLIT") is not None  # A/B runs: one early exchange instead of two
        stage_of = lambda name: (1 if one_early else 0) if name == _engine.K_GMF_USER else (1 if name == _engine.K_USER else 2)
        self._slices = owner_slices(e.flat_regions(), w, self.rank, stage_of)
        self._comm = torch.cuda.Stream(device=e.device)
        self._ready = torch.cuda.Event()
        self._ready.record()  # (creates the CUDA events the library records into)
        self._gmf_ready = torch.cuda.Event()
        self._gmf_ready.record()
        self._comm_done = torch.cuda.Event()

    def _reduce_apply(self, lo, hi, l2, lr_t):
        import ctypes as C
        from . import _engine
        e = self.engine
        nat = _engine.nat
        adam = e.optimizer == "adam"
        nat.check(nat.lib.mr_dp_reduce_apply(self._g_peers, self._p_peers, self.world_size, self.rank,
                                             C.c_void_p(e.m_flat.data_ptr()) if adam else None,
                                             C.c_void_p(e.v_flat.data_ptr()) if adam else None, lo, hi,
                                             nat.OPT_ADAM if adam else nat.OPT_SGD, lr_t, e.beta_1, e.beta_2,
                                             _engine.ADAM_EPSILON, l2, self._mc_g, self._mc_p, e._stream()),
                  "mr_dp_reduce_apply")

    def _peer_step(self, users, items, labels, kw):
        e = self.engine
        out = e.train_grads(users, items, labels, user_ready=self._ready, user_gmf_ready=self._gmf_ready, **kw)
        lr_t = e.step_lr_t()
        main = torch.cuda.current_stream(e.device)
        # user tables: as soon as EVERY rank's gradients of a table are final and its step no longer reads the table --
        # the GMF table right after the per-user sums, the MLP table after the first layer's per-user GEMMs.  The
        # exchange must be over before the step's item-side table GEMMs start (persistent tcgen05 kernels that need whole
        # SMs wait for the exchange CTAs to leave), so every microsecond of head start counts.
        with torch.cuda.stream(self._comm):
            for stage, event, channel in ((0, self._gmf_ready, 2), (1, self._ready, 1)):
                mine = [sl for sl in self._slices if sl[3] == stage]
                if not mine:
                    continue
                self._comm.wait_event(event)
                self._hg.barrier(channel=channel)
                for lo, hi, l2, _ in mine:
                    self._reduce_apply(lo, hi, l2, lr_t)
            self._comm_done.record(self._comm)
        # dense block and item tables: after every rank's step
        self._hg.barrier(channel=0)
        for lo, hi, l2, stage in self._slices:
            if stage == 2:
                self._reduce_apply(lo, hi, l2, lr_t)
        main.wait_event(self._comm_done)
        self._hg.barrier(channel=0)  # all owners' stores have landed: the replicas are whole again
        e.finish_apply()
        return out

    def sync_optimizer_state(self):
        """peer exchange: the Adam state is sharded by owner; this makes every rank hold all of it (checkpoints)."""
        e = self.engine
        if self.exchange != "peer" or e.optimizer != "adam":
            return
        for buf in (e.m_flat, e.v_flat):
            own = torch.zeros_like(buf)
            for lo, hi, _, _ in self._slices:
                own[lo:hi].copy_(buf[lo:hi])
            dist.all_reduce(own, op=dist.ReduceOp.SUM, group=self.group)
            buf.copy_(own)

    def broadcast_parameters(self, src=0):
        """Make every replica start from rank `src`'s weights."""
        e = self.engine
        for t in [e.dense] + list(e._tables.values()):
            dist.broadcast(t, src, group=self.group)

    def _staged(self, users, items, labels):
        """The device copies of a batch uploaded by the previous call's `prefetch`, found by the host arrays' identity."""
        staged, self._prefetched = getattr(self, "_prefetched", None), None
        if staged is not None and staged[0] == (id(users), id(items), id(labels)):
            torch.cuda.current_stream(self.engine.device).wait_event(staged[4])
            return staged[1], staged[2], staged[3]
        return users, items, labels

    def _upload(self, batch):
        from . import _engine
        e = self.engine
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(device=e.device)
        users, items, labels = batch
        with torch.cuda.stream(self._copy_stream):
            dev = (_engine.as_device_i32(users, e.device), _engine.as_device_i32(items, e.device),
                   _engine.as_device_f32(labels, e.device))
            ready = torch.cuda.Event()
            ready.record(self._copy_stream)
        self._prefetched = ((id(users), id(items), id(labels)),) + dev + (ready,)

    def train_step(self, users, items, labels, global_rows, group=0, k=0, grouped=False, prefetch=None):
        """Local forward/backward -> sum of the ranks' gradients -> identical update on every replica.
        Returns the rank-local step outputs (loss/hit/dcg sums over the local rows), a device tensor.
        grouped: see NeuMFEngine.train_step (batches are split by whole groups, so the layout survives).
        prefetch=(users, items, labels): the NEXT rank-local batch (host arrays, pinned for asynchronous copies); it is
        uploaded on a copy stream under this step, and the next call finds it by the identity of the arrays."""
        on_gpu = str(getattr(self.engine, "device", "cpu")).startswith("cuda")
        if on_gpu:
            users, items, labels = self._staged(users, items, labels)
        out = self._step(users, items, labels, global_rows, group, k, grouped)
        if prefetch is not None and on_gpu:
            self._upload(prefetch)
        return out

    def _step(self, users, items, labels, global_rows, group, k, grouped):
        e = self.engine
        # the hidden kernels' l2 term 2*l2*W is part of the gradients this call returns; the all-reduce below SUMS the
        # ranks' gradients, so only rank 0 adds it (the tables' l2 term is added by apply(), after the reduction)
        kw = dict(group=group, k=k, inv_global_batch=1.0 / float(global_rows), grouped=grouped, dense_l2=(self.rank == 0))
        if self.exchange == "peer":
            return self._peer_step(users, items, labels, kw)
        if self.early_user and hasattr(e, "gradient_parts") and e.gradient_parts()[0].numel() > 0:
            # The user tables' gradients (five sixths of the bytes at the ML-20M shape) are final well before the end
            # of the step: their all-reduce starts on the communication stream as soon as the library signals it and
            # runs under the item-side reduction and GEMMs; only the rest is reduced after the step's last kernel.
            if self._comm is None:
                self._comm = torch.cuda.Stream(device=e.device)
                self._ready = torch.cuda.Event()
                self._ready.record()  # (creates the CUDA event the library records into)
            out = e.train_grads(users, items, labels, user_ready=self._ready, **kw)
            g_user, g_rest = e.gradient_parts()
            with torch.cuda.stream(self._comm):
                self._comm.wait_event(self._ready)
                w_user = dist.all_reduce(g_user, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
            w_rest = dist.all_reduce(g_rest, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
            w_user.wait()
            w_rest.wait()
            e.apply()
            return out
        out = e.train_grads(users, items, labels, **kw)
        if self.overlap and hasattr(e, "gradient_regions"):
            # region by region, largest first: the Adam sweep of one region runs (on the compute stream) under the
            # all-reduce of the next ones (on NCCL's stream); work.wait() orders the streams, the host never blocks
            regions = e.gradient_regions()
            works = [dist.all_reduce(g, op=dist.ReduceOp.SUM, group=self.group, async_op=True) for _, g in regions]
            for (name, _), w in zip(regions, works):
                w.wait()
                e.apply_region(name)
            e.finish_apply()
            return out
        for t in e.gradient_tensors():
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        e.apply()
        return out

    def all_reduce_sums(self, t):
        """Sum metric / loss accumulators over ranks (reporting only)."""
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        return t


class ShardedNeuMF(object):
    """Row-sharded embedding tables for models whose tables do not fit one GPU (BASELINE config 5:
    10 M users x 1 M items): owner(row) = row % world, local index = row // world; the dense tower is
    replicated.  One step on every rank:

      1. unique user / item ids of the local batch, grouped by owner;
      2. all-to-all of the ids, owners gather the rows (gather kernel), all-to-all of the rows back:
         the rank now holds a compact cache of exactly the rows its batch needs;
      3. the ordinary fused forward/backward on the cache (ids remapped to cache slots), gradient scale
         1/B_global -> gradient rows of the cache, dense gradients;
      4. all-to-all of the gradient rows to the owners, which sort them by row, sum duplicates in a fixed
         order and apply the sparse-row optimizer (mr_sparse_rows_update); all-reduce of the dense
         gradients and the identical dense update everywhere.

    The result equals the single-GPU step in sparse-row ("lazy") Adam mode on the global batch up to
    summation order.  All arithmetic is in the CUDA library.

    peer_gather (default on GPUs of one box): the shards live in torch symmetric memory, every rank holds the
    peer pointers of all slices, and step 2 is ONE kernel (`mr_gather_rows_sharded`) that reads each needed row
    from its owner's memory over NVLink straight into the cache -- no exchange of gathered rows, no owner-side
    gather, no staging copies; the ids still go to the owners (4 bytes a row) because the gradient rows of
    step 4 follow them.  A symmetric-memory barrier at the start of the step orders the gathers after the
    owners' updates of the previous step.  With peer_gather off, step 2 is the NCCL all-to-all pair."""

    def __init__(self, num_users, num_items, layers_sizes, mf_dim=0, optimizer="adam", lr=1e-3, beta_1=0.9,
                 beta_2=0.999, max_local_rows=1 << 20, seed=None, process_group=None, peer_gather=None):
        import numpy as np
        from . import _engine
        if not dist.is_initialized():
            raise RuntimeError("torch.distributed is not initialised")
        self._engine_mod = _engine
        self.group = process_group
        self.world = dist.get_world_size(process_group)
        self.rank = dist.get_rank(process_group)
        self.num_users, self.num_items = int(num_users), int(num_items)
        self.optimizer = optimizer
        # the per-step row cache + the replicated dense tower: an ordinary engine without table state
        self.cache = _engine.NeuMFEngine(max_local_rows, max_local_rows, layers_sizes, [0.0] * len(layers_sizes),
                                         mf_dim=mf_dim, optimizer=optimizer, lr=lr, beta_1=beta_1, beta_2=beta_2,
                                         table_mode="dense", seed=seed, table_state=False)
        self.capacity = int(max_local_rows)
        e = self.cache
        dev = e.device
        self.f = e.mf_dim
        rng = np.random.default_rng(None if seed is None else seed + 7919 * (self.rank + 1))
        self.shard = {}
        symm = None
        if peer_gather is None:
            peer_gather = dev.type == "cuda" and dist.get_backend(process_group) == "nccl"
        if peer_gather:
            import torch.distributed._symmetric_memory as symm  # peer pointers over NVLink (one box)
        self.peer_gather = bool(peer_gather)
        self._barrier_handle = None
        pg_name = (process_group if process_group is not None else dist.group.WORLD).group_name if peer_gather else None
        for side, total, d in (("user", self.num_users, e.d_u), ("item", self.num_items, e.d_i)):
            rows = (total - self.rank + self.world - 1) // self.world if total > self.rank else 0
            rows_max = (total + self.world - 1) // self.world  # symmetric allocations have one size on all ranks
            tabs = {}
            for kind, width, fan_in in (("mlp", d, total), ("gmf", self.f, total)):
                if width == 0:
                    tabs[kind] = None
                    continue
                lim = (6.0 / (fan_in + width)) ** 0.5  # glorot-uniform of the FULL table (model.py:163)
                if peer_gather:
                    t = symm.empty((max(rows_max, 1), width), dtype=torch.float32, device=dev)
                else:
                    t = torch.empty((max(rows_max, 1), width), dtype=torch.float32, device=dev)
                if seed is None:
                    t.uniform_(-lim, lim)
                else:
                    t.copy_(torch.from_numpy(rng.uniform(-lim, lim, size=tuple(t.shape)).astype("float32")))
                tabs[kind] = {"p": t, "m": torch.zeros(t.shape, dtype=torch.float32, device=dev),
                              "v": torch.zeros(t.shape, dtype=torch.float32, device=dev)}
                if peer_gather:
                    hdl = symm.rendezvous(t, pg_name)
                    tabs[kind]["handle"] = hdl
                    tabs[kind]["peers"] = torch.tensor(list(hdl.buffer_ptrs), dtype=torch.int64, device=dev)
                    if self._barrier_handle is None:
                        self._barrier_handle = hdl
            self.shard[side] = {"rows": rows, "tabs": tabs, "d": d, "total": total}
        self._ws = None

    # ---- helpers --------------------------------------------------------------------------------------
    def _a2a(self, send, send_counts, recv_counts, width=None):
        shape = (sum(recv_counts),) if width is None else (sum(recv_counts), width)
        recv = torch.empty(shape, dtype=send.dtype, device=send.device)
        dist.all_to_all_single(recv, send.contiguous(), output_split_sizes=list(recv_counts),
                               input_split_sizes=list(send_counts), group=self.group)
        return recv

    def _route(self, ids):
        """Unique ids of the batch grouped by owner -> (cache slot of every batch row, unique ids in send
        order, send counts, ids requested from this rank, their counts)."""
        uniq, inv = torch.unique(ids, return_inverse=True)
        owner = uniq % self.world
        perm = torch.argsort(owner, stable=True)
        uniq_s = uniq[perm]
        slot_of_unique = torch.empty_like(perm)
        slot_of_unique[perm] = torch.arange(perm.numel(), device=perm.device)
        slots = slot_of_unique[inv].to(torch.int32)
        send_counts = torch.bincount(owner, minlength=self.world)
        recv_counts = torch.empty_like(send_counts)
        dist.all_to_all_single(recv_counts, send_counts, group=self.group)
        sc, rc = send_counts.tolist(), recv_counts.tolist()
        wanted = self._a2a(uniq_s.to(torch.int32), sc, rc)
        return slots, uniq_s, sc, wanted, rc

    def _fetch(self, side, ids):
        """Steps 1-2 for one side: fills the cache tables, returns the routing for the way back."""
        e = self.cache
        slots, uniq_s, sc, wanted, rc = self._route(ids)
        n_u = int(uniq_s.numel())
        if n_u > self.capacity:
            raise ValueError("batch touches {} distinct {} rows, more than max_local_rows={}".format(n_u, side, self.capacity))
        local = torch.div(wanted, self.world, rounding_mode="floor").to(torch.int32)
        tabs = self.shard[side]["tabs"]
        d = self.shard[side]["d"]
        mlp_name = self._engine_mod.K_USER if side == "user" else self._engine_mod.K_ITEM
        gmf_name = self._engine_mod.K_GMF_USER if side == "user" else self._engine_mod.K_GMF_ITEM
        if self.peer_gather:
            # one kernel per table: every needed row straight from its owner's memory into the cache
            import ctypes as C
            nat = self._engine_mod.nat
            ids32 = uniq_s.to(torch.int32)
            for kind, name in (("mlp", mlp_name), ("gmf", gmf_name)):
                if tabs[kind] is None:
                    continue
                t = tabs[kind]
                nat.check(nat.lib.mr_gather_rows_sharded(C.c_void_p(t["peers"].data_ptr()), self.world, self.shard[side]["total"],
                                                         int(t["p"].shape[1]), C.c_void_p(ids32.data_ptr()), n_u,
                                                         C.c_void_p(e._tables[name].data_ptr()), e._stream()),
                          "mr_gather_rows_sharded")
        else:
            parts = [self._engine_mod.gather_rows(tabs[k]["p"], local) for k in ("mlp", "gmf") if tabs[k] is not None]
            rows = self._a2a(torch.cat(parts, dim=1) if len(parts) > 1 else parts[0], rc, sc, width=sum(p.shape[1] for p in parts))
            e._tables[mlp_name][:n_u].copy_(rows[:, :d])
            if self.f:
                e._tables[gmf_name][:n_u].copy_(rows[:, d:])
        return {"slots": slots, "n": n_u, "send_counts": sc, "recv_counts": rc, "local": local}

    def _push_grads(self, side, route):
        """Step 4 for one side: gradient rows of the cache -> owners -> sorted, summed, applied."""
        import ctypes as C
        nat = self._engine_mod.nat
        e = self.cache
        d, n_u = self.shard[side]["d"], route["n"]
        mlp_name = self._engine_mod.K_USER if side == "user" else self._engine_mod.K_ITEM
        parts = [e.g_tables[mlp_name][:n_u]]
        if self.f:
            parts.append(e.g_tables[self._engine_mod.K_GMF_USER if side == "user" else self._engine_mod.K_GMF_ITEM][:n_u])
        send = torch.cat(parts, dim=1) if len(parts) > 1 else parts[0]
        grads = self._a2a(send, route["send_counts"], route["recv_counts"], width=d + self.f)
        n = int(grads.shape[0])
        if n == 0:
            return
        tabs = self.shard[side]["tabs"]
        nbytes = int(nat.lib.mr_sparse_rows_workspace_bytes(n, d, self.f))
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = torch.empty(nbytes, dtype=torch.uint8, device=e.device)
        adam = self.optimizer == "adam"
        ptr = lambda x: C.c_void_p(x.data_ptr()) if x is not None else C.c_void_p(0)
        g = tabs["gmf"]
        nat.check(nat.lib.mr_sparse_rows_update(
            ptr(tabs["mlp"]["p"]), ptr(tabs["mlp"]["m"]), ptr(tabs["mlp"]["v"]), d,
            ptr(g["p"] if g else None), ptr(g["m"] if g else None), ptr(g["v"] if g else None), self.f,
            self.shard[side]["rows"], ptr(route["local"]), ptr(grads), n, nat.OPT_ADAM if adam else nat.OPT_SGD,
            e.lr, e.step_lr_t(), e.beta_1, e.beta_2, self._engine_mod.ADAM_EPSILON,
            ptr(self._ws), self._ws.numel(), e._stream()), "mr_sparse_rows_update")

    # ---- the step ---------------------------------------------------------------------------------------
    def train_step(self, users, items, labels, global_rows, group=0, k=0, grouped=False):
        e = self.cache
        dev = e.device
        users = self._engine_mod.as_device_i32(users, dev).long()
        items = self._engine_mod.as_device_i32(items, dev).long()
        if self.peer_gather:
            self._barrier_handle.barrier()  # every owner has applied the previous step before anyone reads its rows
        ru = self._fetch("user", users)
        ri = self._fetch("item", items)
        out = e.train_grads(ru["slots"], ri["slots"], labels, group=group, k=k, inv_global_batch=1.0 / float(global_rows),
                            grouped=grouped)  # cache slots are a function of the id, so equal users stay equal
        self._push_grads("user", ru)
        self._push_grads("item", ri)
        dist.all_reduce(e.g_dense, op=dist.ReduceOp.SUM, group=self.group)
        e.apply_dense_only()
        return out

    def gather_full_tables(self):
        """All shards reassembled on every rank (tests / small models only): name -> (rows, dim) tensor."""
        out = {}
        m = self._engine_mod
        for side, total in (("user", self.num_users), ("item", self.num_items)):
            for kind, name in (("mlp", m.K_USER if side == "user" else m.K_ITEM),
                               ("gmf", m.K_GMF_USER if side == "user" else m.K_GMF_ITEM)):
                t = self.shard[side]["tabs"][kind]
                if t is None:
                    continue
                full = torch.zeros((total, t["p"].shape[1]), dtype=torch.float32, device=t["p"].device)
                for r in range(self.world):
                    rows = (total - r + self.world - 1) // self.world if total > r else 0
                    buf = t["p"][:rows].clone() if r == self.rank else torch.empty((rows, t["p"].shape[1]), dtype=torch.float32,
                                                                                 device=t["p"].device)
                    dist.broadcast(buf, r, group=self.group)
                    full[r::self.world] = buf
                out[name] = full
        return out

    def load_full_tables(self, weights):
        """Take this rank's rows out of full (rows, dim) arrays keyed by the Keras names; dense block too."""
        import numpy as np
        m = self._engine_mod
        for side in ("user", "item"):
            for kind, name in (("mlp", m.K_USER if side == "user" else m.K_ITEM),
                               ("gmf", m.K_GMF_USER if side == "user" else m.K_GMF_ITEM)):
                t = self.shard[side]["tabs"][kind]
                if t is None:
                    continue
                mine = np.ascontiguousarray(np.asarray(weights[name], dtype=np.float32)[self.rank::self.world])
                t["p"][:mine.shape[0]].copy_(torch.from_numpy(mine))
        e = self.cache
        for name in e._dense_slices:
            e._view(name).copy_(torch.from_numpy(np.ascontiguousarray(np.asarray(weights[name], dtype=np.float32))).view_as(e._view(name)))
