"""Device-side state of one NeuMF model and the calls into libmovierec_b200.so.

PyTorch is used for what the north star allows it for: allocating device memory, owning streams
and (in data-parallel runs) the NCCL process group.  All arithmetic of the hot path happens in the
hand-written CUDA kernels behind the C ABI (`_native`); nothing here computes on tensors except
trivial bookkeeping (views, zero-fill, scalar accumulation of step outputs).
"""

import ctypes as C
import math

import numpy as np
import torch

from . import _native as nat

# Keras weight names of the reference model (model.py:164,169,179,186) + the GMF extension
K_USER = "user_embedding/embeddings"
K_ITEM = "item_embedding/embeddings"
K_GMF_USER = "gmf_user_embedding/embeddings"
K_GMF_ITEM = "gmf_item_embedding/embeddings"
K_OUT_W = "output/kernel"
K_OUT_B = "output/bias"
ADAM_EPSILON = 1e-7  # legacy Keras Adam: epsilon=None -> K.epsilon()


def hidden_names(i):
    return "hidden_{}/kernel".format(i), "hidden_{}/bias".format(i)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("movierec (B200 build) needs a CUDA device: the hot path has no CPU fallback")


def as_device_i32(x, device):
    """ids -> contiguous int32 device tensor (H2D copy is asynchronous when `x` is pinned)."""
    if isinstance(x, torch.Tensor):
        t = x
    else:
        t = torch.from_numpy(np.ascontiguousarray(np.asarray(x).reshape(-1)))
    t = t.reshape(-1)
    if t.dtype != torch.int32:
        t = t.to(torch.int32)
    return t.to(device, non_blocking=True).contiguous()


def as_device_f32(x, device):
    if isinstance(x, torch.Tensor):
        t = x
    else:
        t = torch.from_numpy(np.ascontiguousarray(np.asarray(x).reshape(-1)))
    t = t.reshape(-1)
    if t.dtype != torch.float32:
        t = t.to(torch.float32)
    return t.to(device, non_blocking=True).contiguous()


class NeuMFEngine(object):
    """Parameters, optimizer state, gradient buffers and workspace of one model replica."""

    def __init__(self, num_users, num_items, layers_sizes, layers_l2reg, mf_dim=0, optimizer="adam",
                 lr=1e-3, beta_1=0.9, beta_2=0.999, table_mode="dense", device=None, seed=None,
                 table_state=True, compute_path=None, item_projection=None, fused_train=None):
        """compute_path: 'auto' | 'simt' | 'tc'; item_projection: 'auto' | 'off' | 'on'; fused_train: 'auto' | 'off'
        (include/movierec_b200.h: MrModel.compute_path / item_projection / fused_train).  None = the module defaults
        (`set_compute_path`, `set_item_projection`, `set_fused_train`), which start as 'auto'."""
        require_cuda()
        self.compute_path = _PATHS[compute_path if compute_path is not None else _DEFAULTS["compute_path"]]
        self.item_projection = _PROJECTIONS[item_projection if item_projection is not None else _DEFAULTS["item_projection"]]
        self.fused_train = _FUSED[fused_train if fused_train is not None else _DEFAULTS["fused_train"]]
        self.device = torch.device(device if device is not None else "cuda:{}".format(torch.cuda.current_device()))
        self.num_users, self.num_items = int(num_users), int(num_items)
        self.L = [int(x) for x in layers_sizes]
        self.l2 = [float(x) for x in layers_l2reg]
        self.mf_dim = int(mf_dim)
        n = len(self.L)
        if not 1 <= n <= nat.MR_MAX_LAYERS:
            raise ValueError("layers_sizes must have 1..{} entries, found {}".format(nat.MR_MAX_LAYERS, n))
        if self.L[0] < 2 or any(not 1 <= w <= nat.MR_MAX_WIDTH for w in self.L) or not 0 <= self.mf_dim <= nat.MR_MAX_WIDTH:
            raise ValueError("layer widths must be in [1, {}] (first >= 2), found {} mf_dim={}".format(
                nat.MR_MAX_WIDTH, self.L, self.mf_dim))
        self.d_u = self.L[0] // 2               # model.py:159
        self.d_i = self.L[0] - self.d_u         # model.py:160
        self.optimizer = optimizer
        self.lr, self.beta_1, self.beta_2 = float(lr), float(beta_1), float(beta_2)
        self.table_mode = table_mode
        if table_mode not in ("dense", "sparse"):
            raise ValueError("table_mode must be 'dense' or 'sparse', found {!r}".format(table_mode))
        if table_mode == "sparse" and self.l2[0] != 0:
            raise ValueError("layers_l2reg[0] != 0 makes embedding gradients dense; use table_mode='dense'")
        self.iterations = 0

        # dense block layout W1,b1,...,w_out,b_out (include/movierec_b200.h: MrModel)
        self._dense_slices = {}
        off = 0
        for i in range(1, n):
            kn, bn = hidden_names(i)
            self._dense_slices[kn] = (off, (self.L[i - 1], self.L[i]))
            off += self.L[i - 1] * self.L[i]
            self._dense_slices[bn] = (off, (self.L[i],))
            off += self.L[i]
        self._dense_slices[K_OUT_W] = (off, (self.mf_dim + self.L[-1], 1))
        off += self.mf_dim + self.L[-1]
        self._dense_slices[K_OUT_B] = (off, (1,))
        off += 1
        self.dense_count = off

        dev, f32 = self.device, torch.float32
        self.user_mlp = torch.empty((self.num_users, self.d_u), dtype=f32, device=dev)
        self.item_mlp = torch.empty((self.num_items, self.d_i), dtype=f32, device=dev)
        self.user_gmf = torch.empty((self.num_users, self.mf_dim), dtype=f32, device=dev) if self.mf_dim else None
        self.item_gmf = torch.empty((self.num_items, self.mf_dim), dtype=f32, device=dev) if self.mf_dim else None
        self.dense = torch.zeros(self.dense_count, dtype=f32, device=dev)
        self._tables = {K_USER: self.user_mlp, K_ITEM: self.item_mlp}
        if self.mf_dim:
            self._tables[K_GMF_USER] = self.user_gmf
            self._tables[K_GMF_ITEM] = self.item_gmf
        self.initialize(seed)

        adam = optimizer == "adam"
        z = lambda t: torch.zeros_like(t) if (t is not None) else None
        # table_state=False: the tables are a per-step cache of rows owned elsewhere (row-sharded runs);
        # their optimizer state lives with the owner, so none is allocated here and apply() is not used
        self.table_state = bool(table_state)
        self.m = {k: z(t) for k, t in self._tables.items()} if (adam and table_state) else {}
        self.v = {k: z(t) for k, t in self._tables.items()} if (adam and table_state) else {}
        self.m_dense = z(self.dense) if adam else None
        self.v_dense = z(self.dense) if adam else None
        # one flat gradient buffer so that a data-parallel caller all-reduces it in one or two calls: the user tables'
        # gradients first (final early in the projected step: MrGrads.user_tables_ready), then dense + item tables
        order = [k for k in (K_USER, K_GMF_USER) if k in self._tables] + ["dense"] + \
                [k for k in (K_ITEM, K_GMF_ITEM) if k in self._tables]
        if table_mode != "dense":
            order = ["dense"]
        pad = lambda x: (x + 63) // 64 * 64  # keep every slice 256-byte aligned (128-bit kernel accesses)
        numel = lambda k: self.dense_count if k == "dense" else self._tables[k].numel()
        self.g_flat = torch.zeros(sum(pad(numel(k)) for k in order), dtype=f32, device=dev)
        self.g_tables = {}
        self._flat_layout = []  # (name, offset, elements) of every region of g_flat, in order
        off = 0
        for k in order:
            if k == "dense":
                self.g_dense = self.g_flat[off:off + self.dense_count]
                self._g_user_end = off  # [0, _g_user_end): the user tables' gradients
            else:
                self.g_tables[k] = self.g_flat[off:off + numel(k)].view_as(self._tables[k])
            self._flat_layout.append((k, off, numel(k)))
            off += pad(numel(k))
        self.p_flat = self.m_flat = self.v_flat = None  # set by rebind_flat()
        self.step_out = torch.zeros(nat.MR_STEP_OUT_FLOATS, dtype=f32, device=dev)
        self._ws = None
        self._structs()

    # ---- parameters --------------------------------------------------------------------------
    def weight_names(self):
        """Keras creation order of the reference model (model.py:161-187), GMF tables last."""
        names = [K_USER, K_ITEM]
        for i in range(1, len(self.L)):
            names.extend(hidden_names(i))
        names.extend([K_OUT_W, K_OUT_B])
        if self.mf_dim:
            names.extend([K_GMF_USER, K_GMF_ITEM])
        return names

    def _view(self, name, base=None):
        if name in self._tables:
            return self._tables[name]
        off, shape = self._dense_slices[name]
        base = self.dense if base is None else base
        return base[off:off + int(np.prod(shape))].view(*shape)

    def initialize(self, seed=None):
        """Initialisers of model.py:163,168,178,186: glorot-uniform tables and hidden kernels,
        lecun-uniform head, zero biases (limits per SURVEY App. A-5)."""
        rng = np.random.default_rng(seed)
        for name in self.weight_names():
            t = self._view(name)
            if name.endswith("bias"):
                t.zero_()
                continue
            if name == K_OUT_W:
                lim = math.sqrt(3.0 / t.shape[0])
            else:
                lim = math.sqrt(6.0 / (t.shape[0] + t.shape[1]))
            t.copy_(torch.from_numpy(rng.uniform(-lim, lim, size=tuple(t.shape)).astype(np.float32)))

    def get_weights(self):
        torch.cuda.current_stream(self.device).synchronize()
        return {k: self._view(k).detach().cpu().numpy().copy() for k in self.weight_names()}

    def set_weights(self, weights):
        """`weights`: dict keyed by Keras names, or a list in `weight_names()` order."""
        if not isinstance(weights, dict):
            weights = dict(zip(self.weight_names(), weights))
        for k in self.weight_names():
            t = self._view(k)
            w = np.asarray(weights[k], dtype=np.float32)
            if tuple(w.shape) != tuple(t.shape):
                raise ValueError("weight {} has shape {}, expected {}".format(k, w.shape, tuple(t.shape)))
            t.copy_(torch.from_numpy(np.ascontiguousarray(w)))

    def get_optimizer_state(self):
        torch.cuda.current_stream(self.device).synchronize()
        st = {"iterations": self.iterations}
        if self.optimizer == "adam":
            for k in self.weight_names():
                st["m/" + k] = (self.m[k] if k in self.m else self._view(k, self.m_dense)).detach().cpu().numpy().copy()
                st["v/" + k] = (self.v[k] if k in self.v else self._view(k, self.v_dense)).detach().cpu().numpy().copy()
        return st

    def set_optimizer_state(self, st):
        self.iterations = int(st["iterations"])
        if self.optimizer == "adam":
            for k in self.weight_names():
                for tag, tabs, dense in (("m/", self.m, self.m_dense), ("v/", self.v, self.v_dense)):
                    dst = tabs[k] if k in tabs else self._view(k, dense)
                    dst.copy_(torch.from_numpy(np.ascontiguousarray(st[tag + k], dtype=np.float32)).view_as(dst))

    def rebind_flat(self, alloc=None):
        """Moves the parameters, the gradients and the optimizer state into flat buffers that share ONE layout (that of
        g_flat: [user tables | dense block | item tables], regions 256-byte aligned), keeping every value, and re-seats
        all views and C structs.  `alloc(numel)` allocates the parameter and the gradient buffer (a data-parallel
        caller passes a symmetric-memory allocator so that peers can address them: DataParallelNeuMF); the optimizer
        state is rank-private.  Element i of p_flat, g_flat, m_flat and v_flat belong together."""
        if self.table_mode != "dense" or not self.table_state:
            raise RuntimeError("rebind_flat needs dense gradient tables and table state on this engine")
        dev, f32 = self.device, torch.float32
        n = self.g_flat.numel()
        alloc = alloc or (lambda count: torch.empty(count, dtype=f32, device=dev))
        adam = self.optimizer == "adam"
        p_flat, g_flat = alloc(n), alloc(n)
        p_flat.zero_()
        g_flat.copy_(self.g_flat)
        m_flat = torch.zeros(n, dtype=f32, device=dev) if adam else None
        v_flat = torch.zeros(n, dtype=f32, device=dev) if adam else None
        for k, off, cnt in self._flat_layout:
            sl = slice(off, off + cnt)
            if k == "dense":
                p_flat[sl].copy_(self.dense)
                if adam:
                    m_flat[sl].copy_(self.m_dense)
                    v_flat[sl].copy_(self.v_dense)
                self.dense, self.g_dense = p_flat[sl], g_flat[sl]
                if adam:
                    self.m_dense, self.v_dense = m_flat[sl], v_flat[sl]
            else:
                shape = self._tables[k].shape
                p_flat[sl].copy_(self._tables[k].reshape(-1))
                if adam:
                    m_flat[sl].copy_(self.m[k].reshape(-1))
                    v_flat[sl].copy_(self.v[k].reshape(-1))
                    self.m[k], self.v[k] = m_flat[sl].view(shape), v_flat[sl].view(shape)
                self._tables[k] = p_flat[sl].view(shape)
                self.g_tables[k] = g_flat[sl].view(shape)
        self.user_mlp, self.item_mlp = self._tables[K_USER], self._tables[K_ITEM]
        if self.mf_dim:
            self.user_gmf, self.item_gmf = self._tables[K_GMF_USER], self._tables[K_GMF_ITEM]
        self.p_flat, self.g_flat, self.m_flat, self.v_flat = p_flat, g_flat, m_flat, v_flat
        self._structs()

    def flat_regions(self):
        """[(name, offset, padded elements, l2 coefficient)] of the flat layout: user tables, dense block, item tables."""
        out = []
        for i, (k, off, cnt) in enumerate(self._flat_layout):
            end = self._flat_layout[i + 1][1] if i + 1 < len(self._flat_layout) else self.g_flat.numel()
            out.append((k, off, end - off, 0.0 if k == "dense" else self.l2[0]))
        return out

    def step_lr_t(self):
        """Step size of the NEXT update as mr_neumf_apply computes it (legacy-Keras Adam folds the bias correction in)."""
        f32 = lambda x: float(np.float32(x))  # the C side holds lr and the betas as floats
        if self.optimizer != "adam":
            return f32(self.lr)
        t = self.iterations + 1
        return f32(self.lr) * math.sqrt(1.0 - f32(self.beta_2) ** t) / (1.0 - f32(self.beta_1) ** t)

    # ---- C structs ------------------------------------------------------------------------------
    def _structs(self):
        self._model_struct()
        self._opt_structs()

    def _model_struct(self):
        m = nat.MrModel()
        m.user_mlp, m.item_mlp = self.user_mlp.data_ptr(), self.item_mlp.data_ptr()
        m.user_gmf = self.user_gmf.data_ptr() if self.mf_dim else None
        m.item_gmf = self.item_gmf.data_ptr() if self.mf_dim else None
        base = self.dense.data_ptr()
        m.dense = base
        for i in range(1, len(self.L)):
            kn, bn = hidden_names(i)
            m.W[i] = base + 4 * self._dense_slices[kn][0]
            m.b[i] = base + 4 * self._dense_slices[bn][0]
        m.w_out = base + 4 * self._dense_slices[K_OUT_W][0]
        m.b_out = base + 4 * self._dense_slices[K_OUT_B][0]
        m.dense_count = self.dense_count
        m.num_users, m.num_items = self.num_users, self.num_items
        m.n_layers = len(self.L)
        for i, w in enumerate(self.L):
            m.L[i] = w
            m.l2[i] = self.l2[i]
        m.mf_dim = self.mf_dim
        m.compute_path, m.item_projection, m.fused_train = self.compute_path, self.item_projection, self.fused_train
        self._model = m

    def _opt_structs(self):

        o = nat.MrOptState()
        o.optimizer = nat.OPT_ADAM if self.optimizer == "adam" else nat.OPT_SGD
        o.table_mode = nat.TABLES_DENSE if self.table_mode == "dense" else nat.TABLES_SPARSE
        o.lr, o.beta_1, o.beta_2, o.epsilon = self.lr, self.beta_1, self.beta_2, ADAM_EPSILON
        o.iterations = self.iterations
        if self.optimizer == "adam":
            # without table state the struct still needs non-NULL pointers; the gradient tables stand in
            # (train_grads in dense mode never reads them, and apply() refuses to run -- see apply())
            ms = self.m if self.table_state else self.g_tables
            vs = self.v if self.table_state else self.g_tables
            o.m_user_mlp, o.m_item_mlp = ms[K_USER].data_ptr(), ms[K_ITEM].data_ptr()
            o.v_user_mlp, o.v_item_mlp = vs[K_USER].data_ptr(), vs[K_ITEM].data_ptr()
            if self.mf_dim:
                o.m_user_gmf, o.m_item_gmf = ms[K_GMF_USER].data_ptr(), ms[K_GMF_ITEM].data_ptr()
                o.v_user_gmf, o.v_item_gmf = vs[K_GMF_USER].data_ptr(), vs[K_GMF_ITEM].data_ptr()
            o.m_dense, o.v_dense = self.m_dense.data_ptr(), self.v_dense.data_ptr()
        self._opt = o

        g = nat.MrGrads()
        g.dense = self.g_dense.data_ptr()
        if self.table_mode == "dense":
            g.user_mlp, g.item_mlp = self.g_tables[K_USER].data_ptr(), self.g_tables[K_ITEM].data_ptr()
            if self.mf_dim:
                g.user_gmf, g.item_gmf = self.g_tables[K_GMF_USER].data_ptr(), self.g_tables[K_GMF_ITEM].data_ptr()
        self._grads = g

    def uses_tensor_cores(self):
        return bool(nat.lib.mr_uses_tensor_cores(C.byref(self._model)))

    def uses_item_projection(self, rows):
        """True when a call over `rows` rows computes the item half of the first layer once per item."""
        return bool(nat.lib.mr_uses_item_projection(C.byref(self._model), int(rows)))

    def uses_user_projection(self, rows, group):
        """True when a grouped train step over `rows` rows also computes the user half once per user."""
        return bool(nat.lib.mr_uses_user_projection(C.byref(self._model), int(rows), int(group)))

    def uses_small_tower(self, rows, group):
        """True when a grouped train step takes the default-tower (64-32-16-8 + GMF 8) thread-per-group kernel."""
        return bool(nat.lib.mr_uses_small_tower(C.byref(self._model), int(rows), int(group)))

    def _workspace(self, nbytes):
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
        return self._ws

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def gradient_tensors(self):
        """The flat gradient buffer a data-parallel caller all-reduces between train_grads and apply."""
        return [self.g_flat]

    def gradient_parts(self):
        """(user part, rest) of the flat gradient buffer: the user tables' gradients, which the projected grouped
        step finishes early (see train_grads(user_ready=...)), and everything else.  The user part is empty in
        sparse table mode."""
        return self.g_flat[:self._g_user_end], self.g_flat[self._g_user_end:]

    # ---- hot path ---------------------------------------------------------------------------------
    def forward(self, users, items, user_div=1, labels=None, want_logits=True, want_probs=True):
        """Fused forward (model.py:154-188).  Returns (logits, probs, loss_sum) device tensors
        (each None when not requested)."""
        users = as_device_i32(users, self.device)
        items = as_device_i32(items, self.device)
        B = items.numel()
        if users.numel() * user_div != B:
            raise ValueError("users ({}) x user_div ({}) != items ({})".format(users.numel(), user_div, B))
        logits = torch.empty(B, dtype=torch.float32, device=self.device) if want_logits else None
        probs = torch.empty(B, dtype=torch.float32, device=self.device) if want_probs else None
        lab = as_device_f32(labels, self.device) if labels is not None else None
        loss = torch.zeros(1, dtype=torch.float32, device=self.device) if labels is not None else None
        nbytes = nat.lib.mr_forward_workspace_bytes(C.byref(self._model), B)
        ws = self._workspace(nbytes)
        nat.check(nat.lib.mr_neumf_forward(C.byref(self._model), _ptr(users), _ptr(items), B, user_div, _ptr(logits),
                                           _ptr(probs), _ptr(lab), _ptr(loss), _ptr(ws), ws.numel(), self._stream()),
                  "mr_neumf_forward")
        return logits, probs, loss

    def users_grouped(self, users, group):
        """True when every `group` consecutive entries of `users` are equal (the generator's layout,
        data_pipeline.py:99-150).  One small kernel and a 4-byte read-back."""
        users = as_device_i32(users, self.device)
        if group < 2 or users.numel() % group:
            return False
        flag = torch.zeros(1, dtype=torch.int32, device=self.device)
        nat.check(nat.lib.mr_users_grouped(_ptr(users), users.numel(), int(group), _ptr(flag), self._stream()),
                  "mr_users_grouped")
        return int(flag.item()) == 0

    def _train_args(self, users, items, labels, group, k, inv_global_batch, grouped=False, dense_l2=True):
        users = as_device_i32(users, self.device)
        items = as_device_i32(items, self.device)
        labels = as_device_f32(labels, self.device)
        B = items.numel()
        if users.numel() != B or labels.numel() != B:
            raise ValueError("users/items/labels must have the same length")
        inv = 1.0 / B if inv_global_batch is None else float(inv_global_batch)
        nbytes = nat.lib.mr_train_workspace_bytes(C.byref(self._model), B)
        ws = self._workspace(nbytes)
        self._opt.iterations = self.iterations
        keep = (users, items, labels, ws)
        flags = nat.TRAIN_USERS_GROUPED if (grouped and group > 1) else 0
        if not dense_l2:
            flags |= nat.TRAIN_NO_DENSE_L2
        args = (C.byref(self._model), C.byref(self._opt), C.byref(self._grads), _ptr(users), _ptr(items), _ptr(labels),
                B, int(group), int(k), flags, inv, _ptr(self.step_out), _ptr(ws), ws.numel(), self._stream())
        return args, keep

    def train_step(self, users, items, labels, group=0, k=0, inv_global_batch=None, grouped=False):
        """One optimisation step (Keras train_on_batch).  Returns a copy of the step outputs
        [loss_sum, hit_sum, dcg_sum, l2_penalty, bad_ids, ...] as a device tensor.
        grouped=True states that every `group` consecutive rows share one user (the generator's layout): the
        tensor-core path then does the user-only work once per group.  The statement is verified on the device;
        a violation sets bit 1 of the bad_ids output and makes the step invalid."""
        args, keep = self._train_args(users, items, labels, group, k, inv_global_batch, grouped)
        nat.check(nat.lib.mr_neumf_train_step(*args), "mr_neumf_train_step")
        self.iterations = int(self._opt.iterations)
        return self.step_out.clone()

    def train_grads(self, users, items, labels, group=0, k=0, inv_global_batch=None, grouped=False, dense_l2=True,
                    user_ready=None, user_gmf_ready=None):
        """Gradients only (no update).  dense_l2=False leaves the hidden kernels' 2*l2*W term out of g_dense: a
        data-parallel caller that sums the ranks' gradients lets exactly one rank add it.
        user_ready: a torch.cuda.Event the library records (on one of its streams) as soon as the user tables'
        gradients -- gradient_parts()[0] -- are final; a stream that waits on it may all-reduce them while the rest
        of the call is still running.  user_gmf_ready: the same for the user GMF table alone (MrGrads.user_gmf_ready),
        which is final earlier still."""
        args, keep = self._train_args(users, items, labels, group, k, inv_global_batch, grouped, dense_l2)
        self._grads.user_tables_ready = user_ready.cuda_event if user_ready is not None else None
        self._grads.user_gmf_ready = user_gmf_ready.cuda_event if user_gmf_ready is not None else None
        nat.check(nat.lib.mr_neumf_train_grads(*args), "mr_neumf_train_grads")
        self._grads.user_tables_ready = None
        self._grads.user_gmf_ready = None
        return self.step_out.clone()

    def apply(self):
        if not self.table_state:
            raise RuntimeError("this engine caches rows owned by other ranks; use apply_dense_only()")
        self._opt.iterations = self.iterations
        nat.check(nat.lib.mr_neumf_apply(C.byref(self._model), C.byref(self._opt), C.byref(self._grads), self._stream()),
                  "mr_neumf_apply")
        self.iterations = int(self._opt.iterations)

    # ---- region-wise apply: lets a data-parallel caller overlap the all-reduce of one region with the update of
    # the previous one (the all-reduce is NVLink-bound, the Adam sweep HBM-bound)
    def gradient_regions(self):
        """[(name, gradient tensor)]: the dense block and every gradient table, largest first."""
        regs = [("dense", self.g_dense)] + [(k, self.g_tables[k]) for k in self.g_tables]
        return sorted(regs, key=lambda r: -r[1].numel())

    def apply_region(self, name):
        """The optimizer sweep of mr_neumf_apply for one region (same kernel, same step size); finish_apply()
        advances the step counter once every region is done."""
        if not self.table_state:
            raise RuntimeError("this engine caches rows owned by other ranks; use apply_dense_only()")
        adam = self.optimizer == "adam"
        lr_t = self.step_lr_t()  # adam_lr_t of api.cu: double arithmetic on the float-valued hyper-parameters
        if name == "dense":
            p, g, m, v, l2 = self.dense, self.g_dense, self.m_dense, self.v_dense, 0.0
        else:
            p, g, l2 = self._tables[name], self.g_tables[name], self.l2[0]
            m, v = (self.m[name], self.v[name]) if adam else (None, None)
        nat.check(nat.lib.mr_optimizer_flat(_ptr(p), _ptr(g), _ptr(m), _ptr(v), p.numel(),
                                            nat.OPT_ADAM if adam else nat.OPT_SGD, lr_t, self.beta_1, self.beta_2,
                                            ADAM_EPSILON, l2, self._stream()), "mr_optimizer_flat")

    def finish_apply(self):
        self.iterations += 1

    def adam_lr_t(self, t):
        """Legacy-Keras Adam step size for step t (1-based): lr*sqrt(1-b2^t)/(1-b1^t)."""
        return self.lr * math.sqrt(1.0 - self.beta_2 ** t) / (1.0 - self.beta_1 ** t)

    def apply_dense_only(self):
        """Optimizer update of the dense block alone from g_dense (row-sharded runs: the table rows are
        updated by their owners through mr_sparse_rows_update).  The step size is step_lr_t(), the one mr_neumf_apply
        takes, so the dense block moves exactly as in a single-GPU step."""
        t = self.iterations + 1
        adam = self.optimizer == "adam"
        lr_t = self.step_lr_t()
        nat.check(nat.lib.mr_optimizer_flat(_ptr(self.dense), _ptr(self.g_dense), _ptr(self.m_dense), _ptr(self.v_dense),
                                            self.dense_count, nat.OPT_ADAM if adam else nat.OPT_SGD, lr_t, self.beta_1,
                                            self.beta_2, ADAM_EPSILON, 0.0, self._stream()), "mr_optimizer_flat")
        self.iterations = t

    def rank_eval(self, users_per_group, items, group, k, want_rank=False, want_probs=False, check_ids=False):
        """Score G groups (positive last) and rank them (model.py:336-455).  Returns
        (pos (G,) int32, sums (2,) float [hit_sum, dcg_sum], rank or None, probs or None).
        check_ids: also leave in `self.last_eval_bad` a one-element device tensor, non-zero when a user / item id was out
        of range (the fused kernels rank such a candidate last without a word)."""
        on_host = lambda x: not (isinstance(x, torch.Tensor) and x.is_cuda)
        if on_host(users_per_group) and on_host(items) and not want_rank and not want_probs:
            n = int(users_per_group.numel() if isinstance(users_per_group, torch.Tensor) else np.asarray(users_per_group).size)
            if n * int(group) >= self.EVAL_PIPELINE_MIN_ROWS:
                return self._rank_eval_from_host(users_per_group, items, n, int(group), int(k), check_ids)
        users = as_device_i32(users_per_group, self.device)
        items = as_device_i32(items, self.device)
        G = users.numel()
        if items.numel() != G * group:
            raise ValueError("items ({}) != groups ({}) x group ({})".format(items.numel(), G, group))
        dev = self.device
        pos = torch.empty(G, dtype=torch.int32, device=dev)
        sums = torch.zeros(2, dtype=torch.float32, device=dev)
        rank = torch.empty((G, group), dtype=torch.int32, device=dev) if want_rank else None
        probs = torch.empty(G * group, dtype=torch.float32, device=dev) if want_probs else None
        nbytes = nat.lib.mr_rank_eval_workspace_bytes(C.byref(self._model), G, group)
        ws = self._workspace(nbytes)
        nat.check(nat.lib.mr_rank_eval(C.byref(self._model), _ptr(users), _ptr(items), G, group, int(k), _ptr(rank),
                                       _ptr(pos), _ptr(probs), _ptr(sums), _ptr(ws), ws.numel(), self._stream()),
                  "mr_rank_eval")
        if check_ids:
            self.last_eval_bad = self._ids_out_of_range(users, items)
        return pos, sums, rank, probs

    def catalogue_topk(self, users, k, exclude=None, targets=None, want_scores=False):
        """The k best items of the whole catalogue for each user (RankLayer order over the probabilities), minus the
        user's exclusion list, and the place of a target item among the same candidates (mr_catalogue_topk).
        exclude: None or (rowptr int64, items int32) -- per user id, an ascending item list (host or device).
        Returns device tensors (items (U, k) int32, scores (U, k) float32, pos (U,) int32 or None, sums (2,) float32
        [hit_sum, dcg_sum] or None, scores_full (U, num_items) float32 or None); pos / sums need targets.  Slots beyond
        the number of candidates hold item -1 / score NaN.  Leaves in `self.last_catalogue_bad` a one-element device
        tensor, non-zero when a user or target id was out of range (such a user's rows are -1 / NaN)."""
        dev = self.device
        users = as_device_i32(users, dev)
        U = users.numel()
        k = int(k)
        t = _targets(targets, U, "users", dev)
        rowptr, items, excl_rows = _exclusion(exclude, dev)
        top_items, top_scores, pos, sums = _selection_outputs(U, k, t, dev)
        full = torch.empty((U, self.num_items), dtype=torch.float32, device=dev) if want_scores else None
        ws = self._workspace(_workspace_bytes(nat.lib.mr_catalogue_topk_workspace_bytes(C.byref(self._model), U, k),
                                              "catalogue_topk", U=U, k=k))
        nat.check(nat.lib.mr_catalogue_topk(C.byref(self._model), _ptr(users), U, k, excl_rows, _ptr(rowptr), _ptr(items),
                                            _ptr(t), _ptr(top_items), _ptr(top_scores), _ptr(pos), _ptr(sums), _ptr(full),
                                            _ptr(ws), ws.numel(), self._stream()), "mr_catalogue_topk")
        bad = _outside(users, self.num_users)
        if t is not None:
            bad = bad + _outside(t, self.num_items)
        self.last_catalogue_bad = bad
        return top_items, top_scores, pos, sums, full

    def catalogue_audience(self, items, k, users=None, exclude=None, targets=None, want_scores=False):
        """The k best users for each of `items` (mr_catalogue_audience): descending probability, the lower user id first
        among ties, over a pool -- every user (users None) or the given ids, sorted and de-duplicated here -- minus the
        item's exclusion list.  exclude: None or (rowptr int64, users int32) -- per ITEM id, an ascending user list
        (host or device), typically the item's raters.  targets (M,): one held-out user per item, never excluded.
        Returns device tensors (users (M, k) int32, scores (M, k) float32, pos (M,) int32 or None, sums (2,) float32
        [hit_sum, dcg_sum] or None, scores_full (U, M) float32 or None, the pool (U,) int32 or None when it is every
        user); pos / sums need targets; pos is the target's place among the item's candidates when < k, else k.  Slots
        beyond the number of candidates hold user -1 / score NaN.  Raises ValueError on a malformed exclusion CSR before
        any launch.  Leaves in `self.last_catalogue_bad` a one-element device tensor, non-zero when an item, pool user
        or target id was out of range (such an item's rows are -1 / NaN; such pool users are never candidates)."""
        dev = self.device
        items = as_device_i32(items, dev)
        M = items.numel()
        k = int(k)
        pool = audience_pool(users)
        U = self.num_users if pool is None else int(pool.size)
        d_pool = None if pool is None else torch.from_numpy(pool if pool.size else np.zeros(1, np.int32)).to(dev)
        t = _targets(targets, M, "items", dev)
        rowptr, excl, excl_rows = _exclusion(exclude, dev)
        top_users, top_scores, pos, sums = _selection_outputs(M, k, t, dev)
        full = torch.empty((U, M), dtype=torch.float32, device=dev) if want_scores else None
        ws = self._workspace(_workspace_bytes(nat.lib.mr_catalogue_audience_workspace_bytes(C.byref(self._model), U, M, k),
                                              "catalogue_audience", U=U, M=M, k=k))
        nat.check(nat.lib.mr_catalogue_audience(C.byref(self._model), _ptr(items if M else None), M, k, _ptr(d_pool), U,
                                                excl_rows, _ptr(rowptr), _ptr(excl), _ptr(t), _ptr(top_users),
                                                _ptr(top_scores), _ptr(pos), _ptr(sums), _ptr(full), _ptr(ws), ws.numel(),
                                                self._stream()), "mr_catalogue_audience")
        bad = _outside(items, self.num_items)
        if t is not None:
            bad = bad + _outside(t, self.num_users)
        if pool is not None and pool.size and (pool[0] < 0 or pool[-1] >= self.num_users):
            bad = bad + 1.0
        self.last_catalogue_bad = bad
        return top_users, top_scores, pos, sums, full, (None if pool is None else d_pool[:U])

    def similar(self, ids, k, side="items", exclude=None, excl_ids=None, want_scores=False):
        """The k nearest items (side "items") or users (side "users") to each of `ids` (mr_similar): similarity is the
        mean of two cosines -- of the rows' first-hidden-layer parts E[x] . W1[side rows] and of their GMF parts
        w_out[:mf_dim] * G[x] -- ordered by descending similarity, the lower id first among ties, leaving out the query
        itself and its exclusion list.  exclude: None or (rowptr int64, ids int32) of ascending lists (host or device);
        query j uses list excl_ids[j] (default j).  Returns device tensors (ids (M, k) int32, similarities (M, k)
        float32, scores_full (M, N) float32 or None); slots beyond the number of candidates, and every slot of an
        out-of-range query, hold -1 / NaN.  Raises ValueError on a malformed exclusion CSR or a model without a hidden
        layer and without GMF, before any launch."""
        if side not in ("items", "users"):
            raise ValueError("side must be 'items' or 'users', found {!r}".format(side))
        dev = self.device
        ids = as_device_i32(ids, dev)
        M = ids.numel()
        k = int(k)
        code, N = (nat.SIDE_ITEMS, self.num_items) if side == "items" else (nat.SIDE_USERS, self.num_users)
        rowptr, excl, excl_rows = _exclusion(exclude, dev)
        e_ids = as_device_i32(excl_ids, dev) if excl_ids is not None else None
        if e_ids is not None and e_ids.numel() != M:
            raise ValueError("excl_ids ({}) and ids ({}) differ in length".format(e_ids.numel(), M))
        nbytes = int(nat.lib.mr_similar_workspace_bytes(C.byref(self._model), code, M, k))
        if nbytes == 0:
            raise ValueError("similar: M={} k={} side={}: {}".format(M, k, side, nat.last_error()))
        top_ids = torch.empty((M, k), dtype=torch.int32, device=dev)
        top_scores = torch.empty((M, k), dtype=torch.float32, device=dev)
        full = torch.empty((M, N), dtype=torch.float32, device=dev) if want_scores else None
        ws = self._workspace(nbytes)
        nat.check(nat.lib.mr_similar(C.byref(self._model), code, _ptr(ids if M else None), M, k, _ptr(e_ids), excl_rows,
                                     _ptr(rowptr), _ptr(excl), _ptr(top_ids), _ptr(top_scores), _ptr(full), _ptr(ws),
                                     ws.numel(), self._stream()), "mr_similar")
        return top_ids, top_scores, full

    def rank_lists(self, users, lists, k, targets=None, want_probs=False):
        """Score and rank ragged candidate lists in one call (mr_rank_lists): list u pairs users[u] with
        items[rowptr[u]:rowptr[u + 1]].  lists = (rowptr int64 (U + 1,), items int32 (nnz,)), host or device; targets
        (U,) are positions in the lists.  Returns device tensors (items (U, k) int32, scores (U, k) float32, top_pos
        (U, k) int32 -- positions within the list --, pos (U,) int32 or None, sums (2,) float32 [hit_sum, dcg_sum] or
        None, probs (nnz,) float32 or None); pos / sums need targets.  Order: descending probability, the earlier
        position first among ties; slots beyond a list's length hold -1 / NaN.  Raises ValueError on a malformed
        rowptr before any launch.  Leaves in `self.last_lists_bad` a one-element device tensor, non-zero when a user
        or item id (or a target) was out of range."""
        dev = self.device
        users = as_device_i32(users, dev)
        U = users.numel()
        rowptr, items = check_csr(*lists, "lists", rows=U, device=dev)
        nnz = items.numel()
        k = int(k)
        t = _targets(targets, U, "users", dev)
        top_pos = torch.empty((U, k), dtype=torch.int32, device=dev)
        top_items, top_scores, pos, sums = _selection_outputs(U, k, t, dev)
        probs = torch.empty(nnz, dtype=torch.float32, device=dev) if want_probs else None
        ws = self._workspace(_workspace_bytes(nat.lib.mr_rank_lists_workspace_bytes(C.byref(self._model), U, nnz, k),
                                              "rank_lists", U=U, nnz=nnz, k=k))
        nat.check(nat.lib.mr_rank_lists(C.byref(self._model), _ptr(users), U, _ptr(rowptr), _ptr(items), nnz, k, _ptr(t),
                                        _ptr(top_pos), _ptr(top_items), _ptr(top_scores), _ptr(pos), _ptr(sums),
                                        _ptr(probs), _ptr(ws), ws.numel(), self._stream()), "mr_rank_lists")
        bad = _outside(users, self.num_users) + _outside(items, self.num_items)
        if t is not None and U:
            lens = rowptr[1:] - rowptr[:-1]
            bad = bad + ((t < 0) | (t.to(torch.int64) >= lens)).any().to(torch.float32).reshape(1)
        self.last_lists_bad = bad
        return top_items, top_scores, top_pos, pos, sums, probs

    def catalogue_targets(self, users, targets, ks, exclude=None):
        """Place of every held-out item of a user among the whole catalogue (mr_catalogue_targets): user users[u] has
        the ascending target list items[rowptr[u]:rowptr[u + 1]] of targets = (rowptr int64 (U + 1,), items int32),
        host or device, and its candidates are every item not on its exclusion list plus its targets.  exclude: as
        catalogue_topk.  ks: 1 to MR_MAX_CUTOFFS cutoffs >= 1.  Returns device tensors (tpos (nnz,) int32 in list
        order, sums (2 + 5 len(ks),) float32: [users with a target, mrr sum] then per cutoff [hit, precision, recall,
        ndcg, map] sums).  Raises ValueError on a malformed rowptr or bad cutoffs before any launch.  Leaves in
        `self.last_catalogue_bad` a one-element device tensor, non-zero when a user or target id was out of range
        (such targets get position num_items)."""
        dev = self.device
        users = as_device_i32(users, dev)
        U = users.numel()
        rowptr, items = check_csr(*targets, "lists", rows=U, device=dev)
        nnz = items.numel()
        kbuf, n_ks = _cutoffs(ks)
        excl_rowptr, excl_items, excl_rows = _exclusion(exclude, dev)
        tpos = torch.empty(nnz, dtype=torch.int32, device=dev)
        sums = torch.zeros(nat.TGT_CUTOFF0 + nat.TGT_PER_CUTOFF * n_ks, dtype=torch.float32, device=dev)
        ws = self._workspace(_workspace_bytes(nat.lib.mr_catalogue_targets_workspace_bytes(C.byref(self._model), U, nnz),
                                              "catalogue_targets", U=U, nnz=nnz))
        nat.check(nat.lib.mr_catalogue_targets(C.byref(self._model), _ptr(users), U, excl_rows, _ptr(excl_rowptr),
                                               _ptr(excl_items), _ptr(rowptr), _ptr(items if nnz else None), nnz, kbuf,
                                               n_ks, _ptr(tpos if nnz else None), _ptr(sums), _ptr(ws), ws.numel(),
                                               self._stream()), "mr_catalogue_targets")
        self.last_catalogue_bad = _outside(users, self.num_users) + _outside(items, self.num_items)
        return tpos, sums

    def fold_in(self, histories, steps, lr, negs, seed=0, init_users=None, optimizer=None, beta_1=None, beta_2=None):
        """Fold-in of U new users (mr_fold_in_users): the item tables and the dense block stay frozen and only each
        user's MLP and GMF rows are optimised, `steps` times, against the user's history and `negs` sampled negatives
        per positive per step.  histories: (rowptr, items) with ascending lists, host or device, or a list of item
        arrays (sorted and de-duplicated here).  init_users (U,): the row of this model a user starts from, -1 = zero
        rows (default: all zero).  optimizer / beta_1 / beta_2 default to the engine's.  Returns device tensors
        (user_mlp (U, d_u), user_gmf (U, mf_dim) or None, loss (U,): the mean BCE of each user's last step before its
        update, NaN for steps = 0 or an empty history).  Raises IndexError on an item or init user out of range and
        ValueError on a malformed CSR or a history that covers every item, before any launch."""
        return self._fold_in("users", histories, steps, lr, negs, seed, init_users, optimizer, beta_1, beta_2)

    def fold_in_items(self, raters, steps, lr, negs, seed=0, init_items=None, optimizer=None, beta_1=None, beta_2=None):
        """Fold-in of M new items (mr_fold_in_items): fold_in with the sides swapped.  The user tables and the dense
        block stay frozen and only each item's MLP and GMF rows are optimised against the item's raters and `negs`
        sampled negative users per rater per step.  raters: (rowptr, users) with ascending lists, host or device, or a
        list of user arrays (sorted and de-duplicated here).  init_items (M,): the row of this model an item starts
        from, -1 = zero rows (default: all zero).  Returns device tensors (item_mlp (M, d_i), item_gmf (M, mf_dim) or
        None, loss (M,)); item_view serves them.  Raises IndexError on a user or init item out of range and ValueError
        on a malformed CSR or a rater list that covers every user, before any launch."""
        return self._fold_in("items", raters, steps, lr, negs, seed, init_items, optimizer, beta_1, beta_2)

    def _fold_in(self, side, lists, steps, lr, negs, seed, init_rows, optimizer, beta_1, beta_2):
        items = side == "items"
        dev = self.device
        num_self, num_other = (self.num_items, self.num_users) if items else (self.num_users, self.num_items)
        rowptr, ids = fold_in_histories(lists, num_other, side)
        U, nnz = rowptr.size - 1, ids.size
        init = None
        if init_rows is not None:
            init = np.asarray(init_rows.cpu() if hasattr(init_rows, "cpu") else init_rows, np.int64).reshape(-1)
            init_name, what, lists_name = ("init_items", "an item", "raters") if items else \
                ("init_users", "a user", "histories")
            if init.size != U:
                raise ValueError("{} ({}) and {} ({}) differ in length".format(init_name, init.size, lists_name, U))
            if init.size and (init.min() < -1 or init.max() >= num_self):
                raise IndexError("{}: {} lies outside [-1, {})".format(init_name, what, num_self))
        optimizer = self.optimizer if optimizer is None else optimizer
        if optimizer not in ("adam", "sgd"):
            raise ValueError("optimizer must be 'adam' or 'sgd', found {!r}".format(optimizer))
        cfg = nat.MrFoldIn()
        cfg.steps, cfg.negs = int(steps), int(negs)
        cfg.optimizer = nat.OPT_ADAM if optimizer == "adam" else nat.OPT_SGD
        cfg.lr = float(lr)
        cfg.beta_1 = float(self.beta_1 if beta_1 is None else beta_1)
        cfg.beta_2 = float(self.beta_2 if beta_2 is None else beta_2)
        cfg.epsilon = ADAM_EPSILON
        cfg.seed = int(seed) & (2 ** 64 - 1)
        d_rowptr = torch.from_numpy(rowptr).to(dev)
        d_ids = torch.from_numpy(ids if nnz else np.zeros(1, np.int32)).to(dev)
        d_init = torch.from_numpy(init.astype(np.int32)).to(dev) if init is not None and U else None
        f32 = torch.float32
        out_mlp = torch.empty((U, self.d_i if items else self.d_u), dtype=f32, device=dev)
        out_gmf = torch.empty((U, self.mf_dim), dtype=f32, device=dev) if self.mf_dim else None
        loss = torch.empty(U, dtype=f32, device=dev)
        name = "mr_fold_in_items" if items else "mr_fold_in_users"
        query = nat.lib.mr_fold_in_items_workspace_bytes if items else nat.lib.mr_fold_in_workspace_bytes
        nbytes = int(query(C.byref(self._model), U, nnz))
        ws = self._workspace(max(nbytes, 256))
        nat.check(getattr(nat.lib, name)(C.byref(self._model), _ptr(d_rowptr), _ptr(d_ids), U, nnz, _ptr(d_init),
                                         C.byref(cfg), _ptr(out_mlp), _ptr(out_gmf), _ptr(loss), _ptr(ws), ws.numel(),
                                         self._stream()), name)
        return out_mlp, out_gmf, loss

    def user_view(self, user_mlp, user_gmf=None):
        """An engine whose users are the rows of user_mlp (U, d_u) / user_gmf (U, mf_dim) -- typically fold_in's
        output -- and which shares this engine's item tables and dense block (not copies: later updates of this
        engine show through).  Every scoring and evaluation call works on it with user id u = row u; training it,
        changing its weights or reading optimizer state raises."""
        return UserViewEngine(self, user_mlp, user_gmf)

    def item_view(self, item_mlp, item_gmf=None):
        """An engine whose catalogue is [this engine's items; the rows of item_mlp (M, d_i) / item_gmf (M, mf_dim)] --
        typically fold_in_items' output -- with new item j at id num_items + j.  It shares this engine's user tables
        and dense block by reference (later updates of this engine show through), but its item tables are a
        concatenated COPY: later updates of this engine's item rows do not.  Every scoring and evaluation call works
        on it, and so do fold_in (a new user's history may hold new items), user_view and item_view; training it,
        changing its weights or reading optimizer state raises."""
        return ItemViewEngine(self, item_mlp, item_gmf)

    def _ids_out_of_range(self, users, items):
        if users.numel() == 0:
            return torch.zeros(1, dtype=torch.float32, device=self.device)
        return torch.maximum(_outside(users, self.num_users), _outside(items, self.num_items))


    # A sweep over host arrays of at least this many rows is cut into chunks whose uploads run on a copy stream under
    # the previous chunk's kernels (the ML-20M sweep uploads 55 MB of candidate ids: 1.5-2 ms next to 4.2 ms of compute)
    EVAL_PIPELINE_MIN_ROWS = 1 << 21
    EVAL_PIPELINE_CHUNKS = 4

    def _rank_eval_from_host(self, users, items, G, group, k, check_ids=False):
        """rank_eval for host inputs (pinned tensors make the copies asynchronous): chunk c + 1 is uploaded while chunk c
        is scored and ranked; positions land in one (G,) tensor, the chunks' metric sums are added in chunk order."""
        def host_i32(x):
            t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(np.asarray(x).reshape(-1)))
            t = t.reshape(-1)
            return t if t.dtype == torch.int32 else t.to(torch.int32)
        users, items = host_i32(users), host_i32(items)
        if items.numel() != G * group:
            raise ValueError("items ({}) != groups ({}) x group ({})".format(items.numel(), G, group))
        dev = self.device
        nch = self.EVAL_PIPELINE_CHUNKS
        per = ((G + nch - 1) // nch + 31) // 32 * 32  # chunk starts stay 128-byte aligned
        bounds = [(lo, min(G, lo + per)) for lo in range(0, G, per)]
        d_users = torch.empty(G, dtype=torch.int32, device=dev)
        d_items = torch.empty(G * group, dtype=torch.int32, device=dev)
        pos = torch.empty(G, dtype=torch.int32, device=dev)
        sums = torch.zeros((len(bounds), 2), dtype=torch.float32, device=dev)
        ws = self._workspace(nat.lib.mr_rank_eval_workspace_bytes(C.byref(self._model), per, group))
        if getattr(self, "_eval_copy_stream", None) is None:
            self._eval_copy_stream = torch.cuda.Stream(device=dev)
        main = torch.cuda.current_stream(dev)
        copy = self._eval_copy_stream
        copy.wait_stream(main)  # (the id buffers were allocated on the main stream)
        ready = []
        with torch.cuda.stream(copy):
            for lo, hi in bounds:
                d_users[lo:hi].copy_(users[lo:hi], non_blocking=True)
                d_items[lo * group:hi * group].copy_(items[lo * group:hi * group], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy)
                ready.append(ev)
        for c, (lo, hi) in enumerate(bounds):
            main.wait_event(ready[c])
            nat.check(nat.lib.mr_rank_eval(C.byref(self._model), _ptr(d_users[lo:hi]), _ptr(d_items[lo * group:hi * group]),
                                           hi - lo, group, k, None, _ptr(pos[lo:hi]), None, _ptr(sums[c]), _ptr(ws),
                                           ws.numel(), self._stream()), "mr_rank_eval")
        d_users.record_stream(copy)
        d_items.record_stream(copy)
        if check_ids:
            self.last_eval_bad = self._ids_out_of_range(d_users, d_items)
        return pos, sums.sum(dim=0), None, None


class _ScoringView(NeuMFEngine):
    """An engine made of another engine's tables with one side replaced or extended: scoring and fold-in only."""

    def _view_rows(self, base, mlp, gmf, d, what, rows):
        self.__dict__.update({k: v for k, v in base.__dict__.items() if k in _VIEW_DESC})
        f32 = torch.float32
        mlp = mlp.to(self.device, f32).contiguous()
        if mlp.dim() != 2 or mlp.shape[1] != d or mlp.shape[0] < 1:
            raise ValueError("{}_mlp must be ({} >= 1, {}), got {}".format(what, rows, d, tuple(mlp.shape)))
        if self.mf_dim:
            if gmf is None:
                raise ValueError("the model has a GMF branch: {}_gmf ({}, {}) is required".format(what, rows, self.mf_dim))
            gmf = gmf.to(self.device, f32).contiguous()
            if tuple(gmf.shape) != (mlp.shape[0], self.mf_dim):
                raise ValueError("{}_gmf must be ({}, {}), got {}".format(what, mlp.shape[0], self.mf_dim,
                                                                         tuple(gmf.shape)))
        else:
            gmf = None
        return mlp, gmf

    def _set_tables(self, base):
        self._tables = dict(base._tables)
        self._tables[K_USER], self._tables[K_ITEM] = self.user_mlp, self.item_mlp
        if self.mf_dim:
            self._tables[K_GMF_USER], self._tables[K_GMF_ITEM] = self.user_gmf, self.item_gmf
        self._ws = None
        self._model_struct()

    def _scoring_only(self, *args, **kwargs):
        raise RuntimeError("a {} view only scores: train, update or save the model it was made from".format(self._side))

    train_step = train_grads = apply = apply_region = finish_apply = apply_dense_only = _scoring_only
    set_weights = initialize = get_optimizer_state = set_optimizer_state = rebind_flat = _scoring_only
    gradient_tensors = gradient_parts = gradient_regions = _scoring_only


class UserViewEngine(_ScoringView):
    """NeuMFEngine.user_view: other user tables in front of a model's item tables and dense block.  Scoring only."""
    _side = "user"

    def __init__(self, base, user_mlp, user_gmf=None):
        self.user_mlp, self.user_gmf = self._view_rows(base, user_mlp, user_gmf, base.d_u, "user", "U")
        self.num_users = int(self.user_mlp.shape[0])
        self.num_items, self.item_mlp, self.item_gmf = base.num_items, base.item_mlp, base.item_gmf
        self._set_tables(base)


class ItemViewEngine(_ScoringView):
    """NeuMFEngine.item_view: a model's user tables and dense block in front of its item tables extended by new rows
    (a concatenated copy).  Scoring and fold-in only."""
    _side = "item"

    def __init__(self, base, item_mlp, item_gmf=None):
        new_mlp, new_gmf = self._view_rows(base, item_mlp, item_gmf, base.d_i, "item", "M")
        self.num_users, self.user_mlp, self.user_gmf = base.num_users, base.user_mlp, base.user_gmf
        self.num_items = base.num_items + int(new_mlp.shape[0])
        self.item_mlp = torch.cat([base.item_mlp, new_mlp])
        self.item_gmf = torch.cat([base.item_gmf, new_gmf]) if self.mf_dim else None
        self._set_tables(base)


# what a view takes from its base engine by value: the model description and the dense block (by reference)
_VIEW_DESC = ("compute_path", "item_projection", "fused_train", "device", "L", "l2", "mf_dim", "d_u", "d_i",
              "optimizer", "lr", "beta_1", "beta_2", "table_mode", "iterations", "_dense_slices", "dense_count", "dense")


_LIST_WORDS = {"users": ("histories", "an item", "a history covers every item"),
               "items": ("raters", "a user", "a rater list covers every user")}


def fold_in_histories(histories, num_other, side="users"):
    """Lists of fold_in (side "users": histories of items) or fold_in_items (side "items": rater lists of users) ->
    host (rowptr int64 (U + 1,), ids int32).  (rowptr, ids) with ascending lists (host or device tensors or arrays) is
    checked as is; a list of id arrays is sorted and de-duplicated per list.  num_other: the number of items (users)
    the ids index.  Raises IndexError on an id outside [0, num_other) and ValueError on a malformed rowptr, a list that
    is not strictly ascending or a list that covers every id."""
    name, id_name, covers = _LIST_WORDS[side]
    host = lambda x: np.asarray(x.cpu() if hasattr(x, "cpu") else x)
    if isinstance(histories, tuple) and len(histories) == 2:
        rowptr = host(histories[0]).astype(np.int64).reshape(-1)
        items = host(histories[1]).astype(np.int64).reshape(-1)
    else:
        parts = [np.unique(host(h).astype(np.int64).reshape(-1)) for h in histories]
        rowptr = np.zeros(len(parts) + 1, np.int64)
        rowptr[1:] = np.cumsum([p.size for p in parts])
        items = np.concatenate(parts) if parts else np.zeros(0, np.int64)
    rowptr, items = (t.numpy() for t in check_csr(rowptr, items, name, ascending=True, limit=num_other, id_name=id_name))
    if np.any(rowptr[1:] - rowptr[:-1] >= num_other):
        raise ValueError("{}: {}, so there is no negative to draw".format(name, covers))
    return rowptr, items


# Kernel selection is part of the model description handed to the library (MrModel), not library state.  These
# module-level defaults only decide what an engine constructed WITHOUT explicit arguments asks for.
_PATHS = {"auto": 0, "simt": 1, "tc": 2}
_PROJECTIONS = {"auto": 0, "off": 1, "on": 2}
_FUSED = {"auto": 0, "off": 1}
_DEFAULTS = {"compute_path": "auto", "item_projection": "auto", "fused_train": "auto"}


def set_compute_path(path):
    """Default for engines constructed from now on: 'auto' (tensor cores where the layer widths allow, else the SIMT
    kernel), 'simt' or 'tc'."""
    _PATHS[path]
    _DEFAULTS["compute_path"] = path


def set_item_projection(mode):
    """Default for engines constructed from now on.  Item half of the first layer once per item instead of once per
    row: 'auto' (when a call has at least twice as many rows as there are items), 'off' or 'on' (wherever the model is
    eligible)."""
    _PROJECTIONS[mode]
    _DEFAULTS["item_projection"] = mode


def set_fused_train(mode):
    """Default for engines constructed from now on: 'auto' (the fused per-tile train kernel wherever it applies) or
    'off' (the kernel-per-layer launch sequence)."""
    _FUSED[mode]
    _DEFAULTS["fused_train"] = mode


def rank_scores(scores, group, k, label_col=None, want_rank=True, device=None, labels=None):
    """RankLayer + metrics on caller-supplied scores (model.py:336-455), on device.  The label column of a group is
    label_col[g], else the argmax of the group's `labels` (model.py:447-448), else the last column."""
    require_cuda()
    device = torch.device(device if device is not None else "cuda:{}".format(torch.cuda.current_device()))
    s = as_device_f32(scores, device)
    if group < 1 or s.numel() % group:
        raise ValueError("scores ({}) not divisible by group width {}".format(s.numel(), group))
    G = s.numel() // group
    pos = torch.empty(G, dtype=torch.int32, device=device)
    sums = torch.zeros(2, dtype=torch.float32, device=device)
    rank = torch.empty((G, group), dtype=torch.int32, device=device) if want_rank else None
    lc = as_device_i32(label_col, device) if label_col is not None else None
    lab = as_device_f32(labels, device) if labels is not None else None
    if lab is not None and lab.numel() != s.numel():
        raise ValueError("labels ({}) and scores ({}) differ in length".format(lab.numel(), s.numel()))
    nbytes = max(int(nat.lib.mr_rank_scores_workspace_bytes(G)), 256)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
    st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
    nat.check(nat.lib.mr_rank_scores(_ptr(s), G, int(group), int(k), _ptr(lc), _ptr(lab), _ptr(rank), _ptr(pos), _ptr(sums),
                                     _ptr(ws), nbytes, st), "mr_rank_scores")
    return rank, pos, sums


def topk_scores(scores, k, exclude=None, excl_ids=None, targets=None, device=None):
    """Top-k of each row of a (U, N) score matrix in the RankLayer order, minus the row's exclusion list
    (mr_topk_scores).  exclude: None or (rowptr int64, items int32); row u uses list excl_ids[u] (default u).
    Returns device tensors (items (U, k) int32, scores (U, k) float32, pos (U,) int32 or None, sums (2,) or None)."""
    require_cuda()
    device = torch.device(device if device is not None else "cuda:{}".format(torch.cuda.current_device()))
    s = scores if isinstance(scores, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(np.asarray(scores)))
    if s.dim() != 2:
        raise ValueError("scores must be (U, N), got shape {}".format(tuple(s.shape)))
    U, N = int(s.shape[0]), int(s.shape[1])
    s = s.to(device, torch.float32).contiguous()
    k = int(k)
    ids = as_device_i32(excl_ids, device) if excl_ids is not None else None
    t = _targets(targets, U, "rows", device)
    rowptr, items, excl_rows = _exclusion(exclude, device)
    top_items, top_scores, pos, sums = _selection_outputs(U, k, t, device)
    nbytes = _workspace_bytes(nat.lib.mr_topk_scores_workspace_bytes(U, N, k), "topk_scores", U=U, N=N, k=k)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
    st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
    nat.check(nat.lib.mr_topk_scores(_ptr(s), U, N, k, _ptr(ids), excl_rows, _ptr(rowptr), _ptr(items), _ptr(t),
                                     _ptr(top_items), _ptr(top_scores), _ptr(pos), _ptr(sums), _ptr(ws), nbytes, st),
              "mr_topk_scores")
    return top_items, top_scores, pos, sums


def audience_pool(users):
    """The pool of an audience call: None (every user) or ids -> host int32, ascending and de-duplicated."""
    if users is None:
        return None
    u = np.asarray(users.cpu() if hasattr(users, "cpu") else users).reshape(-1).astype(np.int64)
    return np.unique(u).astype(np.int32)


def check_csr(rowptr, ids, what, rows=None, ascending=False, limit=None, id_name="an id", device=None):
    """(rowptr, ids) host or device -> (rowptr int64, ids int32) tensors on `device` (default: rowptr's), checked there
    with one read-back.  ValueError unless rowptr starts at 0, never decreases and ends at len(ids) (and has rows + 1
    entries when rows is given), or when ascending and a list is not strictly ascending; IndexError when limit is given
    and an id lies outside [0, limit).  The kernels read lists as given, so every list argument passes through here."""
    def as_t(x):
        if isinstance(x, torch.Tensor):
            return x.reshape(-1)
        a = np.asarray(x).reshape(-1)
        return torch.from_numpy(np.ascontiguousarray(a if a.dtype.kind in "iu" else a.astype(np.int64)))
    rp = as_t(rowptr)
    device = rp.device if device is None else device
    rp = rp.to(device, torch.int64).contiguous()
    it = as_t(ids).to(device)
    n = it.numel()
    if rp.numel() < 1 or (rows is not None and rp.numel() != rows + 1):
        raise ValueError("{}: rowptr has {} entries, expected {}".format(what, rp.numel(),
                                                                         "at least 1" if rows is None else rows + 1))
    flags = [(rp[0] != 0) | (rp[-1] != n) | (rp[1:] < rp[:-1]).any()]
    no = torch.zeros((), dtype=torch.bool, device=device)
    flags.append(((it < 0) | (it >= limit)).any() if limit is not None else no)
    if ascending and n > 1:
        inner = torch.ones(n - 1, dtype=torch.bool, device=device)  # pairs of neighbours inside one list
        starts = rp[1:-1]
        inner[starts[(starts > 0) & (starts < n)] - 1] = False
        flags.append(((it[1:] <= it[:-1]) & inner).any())
    bad_offsets, bad_ids, *unsorted = torch.stack(flags).tolist()
    if bad_offsets:
        raise ValueError("{}: offsets must start at 0, never decrease and end at len(ids) = {}".format(what, n))
    if bad_ids:
        raise IndexError("{}: {} lies outside [0, {})".format(what, id_name, limit))
    if any(unsorted):
        raise ValueError("{}: every list must be strictly ascending".format(what))
    return rp, it.to(torch.int32).contiguous()


def check_exclusion_csr(rowptr, ids):
    """Exclusion lists (rowptr, ids), host or device -> the same as tensors (int64 rowptr, int32 ids) on their own
    device; ValueError unless rowptr starts at 0, never decreases and ends at len(ids), and every list is strictly
    ascending (check_csr)."""
    return check_csr(rowptr, ids, "exclusion lists", ascending=True)


def _exclusion(exclude, device):
    """None | (rowptr, ids) host or device -> (device rowptr int64 or None, device ids int32 or None, rows): uploaded,
    then checked on the device as check_exclusion_csr, so host lists cost no host pass."""
    if exclude is None:
        return None, None, 0
    rowptr, ids = check_csr(*exclude, "exclusion lists", ascending=True, device=device)
    if ids.numel() == 0:  # every list empty: the library still wants a pointer
        ids = torch.zeros(1, dtype=torch.int32, device=device)
    return rowptr, ids, rowptr.numel() - 1


def _targets(targets, n, what, device):
    """One target per row (or None) -> device int32 (or None); ValueError unless there are n of them."""
    if targets is None:
        return None
    t = as_device_i32(targets, device)
    if t.numel() != n:
        raise ValueError("targets ({}) and {} ({}) differ in length".format(t.numel(), what, n))
    return t


def _selection_outputs(R, k, t, device):
    """The outputs of a top-k over R rows: ids (R, k) int32, scores (R, k) float32, and with targets t pos (R,) int32
    and sums (2,) float32 zeros (else None)."""
    ids = torch.empty((R, k), dtype=torch.int32, device=device)
    scores = torch.empty((R, k), dtype=torch.float32, device=device)
    if t is None:
        return ids, scores, None, None
    return ids, scores, torch.empty(R, dtype=torch.int32, device=device), torch.zeros(2, dtype=torch.float32,
                                                                                      device=device)


def _workspace_bytes(nbytes, what, **sizes):
    """A *_workspace_bytes result; ValueError when the library refuses the sizes (0 bytes)."""
    if int(nbytes) == 0:
        raise ValueError("{}: bad sizes {}".format(what, " ".join("{}={}".format(*kv) for kv in sizes.items())))
    return int(nbytes)


def _outside(t, n):
    """One-element float32 device tensor: 1 when an id of t lies outside [0, n), else 0 (also when t is empty)."""
    if t.numel() == 0:
        return torch.zeros(1, dtype=torch.float32, device=t.device)
    return ((t.min() < 0) | (t.max() >= n)).to(torch.float32).reshape(1)


def audience_scores(scores, k, users=None, exclude=None, excl_ids=None, targets=None, device=None):
    """Audiences on a (U, M) score matrix (mr_audience_scores): for each column j the k best rows, row u being user
    users[u] (default u; strictly ascending), ordered by descending score (NaN last, the lower user id first among
    ties), minus the users of the column's exclusion list.  exclude: None or (rowptr int64, users int32); column j uses
    list excl_ids[j] (default j).  targets (M,): one user per column, never excluded.  Returns device tensors
    (users (M, k) int32, scores (M, k) float32, pos (M,) int32 or None -- clipped at k --, sums (2,) or None).  Raises
    ValueError on a malformed exclusion CSR or a pool that is not strictly ascending."""
    require_cuda()
    device = torch.device(device if device is not None else "cuda:{}".format(torch.cuda.current_device()))
    s = scores if isinstance(scores, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(np.asarray(scores)))
    if s.dim() != 2:
        raise ValueError("scores must be (U, M), got shape {}".format(tuple(s.shape)))
    U, M = int(s.shape[0]), int(s.shape[1])
    s = s.to(device, torch.float32).contiguous()
    k = int(k)
    pool = None
    if users is not None:
        h = np.asarray(users.cpu() if hasattr(users, "cpu") else users).reshape(-1).astype(np.int64)
        if h.size != U or np.any(h[1:] <= h[:-1]):
            raise ValueError("users must hold {} strictly ascending ids".format(U))
        pool = torch.from_numpy(h.astype(np.int32)).to(device)
    ids = as_device_i32(excl_ids, device) if excl_ids is not None else None
    t = _targets(targets, M, "columns", device)
    rowptr, excl, excl_rows = _exclusion(exclude, device)
    top_users, top_scores, pos, sums = _selection_outputs(M, k, t, device)
    nbytes = _workspace_bytes(nat.lib.mr_audience_scores_workspace_bytes(U, M, k), "audience_scores", U=U, M=M, k=k)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
    st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
    nat.check(nat.lib.mr_audience_scores(_ptr(s), U, M, k, _ptr(pool), _ptr(ids), excl_rows, _ptr(rowptr), _ptr(excl),
                                         _ptr(t), _ptr(top_users), _ptr(top_scores), _ptr(pos), _ptr(sums), _ptr(ws),
                                         nbytes, st), "mr_audience_scores")
    return top_users, top_scores, pos, sums


def topk_lists(scores, rowptr, k, targets=None, device=None):
    """Top-k of ragged lists of scores (mr_topk_lists): list u is scores[rowptr[u]:rowptr[u + 1]], ordered by
    descending score (NaN last, the earlier position first among ties).  targets (U,) are positions in the lists.
    Returns device tensors (top_pos (U, k) int32, top_scores (U, k) float32, pos (U,) int32 or None, sums (2,) or
    None); slots beyond a list's length hold -1 / NaN.  Raises ValueError on a malformed rowptr."""
    require_cuda()
    device = torch.device(device if device is not None else "cuda:{}".format(torch.cuda.current_device()))
    s = as_device_f32(scores, device)
    n = (rowptr.numel() if isinstance(rowptr, torch.Tensor) else np.asarray(rowptr).size)
    U = max(int(n) - 1, 0)
    rp, _ = check_csr(rowptr, np.zeros(s.numel(), np.int32), "lists", rows=U, device=device)
    nnz = s.numel()
    k = int(k)
    t = _targets(targets, U, "lists", device)
    top_pos, top_scores, pos, sums = _selection_outputs(U, k, t, device)
    nbytes = _workspace_bytes(nat.lib.mr_topk_lists_workspace_bytes(U, nnz, k), "topk_lists", U=U, nnz=nnz, k=k)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
    st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
    nat.check(nat.lib.mr_topk_lists(_ptr(s), U, _ptr(rp), nnz, k, _ptr(t), _ptr(top_pos), _ptr(top_scores), _ptr(pos),
                                    _ptr(sums), _ptr(ws), nbytes, st), "mr_topk_lists")
    return top_pos, top_scores, pos, sums


def _cutoffs(ks):
    """Cutoffs -> (host int32 array for the C ABI, count); ValueError unless 1..MR_MAX_CUTOFFS values, each >= 1."""
    ks = [int(k) for k in np.asarray(ks).reshape(-1)]
    if not 1 <= len(ks) <= nat.MR_MAX_CUTOFFS or min(ks) < 1:
        raise ValueError("cutoffs must be 1 to {} values >= 1, got {}".format(nat.MR_MAX_CUTOFFS, ks))
    return (C.c_int32 * len(ks))(*ks), len(ks)


def targets_scores(scores, targets, ks, exclude=None, excl_ids=None, device=None):
    """Positions of many targets per row of a (U, N) score matrix (mr_targets_scores): row u's ascending targets are
    items[rowptr[u]:rowptr[u + 1]] of targets = (rowptr, items); candidates are the items not on the row's exclusion
    list (exclude / excl_ids as topk_scores) plus the row's targets; order as topk_scores.  Returns device tensors
    (tpos (nnz,) int32 in list order, sums (2 + 5 len(ks),) float32 laid out as NeuMFEngine.catalogue_targets').
    Raises ValueError on a malformed rowptr or bad cutoffs before any launch."""
    require_cuda()
    device = torch.device(device if device is not None else "cuda:{}".format(torch.cuda.current_device()))
    s = scores if isinstance(scores, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(np.asarray(scores)))
    if s.dim() != 2:
        raise ValueError("scores must be (U, N), got shape {}".format(tuple(s.shape)))
    U, N = int(s.shape[0]), int(s.shape[1])
    s = s.to(device, torch.float32).contiguous()
    rowptr, items = check_csr(*targets, "lists", rows=U, device=device)
    nnz = items.numel()
    kbuf, n_ks = _cutoffs(ks)
    ids = as_device_i32(excl_ids, device) if excl_ids is not None else None
    excl_rowptr, excl_items, excl_rows = _exclusion(exclude, device)
    tpos = torch.empty(nnz, dtype=torch.int32, device=device)
    sums = torch.zeros(nat.TGT_CUTOFF0 + nat.TGT_PER_CUTOFF * n_ks, dtype=torch.float32, device=device)
    nbytes = _workspace_bytes(nat.lib.mr_targets_scores_workspace_bytes(U, N, nnz), "targets_scores", U=U, N=N, nnz=nnz)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
    st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
    nat.check(nat.lib.mr_targets_scores(_ptr(s), U, N, _ptr(ids), excl_rows, _ptr(excl_rowptr), _ptr(excl_items),
                                        _ptr(rowptr), _ptr(items if nnz else None), nnz, kbuf, n_ks,
                                        _ptr(tpos if nnz else None), _ptr(sums), _ptr(ws), nbytes, st),
              "mr_targets_scores")
    return tpos, sums


def gather_rows(table, idx):
    """out[i,:] = table[idx[i],:] through the gather kernel (model.py:161-172)."""
    require_cuda()
    idx = as_device_i32(idx, table.device)
    out = torch.empty((idx.numel(), table.shape[1]), dtype=torch.float32, device=table.device)
    st = C.c_void_p(torch.cuda.current_stream(table.device).cuda_stream)
    nat.check(nat.lib.mr_gather_rows(_ptr(table), table.shape[0], table.shape[1], _ptr(idx), idx.numel(), _ptr(out), st),
              "mr_gather_rows")
    return out


def sort_pairs(keys, key_bits):
    require_cuda()
    device = torch.device("cuda:{}".format(torch.cuda.current_device()))
    keys = as_device_i32(keys, device)
    n = keys.numel()
    out_k, out_i = torch.empty_like(keys), torch.empty_like(keys)
    nbytes = int(nat.lib.mr_sort_workspace_bytes(n))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
    st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
    nat.check(nat.lib.mr_sort_pairs(_ptr(keys), n, int(key_bits), _ptr(out_k), _ptr(out_i), _ptr(ws), nbytes, st),
              "mr_sort_pairs")
    return out_k, out_i


def remap_ids(ids, id_limit=None):
    """Dense ids on the device: returns (dense_ids int32 (n,), unique_ids int32 (distinct,)) with
    unique_ids ascending and unique_ids[dense_ids] == ids (np.unique(ids, return_inverse=True) of the oracle)."""
    require_cuda()
    device = torch.device("cuda:{}".format(torch.cuda.current_device()))
    ids = as_device_i32(ids, device)
    n = ids.numel()
    if id_limit is None:
        id_limit = int(ids.max().item()) + 1 if n else 1
    dense, unique = torch.empty_like(ids), torch.empty(max(n, 1), dtype=torch.int32, device=device)
    count = torch.zeros(1, dtype=torch.int64, device=device)
    flag = torch.zeros(1, dtype=torch.int32, device=device)
    nbytes = max(int(nat.lib.mr_remap_workspace_bytes(n)), 256)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
    st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
    nat.check(nat.lib.mr_remap_ids(_ptr(ids), n, int(id_limit), _ptr(dense), _ptr(unique), _ptr(count), _ptr(flag),
                                   _ptr(ws), nbytes, st), "mr_remap_ids")
    if int(flag.item()):
        raise IndexError("remap_ids: an id lies outside [0, {})".format(id_limit))
    return dense, unique[:int(count.item())]


def split_last_two(users, num_users):
    """Leave-last-two-out split on the device (reference data_pipeline.py:190-198).  users: the user id of every
    rating in file order.  Returns (order, part) device int32 tensors: order = row numbers sorted by user (stable),
    part[e] = 2 / 1 / 0 for the test / validation / train rating at position e of that order."""
    require_cuda()
    device = torch.device("cuda:{}".format(torch.cuda.current_device()))
    users = as_device_i32(users, device)
    n = users.numel()
    order, part = torch.empty_like(users), torch.empty_like(users)
    flag = torch.zeros(1, dtype=torch.int32, device=device)
    nbytes = max(int(nat.lib.mr_split_workspace_bytes(n)), 256)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
    st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
    nat.check(nat.lib.mr_split_last_two(_ptr(users), n, int(num_users), _ptr(order), _ptr(part), _ptr(flag), _ptr(ws),
                                        nbytes, st), "mr_split_last_two")
    if int(flag.item()):
        raise IndexError("split_last_two: a user id lies outside [0, {})".format(num_users))
    return order, part


def build_user_csr(users, items, num_users, num_items):
    """Per-user ascending lists of the distinct items of the (user, item) pairs, built on the device: what the
    negative sampler searches.  Returns (rowptr int64 (num_users + 1,), csr_items int32 (pairs,)) device tensors."""
    require_cuda()
    device = torch.device("cuda:{}".format(torch.cuda.current_device()))
    users, items = as_device_i32(users, device), as_device_i32(items, device)
    n = users.numel()
    if items.numel() != n:
        raise ValueError("users ({}) and items ({}) differ in length".format(n, items.numel()))
    rowptr = torch.empty(int(num_users) + 1, dtype=torch.int64, device=device)
    csr = torch.empty(max(n, 1), dtype=torch.int32, device=device)
    flag = torch.zeros(1, dtype=torch.int32, device=device)
    nbytes = max(int(nat.lib.mr_user_csr_workspace_bytes(n)), 256)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
    st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
    nat.check(nat.lib.mr_build_user_csr(_ptr(users), _ptr(items), n, int(num_users), int(num_items), _ptr(rowptr),
                                        _ptr(csr), _ptr(flag), _ptr(ws), nbytes, st), "mr_build_user_csr")
    if int(flag.item()):
        raise IndexError("build_user_csr: an id lies outside [0, {}) x [0, {})".format(num_users, num_items))
    return rowptr, csr[:int(rowptr[-1].item())]


def sample_negatives(rowptr, csr_items, num_items, pos_users, pos_items, first_index, negs, seed, epoch):
    """Device sampler (data_pipeline.py:99-113, 136-150).  Returns (users, items, labels) device
    tensors of length P*(negs+1) laid out as the reference batches (negatives, then the positive)."""
    require_cuda()
    device = rowptr.device
    pos_users = as_device_i32(pos_users, device)
    pos_items = as_device_i32(pos_items, device)
    P = pos_users.numel()
    n = P * (negs + 1)
    xu = torch.empty(n, dtype=torch.int32, device=device)
    xi = torch.empty(n, dtype=torch.int32, device=device)
    y = torch.empty(n, dtype=torch.float32, device=device)
    st = C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
    nat.check(nat.lib.mr_sample_negatives(_ptr(rowptr), _ptr(csr_items), int(num_items), _ptr(pos_users), _ptr(pos_items),
                                          P, int(first_index), int(negs), int(seed) & (2 ** 64 - 1),
                                          int(epoch) & (2 ** 64 - 1), _ptr(xu), _ptr(xi), _ptr(y), st),
              "mr_sample_negatives")
    return xu, xi, y
