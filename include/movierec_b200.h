/* movierec_b200.h -- C ABI of libmovierec_b200.so: the B200 (sm_100a) NeuMF train / ranking-eval hot
 * path behind the `movierec` Python API of carlamb/MovieRecommender-TF-TRT.
 *
 * The reference has no FFI of its own: its hot path is a Keras graph built in
 * movierec/model.py:135-215 and driven by Model.fit_generator (model.py:329-333); batches come from
 * MovieLensDataGenerator.__getitem__ (data_pipeline.py:115-150).  Each entry point below names the
 * reference code whose work it takes over.  The Python face (movierecommender-tf-trt_b200/movierec)
 * binds these with ctypes; INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller unless marked [host]; the library never
 *    allocates or frees device memory; scratch comes through (ws, ws_bytes) sized by the matching
 *    *_workspace_bytes query (host function, no CUDA work);
 *  - every compute call enqueues on `stream` (a cudaStream_t passed as void*) and returns without
 *    synchronising; results are ordered on that stream;
 *  - return value 0 = MR_OK, negative = error (see MrStatus); mr_last_error() gives a thread-local
 *    message for the last failing call on this thread; there is no global mutable state;
 *  - fp32 row-major everywhere; ids are int32; tables are (rows, dim); dense kernels are (in, out)
 *    exactly as Keras stores them, so weights move to/from the reference without transposes;
 *  - results are deterministic run to run: no floating-point atomics anywhere.
 */
#ifndef MOVIEREC_B200_H_
#define MOVIEREC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MR_VERSION 104     /* major*100 + minor */
#define MR_MAX_LAYERS 8    /* len(layers_sizes) <= 8 (model.py:75) */
#define MR_MAX_WIDTH 1024  /* layers_sizes[i] <= 1024, mf_dim <= 1024 */
#define MR_MAX_NEGS 1023   /* negatives per positive handled by the sampler / rank kernels */
#define MR_MAX_TOPK 256    /* k of the catalogue top-k calls */
#define MR_MAX_CUTOFFS 8   /* cutoffs of one mr_targets_scores / mr_catalogue_targets call */

typedef enum MrStatus {
  MR_OK = 0,
  MR_ERR_INVALID = -1,   /* bad argument (null pointer, size, unsupported dimension) */
  MR_ERR_WORKSPACE = -2, /* ws_bytes smaller than the *_workspace_bytes query */
  MR_ERR_CUDA = -3,      /* a CUDA runtime call or launch failed; message has cudaGetErrorString */
  MR_ERR_NO_DEVICE = -4  /* no sm_100 device is current */
} MrStatus;

typedef enum MrOptimizer { MR_OPT_ADAM = 0, MR_OPT_SGD = 1 } MrOptimizer; /* model.py:36-38 */
typedef enum MrTableMode {
  MR_TABLES_DENSE = 0, /* legacy-Keras semantics: every table row is updated every step (reference) */
  MR_TABLES_SPARSE = 1 /* sparse-row ("lazy") update of the rows touched this step only */
} MrTableMode;

/* The model of MovierecModel.build_mlp_model (model.py:135-195) plus the optional GMF branch
 * (mf_dim > 0; absent from the reference, He et al. 2017).  All dense parameters live in ONE
 * contiguous block `dense` of `dense_count` floats laid out W[1], b[1], ..., W[n-1], b[n-1], w_out,
 * b_out; the individual pointers point into it. */
typedef struct MrModel {
  float* user_mlp; /* (num_users, L[0]/2)            "user_embedding"  model.py:161-165 */
  float* item_mlp; /* (num_items, L[0]-L[0]/2)       "item_embedding"  model.py:166-170 */
  float* user_gmf; /* (num_users, mf_dim) or NULL */
  float* item_gmf; /* (num_items, mf_dim) or NULL */
  float* dense;    /* contiguous block holding everything below */
  float* W[MR_MAX_LAYERS]; /* W[l] (L[l-1], L[l]) for l = 1..n_layers-1  "hidden_l" model.py:176-181 */
  float* b[MR_MAX_LAYERS]; /* b[l] (L[l]) */
  float* w_out;    /* (mf_dim + L[n_layers-1]) GMF block first   "output" model.py:184-187 */
  float* b_out;    /* (1) */
  int64_t dense_count;
  int32_t num_users, num_items;
  int32_t n_layers;         /* len(layers_sizes) >= 1 */
  int32_t L[MR_MAX_LAYERS]; /* layers_sizes */
  int32_t mf_dim;
  float l2[MR_MAX_LAYERS];  /* layers_l2reg: l2[0] on the tables, l2[l] on W[l] (model.py:163,168,178) */
  /* Kernel selection.  Part of the model description -- not library state -- so that the workspace-size queries and
   * every launch on this model agree by construction.  Zero-initialised = automatic. */
  int32_t compute_path;     /* MrComputePath */
  int32_t item_projection;  /* MrProjection */
  int32_t fused_train;      /* MrFusedTrain */
} MrModel;

/* Two implementations of the tower exist: the tcgen05 tensor-core path, used when every layer width is a multiple of
 * 32 (<= 256), every non-final width a multiple of 128 and layers_sizes[0] a multiple of 64, and the fp32 SIMT tile
 * kernel for every other shape.  Both are hand-written CUDA. */
enum { MR_PATH_AUTO = 0, MR_PATH_SIMT = 1, MR_PATH_TENSOR = 2 };
/* Item-projected first layer (tensor-core path; replaces, like the rest of the tower, the Embedding + Dense of
 * model.py:154-181).  The first Dense layer is linear before its ReLU, so its item half E_item . W1[item rows] is
 * computed once per ITEM when a call has at least twice as many rows as there are items (AUTO), and gathered per
 * row; the backward pass sums dZ1 per item before the item half of its GEMMs.  Used by the grouped train step with
 * dense gradient tables and by the fused ranking eval when layers_sizes[1] == layers_sizes[0] / 2 and there are at
 * least three layers.  The train step does the same for the user half when, in addition, there are no more users
 * than the step has groups.  ON = wherever the model is eligible. */
enum { MR_PROJECTION_AUTO = 0, MR_PROJECTION_OFF = 1, MR_PROJECTION_ON = 2 };
/* The fused per-tile train kernel (projected steps of the 256-128-64 / GMF 64 tower in groups of five rows): AUTO =
 * used wherever it applies; OFF = the kernel-per-layer launch sequence (kept for shapes the fused kernel does not
 * cover, and for A/B comparisons in the tests). */
enum { MR_FUSED_AUTO = 0, MR_FUSED_OFF = 1 };

/* Optimizer hyper-parameters and state (model.py:197-204).  m/v mirror MrModel's tables and dense
 * block (NULL for SGD).  `iterations` is the number of steps ALREADY applied (Keras' counter). */
typedef struct MrOptState {
  int32_t optimizer;  /* MrOptimizer */
  int32_t table_mode; /* MrTableMode */
  float lr, beta_1, beta_2, epsilon; /* epsilon = 1e-7 (legacy Keras Adam) */
  int64_t iterations;
  float *m_user_mlp, *m_item_mlp, *m_user_gmf, *m_item_gmf, *m_dense;
  float *v_user_mlp, *v_item_mlp, *v_user_gmf, *v_item_gmf, *v_dense;
} MrOptState;

/* Gradient buffers, caller-owned so that a data-parallel caller can all-reduce them between
 * mr_neumf_train_grads and mr_neumf_apply.  Table gradients are full (rows, dim) tables and are
 * required in MR_TABLES_DENSE mode; in MR_TABLES_SPARSE mode they may be NULL (row gradients are
 * reduced per touched row and applied straight to the tables). */
typedef struct MrGrads {
  float* dense;    /* (dense_count) same layout as MrModel.dense */
  float* user_mlp; /* (num_users, d_u) */
  float* item_mlp;
  float* user_gmf;
  float* item_gmf;
  /* Optional cudaEvent_t (NULL = none), recorded by mr_neumf_train_grads at the point of its launch sequence from
   * which the gradients user_mlp and user_gmf are final AND the call no longer reads the model's user tables -- in
   * the projected grouped step that is well before the call's last kernel, on an internal stream.  A data-parallel
   * caller makes its communication stream wait on it and reduces the user tables' gradients -- and may update the user
   * tables in place (mr_dp_reduce_apply) -- under the rest of the step. */
  void* user_tables_ready;
  /* Optional cudaEvent_t (NULL = none): the same for user_gmf ALONE -- its gradients are final and the call no longer
   * reads the model's user_gmf table -- which in the projected grouped step is earlier still (right after the per-user
   * segment sums, before the first layer's per-user GEMMs).  Recorded no later than user_tables_ready. */
  void* user_gmf_ready;
} MrGrads;

/* `flags` of the train step.  MR_TRAIN_USERS_GROUPED: the caller states that the batch has the layout the
 * reference's generator produces (data_pipeline.py:99-150): `group` consecutive rows (one positive and its
 * negatives) share one user.  The tensor-core path then computes everything that depends on the user row alone
 * once per group (user half of the first layer forward, backward and weight gradient on group-summed
 * gradients, one staged user-gradient row per group).  The statement is verified on the device; a violation
 * sets bit 1 of step_out[MR_OUT_BAD_IDS].  Without the flag no layout is assumed.
 * MR_TRAIN_NO_DENSE_L2: leave the hidden kernels' regulariser term 2*l2[l]*W[l] (model.py:178) out of grads.dense.
 * Data-parallel callers that SUM the ranks' gradients pass it on every rank but one, so that the term is counted
 * once (the tables' term is added by mr_neumf_apply, after the reduction). */
enum { MR_TRAIN_USERS_GROUPED = 1, MR_TRAIN_NO_DENSE_L2 = 2 };

/* Per-step scalars written by the train step (device floats, MR_STEP_OUT_FLOATS of them). */
enum { MR_OUT_LOSS_SUM = 0, /* sum over rows of BCE (model.py:213-215), unscaled */
       MR_OUT_HIT_SUM = 1,  /* sum over groups of hit@k  (model.py:454) */
       MR_OUT_DCG_SUM = 2,  /* sum over groups of ln2/ln(pos+2)*hit (model.py:414-415) */
       MR_OUT_L2_PENALTY = 3, /* sum of l2 regulariser terms (0 when all l2 == 0) */
       MR_OUT_BAD_IDS = 4,  /* bit 0: a user/item id was out of range (row skipped: the step is what it would be
                               with any other out-of-range id there); bit 1: MR_TRAIN_USERS_GROUPED
                               was passed but some row's user differs from its group's first row (step invalid) */
       MR_STEP_OUT_FLOATS = 8 };

int mr_version(void);
const char* mr_last_error(void);
/* Number of SMs of the current device (grid sizing is derived from it); <0 on error. */
int mr_device_sm_count(void);

/* Embedding lookup out[i,:] = table[idx[i],:]  -- replaces Embedding+Flatten (model.py:161-172). */
int mr_gather_rows(const float* table, int64_t rows, int32_t dim, const int32_t* idx, int64_t n,
                   float* out, void* stream);

/* Fused forward: gather -> concat -> Dense/ReLU tower -> GMF product -> head -> sigmoid (-> BCE).
 * Replaces the forward graph of model.py:154-188 and the loss of model.py:213-215.
 * Row r uses users[r / user_div] (user_div = 1 for per-row users; = group width when one user id is
 * given per group) and items[r].  logits/probs/labels/loss_sum may each be NULL.  loss_sum receives
 * the un-averaged BCE sum over the B rows. */
size_t mr_forward_workspace_bytes(const MrModel* model, int64_t B);
int mr_neumf_forward(const MrModel* model, const int32_t* users, const int32_t* items, int64_t B,
                     int32_t user_div, float* logits, float* probs, const float* labels,
                     float* loss_sum, void* ws, size_t ws_bytes, void* stream);

/* One optimisation step = Keras train_on_batch inside fit_generator (model.py:329-333):
 * forward + BCE, analytic backward, deterministic sort + segmented reduction of the embedding row
 * gradients, optimizer update (model.py:197-204), and the train-batch HR@k / DCG@k that the
 * compiled metrics report (model.py:207-215).  `group` = num_negs_per_pos + 1 (0 skips metrics),
 * inv_global_batch = 1 / (rows in the GLOBAL batch) is the gradient scale.  step_out receives
 * MR_STEP_OUT_FLOATS floats.  opt->iterations is advanced on the host copy. */
size_t mr_train_workspace_bytes(const MrModel* model, int64_t B);
int mr_neumf_train_step(MrModel* model, MrOptState* opt, MrGrads* grads, const int32_t* users,
                        const int32_t* items, const float* labels, int64_t B, int32_t group, int32_t k,
                        int32_t flags, float inv_global_batch, float* step_out, void* ws, size_t ws_bytes,
                        void* stream);
/* The two halves of the step, for data-parallel callers that all-reduce `grads` in between
 * (MR_TABLES_DENSE).  In MR_TABLES_SPARSE mode mr_neumf_train_grads already applies the table rows
 * and mr_neumf_apply only updates the dense block. */
int mr_neumf_train_grads(MrModel* model, MrOptState* opt, MrGrads* grads, const int32_t* users,
                         const int32_t* items, const float* labels, int64_t B, int32_t group, int32_t k,
                         int32_t flags, float inv_global_batch, float* step_out, void* ws, size_t ws_bytes,
                         void* stream);
int mr_neumf_apply(MrModel* model, MrOptState* opt, const MrGrads* grads, void* stream);
/* ORs 1 into *flag (a device int the caller zeroed) when some users[r] != users[r - r % group]: the check a
 * caller runs before passing MR_TRAIN_USERS_GROUPED for a batch of unknown origin. */
int mr_users_grouped(const int32_t* users, int64_t n, int32_t group, int32_t* flag, void* stream);

/* Ranking evaluation of G groups (one user, `group` candidate items, the positive LAST -- the
 * generator's layout, data_pipeline.py:113,148): forward scores, position of the positive under
 * the RankLayer order (descending, lower index first among ties; model.py:344-352), hit@k and DCG@k
 * sums (model.py:420-455, 361-417).  Replaces Keras validation (SURVEY 3.4).
 * rank (G*group, full permutation) and probs (G*group) may be NULL; pos (G) is always written.
 * sums receives {hit_sum, dcg_sum}. */
size_t mr_rank_eval_workspace_bytes(const MrModel* model, int64_t G, int32_t group);
int mr_rank_eval(const MrModel* model, const int32_t* users, const int32_t* items, int64_t G,
                 int32_t group, int32_t k, int32_t* rank, int32_t* pos, float* probs, float* sums,
                 void* ws, size_t ws_bytes, void* stream);

/* RankLayer + metrics on caller-supplied scores (model.py:336-455).  The label column of group g is
 * label_col[g] when label_col (G) is given, else the argmax of labels[g*group .. (g+1)*group) (first maximum:
 * K.argmax(y_true), model.py:447-448) when labels (G*group) is given, else the last column (the generator's
 * layout).  rank may be NULL. */
size_t mr_rank_scores_workspace_bytes(int64_t G);
int mr_rank_scores(const float* scores, int64_t G, int32_t group, int32_t k, const int32_t* label_col,
                   const float* labels, int32_t* rank, int32_t* pos, float* sums, void* ws, size_t ws_bytes,
                   void* stream);

/* Top-k selection on caller-supplied scores (the counterpart of mr_rank_scores for whole rows): scores is U x N
 * row-major.  For row u the candidates are the items 0..N-1 minus the exclusion list of row r = excl_ids ? excl_ids[u]
 * : u, i.e. excl_items[excl_rowptr[r] .. excl_rowptr[r+1]), sorted ascending as mr_build_user_csr writes it.  Rows
 * r outside [0, excl_rows), ids outside [0, N) and excl_rowptr == NULL mean "nothing excluded".  Order: the RankLayer
 * order (descending score, NaN as -inf, -0 == +0, the lower item id first among ties).
 * targets (U, may be NULL): the target is never excluded; pos[u] = its 0-based place among the row's candidates (N
 * for a target outside [0, N)); sums = {hit_sum, dcg_sum} over the U targets (hit = pos < k, dcg = ln2/ln(pos+2)*hit).
 * pos and sums need targets.  top_items / top_scores (U x k, each may be NULL): the k best candidates in order;
 * slots beyond the number of candidates hold item -1 and score NaN.  1 <= k <= MR_MAX_TOPK.  Deterministic (the
 * selection compares distinct integer keys).  The workspace does not grow with U beyond one chunk of users. */
size_t mr_topk_scores_workspace_bytes(int64_t U, int32_t N, int32_t k);
int mr_topk_scores(const float* scores, int64_t U, int32_t N, int32_t k, const int32_t* excl_ids, int32_t excl_rows,
                   const int64_t* excl_rowptr, const int32_t* excl_items, const int32_t* targets, int32_t* top_items,
                   float* top_scores, int32_t* pos, float* sums, void* ws, size_t ws_bytes, void* stream);

/* The same for the model's probabilities of every (users[u], item) pair, item = 0..num_items-1: the K best unseen items
 * of the whole catalogue per user, and leave-one-out HR / NDCG against every non-excluded item (no reference
 * counterpart; the reference client scores one user x N candidates, trt_client.py:47-57).  Exclusion lists are indexed
 * by user id.  scores (U x num_items, may be NULL) receives the probabilities.  Users are scored in chunks of about
 * 2^22 rows with the launch sequence mr_rank_eval takes for the model, so a pair's probability is the one
 * mr_rank_eval gives it when both take the same item projection.  An out-of-range user gets -1 / NaN rows and
 * pos = num_items; an out-of-range target gets pos = num_items. */
size_t mr_catalogue_topk_workspace_bytes(const MrModel* model, int64_t U, int32_t k);
int mr_catalogue_topk(const MrModel* model, const int32_t* users, int64_t U, int32_t k, int32_t excl_rows,
                      const int64_t* excl_rowptr, const int32_t* excl_items, const int32_t* targets, int32_t* top_items,
                      float* top_scores, int32_t* pos, float* sums, float* scores, void* ws, size_t ws_bytes,
                      void* stream);

/* Many held-out items per row, ranked against the whole catalogue (a per-user last-20 % or temporal split, all of a
 * user's future ratings): row u's targets are tgt_items[tgt_rowptr[u] .. tgt_rowptr[u+1]) (device tgt_rowptr, U + 1
 * int64; lists strictly ascending, as mr_build_user_csr writes them; every segment is clamped to [0, nnz_t), so a
 * malformed rowptr or an unsorted list never makes a kernel leave its arrays -- that list's results are unspecified).
 * U, nnz_t <= INT32_MAX.  Exclusion lists as mr_topk_scores.  Candidates of row u: every item of [0, N) not excluded,
 * plus every target (a target is never excluded).  Order: mr_topk_scores' (descending score, NaN as -inf, -0 == +0,
 * the lower item id first among ties).
 * tpos (nnz_t int32, list order, may be NULL): the number of candidates ordered before the target -- the other targets
 * count as candidates; N for a target outside [0, N) and for every target of an out-of-range user.  With one target
 * per row this is mr_topk_scores' pos, bit for bit.
 * sums (device floats, may be NULL; not both NULL with tpos): for the rows with n >= 1 targets, sorted positions
 * p_1 <= .. <= p_n, cutoff k, h = #{p_j < k} and gain g(p) = ln2 / ln(p + 2):
 *   hit = [p_1 < k], precision = h / k, recall = h / n, ndcg = sum_{p_j < k} g(p_j) / sum_{i < min(k, n)} g(i),
 *   map = sum_{p_j < k} j / (p_j + 1) / min(k, n) (j 1-based), mrr = 1 / (p_1 + 1) (no cutoff).
 * Targets outside [0, N) count in n; rows with an empty list contribute nothing and are not counted.  Accumulated in
 * double in a fixed order that depends on U alone (never on chunking).  ks [host]: 1 <= n_ks <= MR_MAX_CUTOFFS cutoffs,
 * each >= 1 (k > N allowed).  Layout below: 2 + 5 n_ks floats.
 * Deterministic (integer counts, no float atomics).  No host synchronisation, no read-back.  Workspace: one chunk of
 * rows (4 bytes per row) plus about 24 bytes per target, plus a fixed 43 KB. */
enum { MR_TGT_USERS = 0,      /* rows with at least one target */
       MR_TGT_MRR = 1,        /* sum of 1 / (p_1 + 1) */
       MR_TGT_CUTOFF0 = 2,    /* sums[MR_TGT_CUTOFF0 + MR_TGT_PER_CUTOFF * c + m]: metric m at cutoff ks[c] */
       MR_TGT_HIT = 0, MR_TGT_PRECISION = 1, MR_TGT_RECALL = 2, MR_TGT_NDCG = 3, MR_TGT_MAP = 4,
       MR_TGT_PER_CUTOFF = 5 };
size_t mr_targets_scores_workspace_bytes(int64_t U, int32_t N, int64_t nnz_t);
int mr_targets_scores(const float* scores, int64_t U, int32_t N, const int32_t* excl_ids, int32_t excl_rows,
                      const int64_t* excl_rowptr, const int32_t* excl_items, const int64_t* tgt_rowptr,
                      const int32_t* tgt_items, int64_t nnz_t, const int32_t* ks /*[host]*/, int32_t n_ks,
                      int32_t* tpos, float* sums, void* ws, size_t ws_bytes, void* stream);
/* The same on the model's probabilities of every (users[u], item) pair, scored in chunks exactly as mr_catalogue_topk
 * scores them (so a pair's probability is the same in both calls).  Exclusion lists are indexed by user id. */
size_t mr_catalogue_targets_workspace_bytes(const MrModel* model, int64_t U, int64_t nnz_t);
int mr_catalogue_targets(const MrModel* model, const int32_t* users, int64_t U, int32_t excl_rows,
                         const int64_t* excl_rowptr, const int32_t* excl_items, const int64_t* tgt_rowptr,
                         const int32_t* tgt_items, int64_t nnz_t, const int32_t* ks /*[host]*/, int32_t n_ks,
                         int32_t* tpos, float* sums, void* ws, size_t ws_bytes, void* stream);

/* Top-k of ragged lists of caller-supplied scores: list u is scores[rowptr[u] .. rowptr[u+1]) (device rowptr, U + 1
 * int64, rowptr[0] = 0, non-decreasing, rowptr[U] = nnz; U and nnz <= INT32_MAX, no rows when U = 0).  Order: the
 * RankLayer order (descending score, NaN as -inf, -0 == +0, the EARLIER position in the list first among ties), so pos
 * is exactly mr_rank_scores' position for label_col = target, and with the target last exactly mr_rank_eval's rule
 * (the positive loses ties).  top_pos / top_scores (U x k, each may be NULL): the k best positions within the list,
 * -1 / NaN padding beyond the list's length (an empty list is all padding).  targets (U, may be NULL): a position in
 * the list; pos[u] = the number of candidates ordered before it (the list length for a target outside [0, len));
 * sums = {hit_sum, dcg_sum} over the U lists (hit = pos < k, dcg = ln2/ln(pos+2)*hit).  pos and sums need targets.
 * 1 <= k <= MR_MAX_TOPK.  Deterministic (distinct integer keys).  Every list is clamped to [0, nnz), so a malformed
 * rowptr never makes a kernel read or write outside the arrays; its lists' results are unspecified.
 * Workspace: 8 bytes per list + 4 per list + about 8 k + 4 bytes per 512 rows (staged partial results of the lists
 * longer than 1024, which are cut into <= 32 slices), plus alignment.  No host synchronisation, no read-back. */
size_t mr_topk_lists_workspace_bytes(int64_t U, int64_t nnz, int32_t k);
int mr_topk_lists(const float* scores, int64_t U, const int64_t* rowptr, int64_t nnz, int32_t k, const int32_t* targets,
                  int32_t* top_pos, float* top_scores, int32_t* pos, float* sums, void* ws, size_t ws_bytes, void* stream);

/* The same on the model's probabilities of the pairs (users[u], items[j]), j in list u: batched serving (one request =
 * one user and its own candidate list, of any length; the reference client's one user x ~1000 candidates,
 * trt_client.py:47-57) and ranking evaluation with candidate sets of different sizes.  top_items (U x k) =
 * items[rowptr[u] + top_pos], -1 padding; probs (nnz, may be NULL) receives every pair's probability.  An item may
 * appear more than once in a list: each copy is a separate candidate.  An out-of-range user gives its list -1 / NaN in
 * every slot and pos = the list length; an out-of-range item gets probability NaN and ranks as NaN ranks.
 * The launch sequence is a function of the model alone (never of U or nnz), so a list's outputs do not depend on the
 * other lists of the call: tensor-core towers with an eligible item projection that is not MR_PROJECTION_OFF (>= 3
 * layers, mf_dim 32 / 64 / 128) take the projected sequence of mr_rank_eval (item half once per call, user half once
 * per list); the default tower (mr_uses_small_tower's model, projection and fused kernel not OFF) takes its projected
 * CUDA-core forward with the user half computed for the call's users only; every other model takes mr_neumf_forward.
 * A pair then gets the probability mr_rank_eval gives it when both calls take the projected sequence.  Scoring runs in
 * launches of at most 2^22 rows, so the scoring workspace is bounded by one launch (a few bytes per row) plus, on the
 * projected paths, the item projection (num_items x layers_sizes[1] floats) and one row of layers_sizes[1] floats (the
 * default tower: also layers_sizes[0]/2) per list.  On top of mr_topk_lists' workspace: 8 bytes per row. */
size_t mr_rank_lists_workspace_bytes(const MrModel* model, int64_t U, int64_t nnz, int32_t k);
int mr_rank_lists(const MrModel* model, const int32_t* users, int64_t U, const int64_t* rowptr, const int32_t* items,
                  int64_t nnz, int32_t k, const int32_t* targets, int32_t* top_pos, int32_t* top_items, float* top_scores,
                  int32_t* pos, float* sums, float* probs, void* ws, size_t ws_bytes, void* stream);

/* Fold-in of new users (or of known users whose history has grown): the item tables and the dense block stay frozen
 * and only each user's two embedding rows (MLP, GMF) are optimised against the user's history and sampled negatives --
 * the standard answer for embedding models with no closed-form user solve, and the protocol of "strong generalisation"
 * evaluation.  The results are plain (U, dim) tables: a copy of the MrModel whose user_mlp / user_gmf point at them
 * and whose num_users = U is served and evaluated by every call above, unchanged.
 * Histories: a CSR over the U new users (device rowptr U + 1 int64, rowptr[0] = 0, non-decreasing, rowptr[U] = nnz;
 * device items, each list strictly ascending, ids in [0, num_items), no list covering every item -- the format of the
 * exclusion lists).  init_users (device, U, may be NULL = all -1): the model row user u starts from, -1 = zero rows.
 * The model is never written.  For user u, with list S of n items, and step t = 0 .. steps-1:
 *   1. the positive at position j of S draws `negs` negatives from the items not in S with mr_sample_negatives' rule
 *      (index = j, epoch = t, seed; with fewer candidates than negs, with replacement) -- n (negs + 1) rows;
 *   2. forward and BCE over those rows, loss = their mean;
 *   3. the gradient with respect to u's MLP and GMF rows only, plus 2 l2[0] row;
 *   4. one legacy-Keras Adam step (per-user m and v from zero, step size lr sqrt(1-b2^(t+1)) / (1-b1^(t+1))) or SGD.
 * A user's result depends only on the model, its list, its initial rows and cfg (never on the other users of the call
 * or their order) and is bit-identical run to run: fixed summation orders, no float atomics.
 * out_loss (U, may be NULL): the mean BCE of the last step, before its update; NaN when steps = 0 or the list is
 * empty.  Validation: the sizes and cfg on the host; then one small kernel checks the CSR, the item ids and
 * init_users and the call reads back one word (the only synchronisation) before any other launch -- MR_ERR_INVALID
 * for a malformed rowptr, an unsorted list, an id out of range or a list covering every item.
 * Workspace: the item half of the first layer over the item table (num_items x layers_sizes[1] floats; none without
 * a hidden layer), the transposed dense block and the sort of the users by history length. */
typedef struct MrFoldIn {     /* [host] */
  int32_t steps;              /* optimisation steps per user (0 = return the initial rows) */
  int32_t negs;               /* negatives per positive per step, 1..MR_MAX_NEGS */
  int32_t optimizer;          /* MrOptimizer */
  float lr, beta_1, beta_2, epsilon;
  uint64_t seed;
} MrFoldIn;
size_t mr_fold_in_workspace_bytes(const MrModel* model, int64_t U, int64_t nnz);
int mr_fold_in_users(const MrModel* model, const int64_t* rowptr, const int32_t* items, int64_t U, int64_t nnz,
                     const int32_t* init_users, const MrFoldIn* cfg /*[host]*/, float* out_user_mlp /* (U, L[0]/2) */,
                     float* out_user_gmf /* (U, mf_dim), NULL when mf_dim == 0 */, float* out_loss, void* ws,
                     size_t ws_bytes, void* stream);

/* On-device negative sampler -- replaces _get_random_negatives_and_positive
 * (data_pipeline.py:99-113): for positive p (global index first_index + p, user pos_users[p]) draw
 * `negs` items uniformly from the items NOT in the user's sorted interaction list
 * csr_items[csr_rowptr[u] .. csr_rowptr[u+1]), without replacement unless there are fewer
 * candidates than `negs`, then append the positive.  Counter-based Philox4x32-10 keyed by
 * (seed, epoch, positive index, draw): the output is a pure function of its arguments.
 * Writes out_users (P*(negs+1), user repeated), out_items (negatives then the positive) and
 * out_labels ([0]*negs + [1]); each may be NULL. */
int mr_sample_negatives(const int64_t* csr_rowptr, const int32_t* csr_items, int32_t num_items,
                        const int32_t* pos_users, const int32_t* pos_items, int64_t P,
                        int64_t first_index, int32_t negs, uint64_t seed, uint64_t epoch,
                        int32_t* out_users, int32_t* out_items, float* out_labels, void* stream);

/* Gather from a ROW-SHARDED table over peer pointers: row id lives on rank id % world at local index id / world;
 * shards is a DEVICE array of `world` pointers to the ranks' slices (each (ceil(total_rows/world), dim) fp32 in the
 * owning GPU's memory, mapped into this process through NVLink peer access -- e.g. torch symmetric memory).
 * out[i,:] = row ids[i] (NaN for an out-of-range id).  This one kernel is the gather AND the exchange of the
 * gathered rows of a row-sharded step.  The caller orders it against the owners' updates (a cross-rank barrier).
 * Precondition (not checked): every shard base is 16-byte aligned -- allocation starts are; when dim % 4 == 0 and out
 * is 16-byte aligned the rows are read as float4. */
int mr_gather_rows_sharded(const float* const* shards, int32_t world, int64_t total_rows, int32_t dim,
                           const int32_t* ids, int64_t n, float* out, void* stream);

/* Owner-side update of ROW-SHARDED tables (data-parallel runs whose tables do not fit one GPU): n pairs
 * (local row id, gradient row [g0 | g1]) received from all ranks, duplicates allowed.  The pairs are
 * stably sorted by row id and summed per id by a tree over 32-entry chunks of the sorted list, whose order depends
 * only on the positions of the pairs (deterministic, no atomics); then the sparse-row Adam / SGD update is applied
 * once per id to table0 (num_rows x d0) and table1 (num_rows x d1; d1 may be 0).  Ids outside [0, num_rows) are
 * ignored: no row changes for them, and the other ids' rows are updated exactly as without them.
 * lr_t is Adam's bias-corrected step size lr*sqrt(1-b2^t)/(1-b1^t) for the current step. */
size_t mr_sparse_rows_workspace_bytes(int64_t n, int32_t d0, int32_t d1);
int mr_sparse_rows_update(float* table0, float* m0, float* v0, int32_t d0, float* table1, float* m1, float* v1,
                          int32_t d1, int32_t num_rows, const int32_t* row_ids, const float* grad_rows, int64_t n,
                          int32_t optimizer, float lr, float lr_t, float beta_1, float beta_2, float epsilon,
                          void* ws, size_t ws_bytes, void* stream);

/* Opt-in profiling for benchmarks (thread-local): between mr_profile_begin and mr_profile_end every
 * entry point records CUDA events on the caller's stream at its phase boundaries.  mr_profile_end
 * synchronises on the last event and returns, per phase, the summed device time in ms and the
 * number of intervals, plus the number of kernels this library launched since mr_profile_begin.
 * All three outputs are [host] arrays/scalars; MR_NUM_PHASES entries each for the first two. */
enum { MR_PHASE_TILE_TRAIN = 0, /* fused gather+tower+head+BCE+backward kernel */
       MR_PHASE_MISC = 1,       /* transposes, dense-gradient reduction, loss sum, memsets */
       MR_PHASE_SORT = 2,       /* radix sort of row ids */
       MR_PHASE_SEGREDUCE = 3,  /* segmented reduction + row update */
       MR_PHASE_OPTIMIZER = 4,  /* Adam / SGD sweeps */
       MR_PHASE_TILE_FORWARD = 5, /* fused forward kernel (predict / eval) */
       MR_PHASE_RANK = 6,       /* positions + metric sums */
       MR_PHASE_SAMPLER = 7,
       MR_PHASE_TC_DENSE_FWD = 8,  /* tcgen05 forward layers (gather fused into the first) */
       MR_PHASE_TC_DENSE_BWD = 9,  /* tcgen05 backward-activation layers */
       MR_PHASE_TC_WGRAD = 10,     /* tcgen05 weight-gradient layers */
       MR_PHASE_HEAD = 11,         /* GMF + output unit + BCE (+ their gradients) */
       MR_PHASE_H1_GATHER = 12,    /* item-projected first layer: gather + add + ReLU of the projected rows */
       MR_PHASE_FUSED_TILE = 13,   /* fused per-tile train kernel of the projected tower (tc_fused.cu) */
       MR_NUM_PHASES = 14 };
int mr_profile_begin(void);
int mr_profile_end(float* phase_ms, int64_t* phase_count, int64_t* kernel_launches);

/* Which kernels a call on this model takes (see MrModel.compute_path / item_projection). */
int mr_uses_tensor_cores(const MrModel* model);

int mr_uses_item_projection(const MrModel* model, int64_t rows);
/* The train step does the same for the user half (E_user . W1[user rows] + b1 once per user, per-user sums of the
 * group sums of dZ1) when, in addition, there are no more users than the step has groups. */
int mr_uses_user_projection(const MrModel* model, int64_t rows, int32_t group);
/* 1 when a grouped train step (MR_TRAIN_USERS_GROUPED, dense gradient tables) over `rows` rows in groups of `group` on
 * this model takes the default-tower kernel: the reference's DEFAULT_PARAMS tower 64-32-16-8 (trainer.py) with GMF 8,
 * both halves of the first layer projected over the tables and everything per row in one thread-per-group kernel on
 * CUDA cores (the widths are below the tensor-core tiles).  Same results as the generic kernel up to summation order.
 * MR_PROJECTION_OFF or MR_FUSED_OFF on the model keep the generic kernel. */
int mr_uses_small_tower(const MrModel* model, int64_t rows, int32_t group);

/* Building blocks exposed for tests and for data-parallel callers.  (The tcgen05 self-tests, the descriptor probe
 * and the issue-rate probe are diagnostics: include/movierec_b200_diag.h, libmovierec_b200_diag.so.) */
/* Dataset preparation on the device (SURVEY 8 (f) 2).
 * mr_split_last_two replaces the pandas groupby of load_ratings_train_test_sets (movierec/data_pipeline.py:190-198):
 * order[e] = row number of the e-th rating when the ratings are ordered by user, file order kept inside a user (a
 * stable sort); part[e] = 2 for the last rating of its user (test), 1 for the one before it (validation), 0
 * otherwise (train).  mr_build_user_csr builds what the sampler searches (the per-positive pandas filter of
 * data_pipeline.py:103-112 restated as a table): rowptr [num_users + 1] int64 and, per user, the ascending list of
 * the DISTINCT items of its (user, item) pairs; rowptr[num_users] = number of distinct pairs <= n (csr_items has room
 * for n).  *flag |= 1 when an id lies outside [0, num_users) / [0, num_items): such pairs are left out of the lists,
 * and the split of such input is undefined.  All arrays [device]; flag must be zeroed by the caller. */
/* mr_remap_ids: dense ids for datasets whose ids are sparse or 1-based (the reference keeps the raw MovieLens ids and
 * sizes its tables by constants, movielens_utils.py:51-55; SURVEY App. B-6).  dense_ids[i] = rank of ids[i] among
 * the DISTINCT ids in ascending order, unique_ids[r] = the id of rank r (room for n), *num_unique = their number
 * [device].  Ids outside [0, id_limit) get dense id -1 and raise bit 0 of *flag. */
size_t mr_remap_workspace_bytes(int64_t n);
int mr_remap_ids(const int32_t* ids, int64_t n, int32_t id_limit, int32_t* dense_ids, int32_t* unique_ids,
                 int64_t* num_unique, int32_t* flag, void* ws, size_t ws_bytes, void* stream);
size_t mr_split_workspace_bytes(int64_t n);
int mr_split_last_two(const int32_t* users, int64_t n, int32_t num_users, int32_t* order, int32_t* part, int32_t* flag,
                      void* ws, size_t ws_bytes, void* stream);
size_t mr_user_csr_workspace_bytes(int64_t n);
int mr_build_user_csr(const int32_t* users, const int32_t* items, int64_t n, int32_t num_users, int32_t num_items,
                      int64_t* rowptr, int32_t* csr_items, int32_t* flag, void* ws, size_t ws_bytes, void* stream);
/* Stable LSD radix sort of (key, original index) pairs on the low `key_bits` bits. */
size_t mr_sort_workspace_bytes(int64_t n);
int mr_sort_pairs(const int32_t* keys, int64_t n, int32_t key_bits, int32_t* sorted_keys,
                  int32_t* sorted_index, void* ws, size_t ws_bytes, void* stream);
/* Data-parallel replicas on ONE box (SURVEY 8e): all-reduce(sum) of the gradients + optimizer step + all-gather of the
 * new weights as one kernel over NVLink peer memory.  grad_peers / param_peers are HOST arrays of `world` device
 * pointers: rank r's flat gradient buffer and flat parameter buffer (same layout on every rank, 16-byte aligned,
 * mapped into this process by peer access -- e.g. torch symmetric memory; entry `rank` is this rank's own buffer).
 * world is 1..8 or 16; m and v (Adam) are 16-byte aligned too.  Violations return MR_ERR_INVALID before any launch.
 * For the elements [lo, hi) this rank owns (multiples of 4):
 *     g = grad_peers[0][i] + grad_peers[1][i] + ... (rank order, the same on every rank) + 2*l2*p[i]
 *     Adam / SGD step of mr_optimizer_flat with THIS rank's m[i], v[i] (optimizer state is sharded by owner)
 *     param_peers[r][i] = new value, for every r.
 * grad_multicast / param_multicast (both or neither; NULL = peer loads and stores): NVSwitch multicast addresses of the
 * same two buffers (cuMulticast* / torch symmetric memory's multicast_ptr).  The sum is then one multimem.ld_reduce
 * and the distribution one multimem.st per 16 bytes -- the switch adds and replicates -- which halves the NVLink bytes
 * per rank; the order of the switch's additions is its own, the replicas still end bit-identical.
 * The caller orders the launch against the other ranks with cross-rank barriers: every rank's gradients of the region
 * final and its reads of the region's parameters done before, all owners' launches complete before the parameters
 * are read again.  No reference counterpart (the reference is single-process). */
int mr_dp_reduce_apply(const float* const* grad_peers, float* const* param_peers, int32_t world, int32_t rank,
                       float* m, float* v, int64_t lo, int64_t hi, int32_t optimizer, float lr_t, float beta_1,
                       float beta_2, float epsilon, float l2, const float* grad_multicast, float* param_multicast,
                       void* stream);

/* Elementwise legacy-Keras Adam / SGD over a flat buffer (l2 adds 2*l2*p to the gradient). */
int mr_optimizer_flat(float* p, const float* g, float* m, float* v, int64_t n, int32_t optimizer,
                      float lr_t, float beta_1, float beta_2, float epsilon, float l2, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MOVIEREC_B200_H_ */
