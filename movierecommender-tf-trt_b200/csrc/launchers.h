// Host-side launch functions shared between the .cu files and the C-ABI layer (api.cu).
#pragma once

#include "common.cuh"

namespace mr {

// ---- neumf_kernels.cu ------------------------------------------------------------------------
struct TileLaunch {
  const MrModel* model;
  bool train;
  const float* wt;  // transposed hidden kernels, dense-block layout (train only)
  const int32_t* users;
  const int32_t* items;
  const float* labels;
  int64_t B;
  int32_t user_div;
  float inv_batch;
  float* logits;
  float* probs;
  float* loss_partial;   // (max_tile_ctas())
  float* dense_partial;  // (max_tile_ctas(), dense_stride)
  int64_t dense_stride;
  float* stage_u;
  float* stage_i;
  int32_t* flags;
};
int max_tile_ctas();
int choose_tile_rows(const MrModel& m, bool train);
int launch_neumf_tiles(const TileLaunch& a, cudaStream_t st, int* grid_out);
int launch_transpose_kernels(const MrModel& m, float* wt, cudaStream_t st);
int launch_dense_reduce(const MrModel& m, const float* partial, int64_t stride, int grid_ctas, float* out,
                        cudaStream_t st, bool with_l2 = true);
int launch_sum_partials(const float* partial, int n, float* out, cudaStream_t st);
int launch_l2_penalty(const float* x, int64_t n, float coef, float* out, cudaStream_t st);

// ---- gather.cu -------------------------------------------------------------------------------
int launch_gather_rows(const float* table, int64_t rows, int dim, const int32_t* idx, int64_t n, float* out,
                       cudaStream_t st);

// ---- radix_sort.cu ---------------------------------------------------------------------------
size_t sort_workspace_bytes(int64_t n);
// num_rows >= 0: every key outside [0, num_rows) is replaced by the sentinel num_rows as it is loaded (out_keys then
// holds the sentinel), so an out-of-range id sorts after all valid ids instead of among the valid id that shares its
// low key_bits bits.  key_bits must then cover num_rows itself.
int launch_sort_pairs(const int32_t* keys, int64_t n, int key_bits, int32_t* out_keys, int32_t* out_index,
                      void* ws, size_t ws_bytes, cudaStream_t st, int32_t num_rows = -1);

// ---- segreduce.cu ----------------------------------------------------------------------------
struct RowUpdate {       // what to do with each reduced row gradient
  int mode;              // MrTableMode
  int optimizer;         // MrOptimizer
  float lr_t, beta_1, beta_2, epsilon, lr;
  // two tables share one staged row: columns [0,d0) -> table 0, [d0,d0+d1) -> table 1
  int d0, d1;
  int num_rows;          // rows of both tables; ids outside [0, num_rows) are skipped
  float *p0, *m0, *v0, *g0;  // table / Adam state / dense gradient table (mode DENSE writes g)
  float *p1, *m1, *v1, *g1;
};
size_t segreduce_workspace_bytes(int64_t n, int ld);
int launch_segreduce(const int32_t* sorted_keys, const int32_t* sorted_index, int64_t n, const float* staged,
                     const RowUpdate& u, void* ws, size_t ws_bytes, cudaStream_t st);

// ---- optimizer.cu ----------------------------------------------------------------------------
constexpr int kMaxOptRegions = 5;
struct OptRegions {
  float* p[kMaxOptRegions];
  const float* g[kMaxOptRegions];
  float* m[kMaxOptRegions];
  float* v[kMaxOptRegions];
  int64_t n[kMaxOptRegions];
  float l2[kMaxOptRegions];
  int count;
  int block_start[kMaxOptRegions + 1];
};
// the sweep of launch_optimizer_flat over several buffers in one launch
int launch_optimizer_regions(OptRegions r, int optimizer, float lr_t, float beta_1, float beta_2, float epsilon,
                             cudaStream_t st);
int launch_optimizer_flat(float* p, const float* g, float* m, float* v, int64_t n, int optimizer, float lr_t,
                          float beta_1, float beta_2, float epsilon, float l2, cudaStream_t st);

// ---- rank.cu ---------------------------------------------------------------------------------
size_t rank_partials_count(int64_t G);
// label column of group g: label_col[g], else argmax of labels[g * group ..] (labels != NULL), else the last column
int launch_rank_scores(const float* scores, int64_t G, int group, int k, const int32_t* label_col, int32_t* rank,
                       int32_t* pos, float* sums, float* partials, cudaStream_t st, const float* labels = nullptr);

// ---- topk.cu: top-k selection over rows of scores with per-row exclusion lists ------------------------------
struct TopkArgs {
  const float* scores;  // the chunk's rows: U x N, row 0 = global row u0
  int64_t U, u0;
  int32_t N, k;
  // every array below is indexed by the GLOBAL row u0 + u
  const int32_t* excl_ids;  // exclusion list of row u = excl_ids[u] (NULL: u); lists outside [0, excl_rows) are empty
  int32_t excl_rows;
  const int64_t* excl_rowptr;
  const int32_t* excl_items;
  const int32_t* targets;   // NULL = no positions
  const int32_t* users;     // optional: a row whose users[u] lies outside [0, num_users) gets -1 / NaN and pos = N
  int32_t num_users;
  int32_t* top_items;
  float* top_scores;
  int32_t* pos;
};
size_t topk_workspace_bytes(int64_t U, int32_t N, int32_t k);  // per chunk of U rows
int launch_topk(const TopkArgs& a, void* ws, cudaStream_t st);
// sums = {hit_sum, dcg_sum} of pos[0, U) in a fixed order, no workspace
int launch_topk_metrics(const int32_t* pos, int64_t U, int k, float* sums, cudaStream_t st);
// Ragged lists: list u is scores[rowptr[u] .. rowptr[u+1]) (segments clamped to [0, nnz)); keys carry the position
// in the list, so ties go to the earlier position.  Outputs per list u (each may be NULL): top_pos / top_items
// (items[start + pos]) / top_scores (U x k, -1 / NaN padding), pos[u] (needs targets: positions in the list).
struct TopkListsArgs {
  const float* scores;
  const int64_t* rowptr;
  int64_t U, nnz;
  int32_t k;
  const int32_t* targets;
  const int32_t* users;  // optional: a list whose users[u] lies outside [0, num_users) gets -1 / NaN and pos = len
  int32_t num_users;
  const int32_t* items;  // needed with top_items
  int32_t* top_pos;
  int32_t* top_items;
  float* top_scores;
  int32_t* pos;
};
size_t topk_lists_workspace_bytes(int64_t U, int64_t nnz, int32_t k);
// sums (may be NULL, needs targets) = {hit_sum, dcg_sum} of the U lists' positions
int launch_topk_lists(const TopkListsArgs& a, float* sums, void* ws, cudaStream_t st);
// seg[r] = the list holding row r (in [0, U)), or users[that list] when users != NULL
int launch_list_rows(const int64_t* rowptr, int64_t U, int64_t nnz, const int32_t* users, int32_t* seg, cudaStream_t st);
// out[r] = r % N for r < rows
int launch_tile_iota(int32_t* out, int64_t rows, int32_t N, cudaStream_t st);
// Positions of many targets per row: row u's targets are tgt_items[tgt_rowptr[u] .. tgt_rowptr[u+1]) (segments clamped
// to [0, nnz_t)); candidates, order and exclusion lists as TopkArgs, a target never excluded.
struct TargetsArgs {
  const float* scores;  // the chunk's rows: U x N, row 0 = global row u0
  int64_t U, u0;
  int32_t N;
  // every array below is indexed by the GLOBAL row u0 + u
  const int32_t* excl_ids;
  int32_t excl_rows;
  const int64_t* excl_rowptr;
  const int32_t* excl_items;
  const int64_t* tgt_rowptr;
  const int32_t* tgt_items;
  int64_t nnz_t;
  const int32_t* users;  // optional: a row whose users[u] lies outside [0, num_users) gives every target position N
  int32_t num_users;
  int32_t* tpos;  // may be NULL
};
constexpr int kTgtSumsMax = MR_TGT_CUTOFF0 + MR_TGT_PER_CUTOFF * MR_MAX_CUTOFFS;
struct TargetCutoffs {
  int32_t k[MR_MAX_CUTOFFS];
  int32_t n;
};
// Workspace of one call: sorted keys, merge scratch and positions (in sorted order) per target, histogram bins per
// target plus one per row of a chunk (C rows), per-block metric partials.
struct TargetsWs {
  unsigned long long *keys, *tmp;
  int32_t *hist, *spos;
  double* partials;
  size_t total;
};
TargetsWs carve_targets(void* ws, int64_t C, int64_t nnz_t);
size_t targets_workspace_bytes(int64_t C, int64_t nnz_t);
// The chunk's positions: w.spos (ascending per row) and a.tpos (list order)
int launch_targets_chunk(const TargetsArgs& a, const TargetsWs& w, cudaStream_t st);
// sums (MR_TGT_* layout, may be NULL) from the positions of all U rows, in a fixed order
int launch_targets_metrics(const int64_t* tgt_rowptr, int64_t U, int64_t nnz_t, const int32_t* spos,
                           const TargetCutoffs& ks, float* sums, double* partials, cudaStream_t st);

// ---- sampler.cu ------------------------------------------------------------------------------
int launch_sample_negatives(const int64_t* rowptr, const int32_t* csr_items, int32_t num_items,
                            const int32_t* pos_users, const int32_t* pos_items, int64_t P, int64_t first_index,
                            int negs, uint64_t seed, uint64_t epoch, int32_t* out_users, int32_t* out_items,
                            float* out_labels, cudaStream_t st);

// ---- fold_in.cu: per-user optimisation of the user rows against a history, everything else frozen ----------------
struct FoldInArgs {
  const MrModel* model;
  const float* wt;          // transposed hidden kernels, dense-block layout
  const float* Pi;          // (num_items x L1) item half of the first layer; NULL without a hidden layer
  const int64_t* rowptr;
  const int32_t* items;
  const int32_t* init_users;
  const int32_t* order;     // the U users, longest history first
  int64_t U;
  MrFoldIn cfg;
  float* out_mlp;
  float* out_gmf;
  float* out_loss;
};
bool fold_in_supported(const MrModel& m);
int launch_fold_in(const FoldInArgs& a, cudaStream_t st);
// Pi = E_item . W1[item rows] with one thread per output (any widths)
int launch_fold_in_project(const MrModel& m, float* Pi, cudaStream_t st);
// flags[0] |= 1 malformed rowptr or unsorted list, 2 item out of range, 4 init user out of range, 8 a list covering
// every item; keys[u] = num_items - length of list u (the longest history sorts first)
int launch_fold_in_check(const int64_t* rowptr, const int32_t* items, int64_t U, int64_t nnz, int32_t num_items,
                         const int32_t* init_users, int32_t num_users, int32_t* keys, int32_t* flags, cudaStream_t st);

// ---- tc_dense.cu / tc_wgrad.cu / head.cu: tensor-core path of the train step ------------------------
enum { TC_EPI_BIAS_RELU = 0, TC_EPI_MASK = 1, TC_EPI_STAGE = 2, TC_EPI_HEAD_DOT = 3 };
struct TcDenseArgs {
  bool gather;            // A = [user row | item row] gathered by id, else a_dense
  const float* a_dense;
  const float* proj_i;    // A = relu(proj_i[items[row0 + r]] + proj_u[r / proj_div]) (rows of K floats): the item-projected
  const float* proj_u;    // first layer computed by this layer's producers; needs items / num_items
  int32_t proj_div;
  const int32_t* proj_ids;  // optional: row r reads proj_u[proj_ids[row0 + r]] (proj_u_rows rows) instead of r / proj_div
  int32_t proj_u_rows;
  const float* user_tab;
  const float* item_tab;
  const int32_t* users;
  const int32_t* items;
  int32_t num_users, num_items, d_u;
  int32_t user_div;       // gather: row r uses users[r / user_div]
  int32_t user_mul;       // gather (user_div == 1): row r uses users[r * user_mul] (one row per group of a grouped batch)
  const float* b_packed;  // launch_pack_weights output
  int32_t N, K;
  int64_t rows, row0;
  int epilogue;
  const float* bias;          // TC_EPI_BIAS_RELU, optional; TC_EPI_HEAD_DOT, required
  const float* head_w;        // TC_EPI_HEAD_DOT: out[r] = relu(acc[r] + bias) . head_w  (out: one float per row)
  const float* addend;        // TC_EPI_BIAS_RELU, optional: row r adds addend[r / addend_div] (launch-local rows x N)
  int32_t addend_div;
  bool linear;                // TC_EPI_BIAS_RELU without the ReLU
  const uint32_t* mask_bits;  // TC_EPI_MASK: ReLU bits written by the forward layer
  uint32_t* bits_out;         // TC_EPI_BIAS_RELU, optional
  float* out;
  int32_t out_ld;             // row stride of `out` in floats (0 = N, a multiple of 4 otherwise)
  float* stage_u;
  float* stage_i;
  int32_t su, si;
};
int launch_tc_dense(const TcDenseArgs& a, cudaStream_t st);
int launch_pack_weights(const float* W, int K_in, int N_out, int transpose, float* dst, cudaStream_t st);

struct TcWgradArgs {
  bool gather;            // A rows = [user row | item row] gathered by id, else a_dense [rows x Fa]
  const float* a_dense;
  const float* user_tab;
  const float* item_tab;
  const int32_t* users;
  const int32_t* items;
  int32_t num_users, num_items, d_u;
  int32_t user_mul;       // gather: user rows read users[(row0 + r) * user_mul]; d_u = 0 / Fa selects one table
  const float* z;         // [rows x Fb] launch-local rows
  int32_t Fa, Fb;
  int64_t rows, row0;
  float* dw_partial;      // per-CTA rows of the dense-gradient partial buffer, this layer's W section
  float* db_partial;      // same, bias section
  int64_t partial_stride;
  bool first;             // overwrite instead of accumulate
};
int tc_wgrad_grid();
int launch_tc_wgrad(const TcWgradArgs& a, cudaStream_t st);

struct HeadArgs {
  const MrModel* model;
  const float* h_last;    // [rows x L_last] launch-local rows
  bool h_is_dot;          // launch_head_rank: h_last holds [rows] floats, the last layer already dotted with its
                          // output-unit weights (tc_dense TC_EPI_HEAD_DOT)
  const int32_t* users;
  const int32_t* items;
  const float* labels;    // NULL = forward only
  int64_t rows, row0;
  int32_t user_div;       // row r uses users[r / user_div]
  int32_t group;          // > 0 (train): grouped batch, stage_u holds ONE row per group (index row / group)
  float inv_batch;
  float* logits;          // global rows, may be NULL
  float* probs;           // global rows, may be NULL
  float* dz_last;         // [rows x L_last] launch-local rows (train)
  float* stage_u;         // GMF row gradients go to columns [d_u, d_u+f) / [d_i, d_i+f) (train)
  float* stage_i;
  float* head_partial;    // head_partial_floats() accumulators, zeroed once per step (train)
  int32_t* flags;
};
// once per step: d w_out / d b_out (row 0 of the dense partial buffer) and loss_sum += the CTA partials
int launch_head_reduce(const MrModel& m, const float* head_partial, float* d_wout_row0, float* d_bout_row0,
                       float* loss_sum, cudaStream_t st);
int head_grid();
bool head_supports_group(const MrModel& m, int group);
size_t head_partial_floats(const MrModel& m);
int launch_head(const HeadArgs& a, cudaStream_t st);
bool head_rank_supported(const MrModel& m);
bool head_rank_takes_dot(const MrModel& m, int group);  // launch_head_rank accepts h_is_dot for this model
int launch_head_rank(const HeadArgs& a, int group, int32_t* pos, float* probs, cudaStream_t st);
// catalogue sweep head: probs[r] from the partial logit h_dot[r] (tc_dense TC_EPI_HEAD_DOT) and the GMF term of
// (users[r / group], item r % group), with the per-row arithmetic of launch_head_rank's partial-logit kernel
bool catalogue_head_supported(const MrModel& m);
int launch_catalogue_head(const MrModel& m, const float* h_dot, const int32_t* users, int64_t rows, int group,
                          float* probs, cudaStream_t st);
// the same for candidate lists: global row row0 + r pairs users[seg[row0 + r]] (seg < num_lists) with items[row0 + r];
// h_dot launch-local, probs global
int launch_lists_head(const MrModel& m, const float* h_dot, const int32_t* users, int64_t num_lists, const int32_t* seg,
                      const int32_t* items, int64_t row0, int64_t rows, float* probs, cudaStream_t st);
// metric sums from positions (rank.cu): sums = {hit_sum, dcg_sum}
int launch_rank_metrics(const int32_t* pos, int64_t G, int k, float* sums, float* partials, cudaStream_t st);

// row-sharded tables over peer pointers (gather.cu): shards = device array of `world` table-slice pointers
int launch_gather_rows_sharded(const float* const* shards, int world, int64_t total_rows, int dim, const int32_t* ids,
                               int64_t n, float* out, cudaStream_t st);

// data-parallel replicas (dp_exchange.cu): sum of the ranks' gradients + optimizer + store to every replica for
// elements [lo, hi) of a region; grad_peers / param_peers are HOST arrays of `world` peer-mapped device pointers
int launch_dp_reduce_apply(const float* const* grad_peers, float* const* param_peers, int world, int rank, float* m,
                           float* v, int64_t lo, int64_t hi, int optimizer, float lr_t, float beta_1, float beta_2,
                           float epsilon, float l2, const float* grad_multicast, float* param_multicast,
                           cudaStream_t st);

// ---- the reference's default tower 64-32-16-8 + GMF 8 as a projected grouped step on CUDA cores (small_tower.cu) ----
struct SmallTowerArgs {
  const MrModel* model;
  const float *Pi, *Pu;  // E_item . W1i (num_items x L1), E_user . W1u + b1 (num_users x L1)
  const int32_t *users, *items;
  const float* labels;
  int64_t B;
  float inv_batch;
  float* probs;
  float *stage_i, *stage_u;  // [dZ1 | GMF row gradient] per row / per group
  float* dense_partial;      // rows of dense_stride floats, one per CTA: layers >= 2 and the output unit
  int64_t dense_stride;
  float* loss_partial;
  int32_t* flags;
  int max_ctas;
};
bool small_tower_supported(const MrModel& m, int group);
int launch_small_tower_train(const SmallTowerArgs& a, cudaStream_t st, int* grid_out);
// forward of the same tower: probs[row] for rows whose user is users[row / group]; with seg (candidate lists), row r
// belongs to list seg[r] < num_lists, whose user is users[seg[r]] and whose Pu row is seg[r]
int launch_small_tower_forward(const MrModel& m, const float* Pi, const float* Pu, const int32_t* users,
                               const int32_t* items, int64_t rows, int group, float* probs, cudaStream_t st,
                               const int32_t* seg = nullptr, int64_t num_lists = 0);
// out = A (rows x K) . W (K x N, or its transpose read from an N x K array when `transpose`) (+ bias)
int launch_small_rows_gemm(const float* A, int64_t rows, int K, const float* W, int ldw, int N, bool transpose,
                           const float* bias, float* out, cudaStream_t st);
// dW (32 x 32) = E^T . S, db = colsum(S) into per-CTA rows of a partial buffer
int launch_small_table_wgrad(const float* E, const float* S, int64_t rows, float* dw_partial, float* db_partial,
                             int64_t stride, int max_ctas, cudaStream_t st, int* grid_out);

// ---- grouped batches (gather.cu): one positive and its negatives share the user ----------------------------
// out[g] = sum_{j < group} in[g * group + j]  (rows of `width` floats, width % 4 == 0, row strides in_ld / out_ld
// floats, 0 = width), fixed order
int launch_group_sum_rows(const float* in, int64_t groups, int group, int width, float* out, cudaStream_t st,
                          int in_ld = 0, int out_ld = 0);
// Item-projected first layer: H1[r] = relu(Pi[items[row0 + r]] + Zu[r / group]) and its ReLU bits; Pi holds
// E_item . W1[item rows] for every item (width floats per row), Zu the user half + bias of each group -- or, with
// `users` (one id per row, global rows), of each USER: row r then adds Zu[users[row0 + r]].
int launch_h1_from_projection(const float* Pi, int32_t num_items, const int32_t* items, int64_t row0, int64_t rows,
                              const float* Zu, int group, const int32_t* users, int32_t num_users, int width, float* H1,
                              uint32_t* bits, cudaStream_t st);
// out[g] = ids[g * group]
int launch_group_heads(const int32_t* ids, int64_t groups, int group, int32_t* out, cudaStream_t st);
// *flag = 1 when some ids[r] != ids[r - r % group]
int launch_check_grouped(const int32_t* ids, int64_t n, int group, int32_t* flag, cudaStream_t st);

// ---- dataset.cu: split and per-user item lists on the device ------------------------------------------------------
size_t split_workspace_bytes(int64_t n);
int launch_split_last_two(const int32_t* users, int64_t n, int32_t num_users, int32_t* order, int32_t* part,
                          int32_t* flag, void* ws, size_t ws_bytes, cudaStream_t st);
size_t remap_workspace_bytes(int64_t n);
int launch_remap_ids(const int32_t* ids, int64_t n, int32_t limit, int32_t* dense, int32_t* unique, int64_t* num_unique,
                     int32_t* flag, void* ws, size_t ws_bytes, cudaStream_t st);
size_t user_csr_workspace_bytes(int64_t n);
int launch_build_user_csr(const int32_t* users, const int32_t* items, int64_t n, int32_t num_users, int32_t num_items,
                          int64_t* rowptr, int32_t* csr_items, int32_t* flag, void* ws, size_t ws_bytes,
                          cudaStream_t st);

// ---- tc_fused.cu: the projected tower's per-row work of a grouped train step in ONE kernel ----------------------
struct FusedTrainArgs {
  const float* Pi;        // [num_items x L1] item half of the first layer
  const float* Pu;        // [num_users x L1] user half + bias
  const float* user_gmf;
  const float* item_gmf;
  const int32_t* users;
  const int32_t* items;
  const float* labels;
  int32_t num_users, num_items;
  int64_t rows;
  int32_t group;
  const float* W2;        // (L1, L2) Keras layout; packed into w2_image by the launcher
  uint16_t* w2_image;     // fused_w2_image_bytes() of workspace
  const float* b2;
  const float* w_out;
  const float* b_out;
  float inv_batch;
  float* probs;
  float* stage_i;         // [rows x si]: dZ1 | d gmf_i
  float* stage_u;         // [rows / group x su]: group sums of dZ1 | d gmf_u
  int32_t si, su;
  float* partial;         // dense-gradient partial rows (one per CTA, zeroed by the caller), stride partial_stride
  int64_t partial_stride;
  int64_t off_w2, off_b2, off_wout, off_bout;
  float* loss_partial;    // one float per CTA (written, not accumulated)
  int32_t* flags;
};
bool fused_train_supported(const MrModel& m, int group);
size_t fused_w2_image_bytes();
int launch_fused_train(const FusedTrainArgs& a, cudaStream_t st, int* grid_out);
int launch_bf16x3_selftest(const float* A, const float* B, float* D, int N, int K, int a_mn, int b_mn, cudaStream_t st);

// ---- tc_selftest.cu ---------------------------------------------------------------------------
int launch_tc_rate(int N, int iters, int nbuf, int flags, int writers, int write_iters, long long* out, int grid,
                   cudaStream_t st);
int launch_tc_probe(const float* raw_a, int n_words, int start_off, int lbo, int sbo, int a_mn, float* D,
                    cudaStream_t st);
int launch_tc_selftest(const float* A, const float* B, float* D, int N, int K, int a_mn, int b_mn, int three_x,
                       cudaStream_t st);

}  // namespace mr
