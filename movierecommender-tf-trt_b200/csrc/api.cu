// C-ABI layer of libmovierec_b200.so (declared in include/movierec_b200.h): argument validation,
// workspace carving and the launch sequence of each entry point.  No device memory is allocated
// here and nothing synchronises; every launch goes to the caller's stream.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "launchers.h"
#include "neumf_tile.cuh"

namespace mr {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error in %s: %s", what, cudaGetErrorString(e));
  return MR_ERR_CUDA;
}

int sm_count() {
  static thread_local int cached_dev = -1, cached = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    cudaGetLastError();
    return kB200Sms;  // sizing queries must work without a device
  }
  if (dev != cached_dev) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) {
      cudaGetLastError();
      return kB200Sms;
    }
    cached = n;
    cached_dev = dev;
  }
  return cached;
}

// ---- opt-in profiling (thread-local) -----------------------------------------------------------------
struct Profiler {
  bool on = false;
  bool overflow = false;
  std::vector<cudaEvent_t> events;
  std::vector<int> phase;
  size_t used = 0;
  int64_t launches = 0;
};
static thread_local Profiler g_prof;
constexpr size_t kMaxProfEvents = 1 << 16;

void count_launch() { g_prof.launches += 1; }

void prof_mark(int phase, cudaStream_t st) {
  Profiler& p = g_prof;
  if (!p.on) return;
  if (p.used >= kMaxProfEvents) {
    p.overflow = true;
    return;
  }
  if (p.used == p.events.size()) {
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) {
      cudaGetLastError();
      p.overflow = true;
      return;
    }
    p.events.push_back(e);
    p.phase.push_back(-1);
  }
  cudaEventRecord(p.events[p.used], st);
  p.phase[p.used] = phase;
  p.used += 1;
}

// flags[0]: out-of-range id seen, flags[1]: grouped-batch promise violated -> bits 0 and 1 of the output
// ---- side stream (thread-local, per device): the id sorts of the train step do not depend on the tower, so they
// run next to it (the tower's persistent CTAs leave room for small kernels).  Fork and join are events on the
// caller's stream: the call stays asynchronous and capturable.
struct SideStream {
  int dev = -1;
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  cudaEvent_t fork2 = nullptr, join2 = nullptr;  // second excursion of a step: the user-side segmented reduction
  // the train step's last reads of the user GMF table: the user-side reduction (side stream) and the level 0 of an
  // item-side reduction that forms the GMF item gradient from it (caller's stream)
  cudaEvent_t user_sums = nullptr, gmf_read = nullptr;
};
static thread_local SideStream g_side;

static SideStream* side_stream() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  SideStream& s = g_side;
  if (s.dev != dev) {
    s = SideStream{};
    if (cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.fork2, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.join2, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.user_sums, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.gmf_read, cudaEventDisableTiming) != cudaSuccess) {
      cudaGetLastError();
      s = SideStream{};
      return nullptr;
    }
    s.dev = dev;
  }
  return &s;
}

__global__ void flag_to_float_kernel(const int32_t* flags, float* out) {
  *out = (float)((flags[0] ? 1 : 0) | (flags[1] ? 2 : 0));
}

static int bits_for(int64_t n) {
  int b = 1;
  while (b < 31 && ((int64_t)1 << b) < n) ++b;
  return b;
}

// Sort of the row ids that key a segmented reduction over a table of num_rows rows: ids outside [0, num_rows) sort as
// the sentinel num_rows (one value more than the valid ids, hence bits_for(num_rows + 1)), after every valid id, so
// they can never split a valid id's run; the reduction skips the sentinel's run.
static int sort_row_ids(const int32_t* ids, int64_t n, int32_t num_rows, int32_t* sorted_keys, int32_t* sorted_index,
                        void* ws, size_t ws_bytes, cudaStream_t st) {
  return launch_sort_pairs(ids, n, bits_for((int64_t)num_rows + 1), sorted_keys, sorted_index, ws, ws_bytes, st,
                           num_rows);
}

static int check_model(const MrModel* m) {
  MR_REQUIRE(m != nullptr, "model is NULL");
  MR_REQUIRE(m->n_layers >= 1 && m->n_layers <= MR_MAX_LAYERS, "n_layers=%d out of [1,%d]", m->n_layers, MR_MAX_LAYERS);
  MR_REQUIRE(m->L[0] >= 2, "layers_sizes[0]=%d must be >= 2", m->L[0]);
  for (int l = 0; l < m->n_layers; ++l)
    MR_REQUIRE(m->L[l] >= 1 && m->L[l] <= MR_MAX_WIDTH, "layers_sizes[%d]=%d out of [1,%d]", l, m->L[l], MR_MAX_WIDTH);
  MR_REQUIRE(m->mf_dim >= 0 && m->mf_dim <= MR_MAX_WIDTH, "mf_dim=%d out of range", m->mf_dim);
  MR_REQUIRE(m->num_users > 0 && m->num_items > 0, "num_users/num_items must be > 0");
  MR_REQUIRE(m->user_mlp && m->item_mlp && m->dense && m->w_out && m->b_out, "model has NULL parameter pointers");
  if (m->mf_dim > 0) MR_REQUIRE(m->user_gmf && m->item_gmf, "mf_dim > 0 but GMF tables are NULL");
  // dense block layout: W[1], b[1], ..., w_out, b_out
  int64_t off = 0;
  for (int l = 1; l < m->n_layers; ++l) {
    MR_REQUIRE(m->W[l] == m->dense + off, "W[%d] is not at its offset in the dense block", l);
    off += (int64_t)m->L[l - 1] * m->L[l];
    MR_REQUIRE(m->b[l] == m->dense + off, "b[%d] is not at its offset in the dense block", l);
    off += m->L[l];
  }
  MR_REQUIRE(m->w_out == m->dense + off, "w_out is not at its offset in the dense block");
  off += m->mf_dim + m->L[m->n_layers - 1];
  MR_REQUIRE(m->b_out == m->dense + off, "b_out is not at its offset in the dense block");
  off += 1;
  MR_REQUIRE(m->dense_count == off, "dense_count=%lld, expected %lld", (long long)m->dense_count, (long long)off);
  MR_REQUIRE(choose_tile_rows(*m, true) > 0, "layer widths too large for the fused kernel's shared memory");
  return MR_OK;
}

static bool any_l2(const MrModel& m) {
  for (int l = 0; l < m.n_layers; ++l)
    if (m.l2[l] != 0.f) return true;
  return false;
}

// ---- tensor-core path (tcgen05 3xTF32): eligibility, workspace and launch sequence ----------------------
static bool tc_eligible(const MrModel& m) {
  if (m.n_layers < 2) return false;
  if (m.L[0] % 64) return false;  // d_u = L0/2 must be a multiple of 32 (K-chunks never straddle the two tables)
  for (int l = 0; l < m.n_layers; ++l)
    if (m.L[l] % 32 || m.L[l] > 256) return false;
  for (int l = 0; l + 1 < m.n_layers; ++l)
    if (m.L[l] % 128) return false;  // input width of every dense layer = M of the weight-gradient MMAs
  for (int l = 1; l < m.n_layers; ++l)
    if (m.L[l] & (m.L[l] - 1)) return false;  // output widths 32/64/128/256 (bias-gradient column ownership)
  if (m.mf_dim + m.L[m.n_layers - 1] > 512) return false;
  const uintptr_t a = reinterpret_cast<uintptr_t>(m.user_mlp) | reinterpret_cast<uintptr_t>(m.item_mlp) |
                      reinterpret_cast<uintptr_t>(m.dense);
  return (a & 15) == 0;
}

static bool use_tc(const MrModel& m) { return m.compute_path != MR_PATH_SIMT && tc_eligible(m); }

// Item-projected first layer (grouped train step, fused ranking eval).  The first Dense layer is linear before its
// ReLU, so E_item . W1[item rows] is a function of the item alone: with `rows` rows per step and num_items << rows
// it is computed once per ITEM (Pi, one GEMM over the item table) and the per-row part of the layer becomes a
// gather + add + ReLU.  Backward by the same linearity: dZ1 rows are segment-summed by item FIRST (the sorted
// segmented reduction that already exists, fed dZ1 instead of dZ1 . W1i^T), then the item half of the backward
// GEMM and of the weight gradient run on num_items rows instead of `rows`.  Same values up to summation order.
// Needs L1 == d_i so that the staged item rows keep their width d_i + f, and dense gradient tables.
// (selector: MrModel.item_projection -- part of the model description, so that workspace sizing and the launch
// sequence of every call on that model agree).  any_rows: a choice of the model alone, AUTO as at any row count.
static bool item_proj_ok(const MrModel& m, int64_t rows, bool any_rows = false) {
  if (m.item_projection == MR_PROJECTION_OFF || !use_tc(m) || m.n_layers < 3) return false;
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u;
  if (d_i % 128 || d_i > 256 || m.L[1] != d_i) return false;
  if (m.item_projection == MR_PROJECTION_ON || any_rows) return true;
  return 2 * (int64_t)m.num_items <= rows;  // three GEMMs over num_items rows replace three over `rows` rows
}

// The same for the user half (train step): with no more users than a step has groups, E_user . W1[user rows] + b1 is
// computed once per USER (Pu), and the group sums of dZ1 are segment-summed by user before the user half of the
// backward GEMM and of the weight gradient.  Needs the item projection and L1 == d_u.
static bool user_proj_ok(const MrModel& m, int64_t rows, int group) {
  if (!item_proj_ok(m, rows) || group < 2) return false;
  if (m.L[1] != m.L[0] / 2) return false;
  return m.item_projection == MR_PROJECTION_ON || (int64_t)m.num_users <= rows / group;
}

// The reference's default tower (64-32-16-8, GMF 8) takes the same two projections on CUDA cores (small_tower.cu):
// grouped batches of five rows, dense gradient tables, at least twice as many rows as items and no more users than
// groups (or MR_PROJECTION_ON).  MR_PROJECTION_OFF / MR_FUSED_OFF keep the generic tile kernel (A/B runs, tests).
static bool small_proj_ok(const MrModel& m, int64_t rows, int group) {
  if (use_tc(m) || m.item_projection == MR_PROJECTION_OFF || m.fused_train == MR_FUSED_OFF) return false;
  if (group < 1 || !small_tower_supported(m, group) || rows % group) return false;
  if (m.item_projection == MR_PROJECTION_ON) return true;
  return 2 * (int64_t)m.num_items <= rows && (int64_t)m.num_users <= rows / group;
}

// ranking eval of the default tower: one user id per group of candidates, Pi / Pu over the tables first
static bool small_eval_ok(const MrModel& m, int64_t rows, bool any_rows = false) {
  if (use_tc(m) || m.item_projection == MR_PROJECTION_OFF || m.fused_train == MR_FUSED_OFF) return false;
  if (!small_tower_supported(m, 5)) return false;
  if (m.item_projection == MR_PROJECTION_ON || any_rows) return true;
  return 2 * ((int64_t)m.num_items + m.num_users) <= rows;
}

struct SmallWs {
  float *Pi, *Pu, *Si, *Su;
  size_t total;
};
static SmallWs carve_small(const MrModel& m, void* ws) {
  SmallWs w{};
  Carver cv(ws);
  w.Pi = cv.take<float>((size_t)m.num_items * m.L[1]);
  w.Pu = cv.take<float>((size_t)m.num_users * m.L[1]);
  w.Si = cv.take<float>((size_t)m.num_items * m.L[1]);
  w.Su = cv.take<float>((size_t)m.num_users * m.L[1]);
  w.total = cv.off;
  return w;
}

// Rows per launch of the tensor-core kernels: the whole batch up to 2^21 rows (persistent CTAs need many
// tiles each to reach steady state: one launch of 1,310,720 rows instead of two of 655,360 takes the ML-20M step
// from 2.48 to 2.45 ms, and four of 327,680 cost +0.25 ms; intermediates are ~2.3 KB of workspace per row), split
// evenly above.
constexpr int64_t kTcSubBatchCap = (int64_t)1 << 21;    // train / forward
constexpr int64_t kEvalSubBatchCap = (int64_t)1 << 22;  // ranking eval

static int64_t tc_sub_batch(int64_t B) {
  const int64_t cap = kTcSubBatchCap;
  const int64_t parts = B <= cap ? 1 : (B + cap - 1) / cap;
  const int64_t sb = ((B < 1 ? 1 : B) + parts - 1) / parts;
  return (sb + 127) / 128 * 128;
}

struct TcWs {
  float* pack_f[MR_MAX_LAYERS];  // forward operand of W[l]   (rows = output unit)
  float* pack_b[MR_MAX_LAYERS];  // backward operand of W[l]  (rows = input unit)
  float* H[MR_MAX_LAYERS];       // activations of a sub-batch, H[l] (SB x L[l])
  float* dZ[MR_MAX_LAYERS];      // pre-activation gradients of a sub-batch
  uint32_t* bits[MR_MAX_LAYERS]; // ReLU bits (H[l] > 0), one word per 32 units, written by the forward layer
  float* head_partial;
  // grouped batches (train): first-layer operands split into the user rows and the item rows of W[1]
  float* pack_fu;  // forward, user rows   (d_u x L1)
  float* pack_fi;  // forward, item rows   (d_i x L1)
  float* pack_bu;  // backward, user rows
  float* pack_bi;  // backward, item rows
  float* Zu;       // (sub-batch groups x L1): user half of the first layer + bias, one row per group
  float* S1;       // (sub-batch groups x L1): dZ[1] summed over the rows of each group
  // item-projected first layer (item_proj_ok)
  float* Pi;       // (num_items x L1): E_item . W1[item rows]
  float* Si;       // (num_items x L1): dZ[1] summed over the rows of each item (train)
  float* Pu;       // (num_users x L1): E_user . W1[user rows] + b1 (train, user_proj_ok)
  float* Su;       // (num_users x L1): dZ[1] summed over the rows of each user (train)
  uint16_t* w2_image;  // fused train kernel: W[2] as its shared-memory operand image (tc_fused.cu)
  size_t total;
};

// Grouped first layer: the user half runs once per group.  Needs whole groups per sub-batch, both halves of
// the first layer wide enough for the weight-gradient MMAs (M = 128) and the grouped head kernel.
static bool tc_grouped_ok(const MrModel& m, int64_t B, int group) {
  if (group < 2 || !tc_eligible(m) || !head_supports_group(m, group)) return false;
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u;
  if (d_u % 128 || d_i % 128 || d_u > 256 || d_i > 256) return false;
  if (B % group) return false;
  const int64_t cap = kTcSubBatchCap;
  const int64_t parts = B <= cap ? 1 : (B + cap - 1) / cap;
  if (parts > 1 && (tc_sub_batch(B) % group)) return false;  // sub-batch boundaries must not split a group
  return true;
}

static TcWs carve_tc(const MrModel& m, bool train, int64_t B, void* ws) {
  TcWs t{};
  Carver cv(ws);
  const int64_t sb = tc_sub_batch(B);
  for (int l = 1; l < m.n_layers; ++l) {
    const size_t kn = (size_t)m.L[l - 1] * m.L[l];
    t.pack_f[l] = cv.take<float>(2 * kn);
    if (train) t.pack_b[l] = cv.take<float>(2 * kn);
    t.H[l] = cv.take<float>((size_t)sb * m.L[l]);
    if (train) t.dZ[l] = cv.take<float>((size_t)sb * m.L[l]);
    if (train) t.bits[l] = cv.take<uint32_t>((size_t)sb * (m.L[l] / 32));
  }
  t.head_partial = cv.take<float>(head_partial_floats(m));
  if (train && m.n_layers >= 2) {
    const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u;
    t.pack_fu = cv.take<float>((size_t)2 * d_u * m.L[1]);
    t.pack_fi = cv.take<float>((size_t)2 * d_i * m.L[1]);
    t.pack_bu = cv.take<float>((size_t)2 * d_u * m.L[1]);
    t.pack_bi = cv.take<float>((size_t)2 * d_i * m.L[1]);
    const int64_t sg = sb / 2 + 1;  // groups per sub-batch (group >= 2)
    t.Zu = cv.take<float>((size_t)sg * m.L[1]);
    t.S1 = cv.take<float>((size_t)sg * m.L[1]);
    if (item_proj_ok(m, B)) {
      t.Pi = cv.take<float>((size_t)m.num_items * m.L[1]);
      t.Si = cv.take<float>((size_t)m.num_items * m.L[1]);
      if (m.L[1] == d_u) {  // user projection: decided per call (it depends on the group size)
        t.Pu = cv.take<float>((size_t)m.num_users * m.L[1]);
        t.Su = cv.take<float>((size_t)m.num_users * m.L[1]);
      }
    }
    t.w2_image = cv.take<uint16_t>(fused_w2_image_bytes() / sizeof(uint16_t));
  }
  t.total = cv.off;
  return t;
}

// First layer of a grouped batch, rows [r0, r1): the user half once per group, Zu = E_user[user of the group] .
// W1[user rows] + b1, and the item half per row.  A train workspace (ReLU bits) writes H1 and its bits; an eval
// workspace has no Pu.  The cases:
//  - eval with Pi: Zu, then the second layer's producers read relu(Pi[item] + Zu[group]) (H1 never exists in memory);
//  - train with Pu: H1 = relu(Pi[item] + Pu[user]), the user half once per USER;
//  - train with Pi only: Zu, then H1 = relu(Pi[item] + Zu[group]);
//  - eval or train without Pi: Zu, then H1 = relu(E_item[item] . W1[item rows] + Zu[group]).
// Zu rows [0, rows) = E_user[users[(row0 + r) * user_mul]] . W1[user rows] + b1 (a zero row for an out-of-range user).
static int tc_user_half(const MrModel& m, const TcWs& t, const int32_t* users, int user_mul, int64_t row0, int64_t rows,
                        cudaStream_t st) {
  TcDenseArgs a{};
  a.gather = true;
  a.user_tab = m.user_mlp;
  a.users = users;
  a.num_users = m.num_users;
  a.num_items = m.num_items;
  a.d_u = m.L[0] / 2;
  a.user_div = 1;
  a.user_mul = user_mul;
  a.b_packed = t.pack_fu;
  a.N = m.L[1];
  a.K = m.L[0] / 2;
  a.rows = rows;
  a.row0 = row0;
  a.epilogue = TC_EPI_BIAS_RELU;
  a.bias = m.b[1];
  a.linear = true;
  a.out = t.Zu;
  return launch_tc_dense(a, st);
}

static int tc_grouped_first_layer(const MrModel& m, const TcWs& t, const int32_t* users, const int32_t* items, int64_t r0,
                                  int64_t r1, int group, bool users_per_group, cudaStream_t st) {
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u;
  const bool train = t.bits[1] != nullptr;
  if (train && t.Pu != nullptr) {
    prof_mark(MR_PHASE_H1_GATHER, st);
    const int rc = launch_h1_from_projection(t.Pi, m.num_items, items, r0, r1 - r0, t.Pu, group, users, m.num_users,
                                             m.L[1], t.H[1], t.bits[1], st);
    if (rc == MR_OK) prof_mark(MR_PHASE_TC_DENSE_FWD, st);
    return rc;
  }
  // `users` holds one id per group, or one per row
  int rc = tc_user_half(m, t, users, users_per_group ? 1 : group, r0 / group, (r1 - r0) / group, st);
  if (rc != MR_OK || (!train && t.Pi != nullptr)) return rc;
  if (t.Pi != nullptr) {
    prof_mark(MR_PHASE_H1_GATHER, st);
    rc = launch_h1_from_projection(t.Pi, m.num_items, items, r0, r1 - r0, t.Zu, group, nullptr, 0, m.L[1], t.H[1],
                                   t.bits[1], st);
    if (rc == MR_OK) prof_mark(MR_PHASE_TC_DENSE_FWD, st);
    return rc;
  }
  TcDenseArgs b{};
  b.gather = true;
  b.item_tab = m.item_mlp;
  b.items = items;
  b.num_users = m.num_users;
  b.num_items = m.num_items;
  b.d_u = 0;
  b.user_div = 1;
  b.b_packed = t.pack_fi;
  b.N = m.L[1];
  b.K = d_i;
  b.rows = r1 - r0;
  b.row0 = r0;
  b.epilogue = TC_EPI_BIAS_RELU;
  b.addend = t.Zu;
  b.addend_div = group;
  b.out = t.H[1];
  b.bits_out = t.bits[1];
  return launch_tc_dense(b, st);
}

// Forward of rows [r0, r1) on the tensor cores; leaves H[1..n-1] of the sub-batch in the workspace.  group > 0: a
// grouped batch, whose first layer tc_grouped_first_layer runs.  proj_ids (candidate lists): t.Zu already holds
// proj_u_rows user halves and row r reads Zu[proj_ids[r]].  head_dot: H[n-1] holds one float per row, the last
// layer's output dotted with w_out[MLP columns].
static int tc_forward_rows(const MrModel& m, const TcWs& t, const int32_t* users, const int32_t* items, int user_div,
                           int64_t r0, int64_t r1, cudaStream_t st, int group = 0, bool users_per_group = false,
                           bool head_dot = false, const int32_t* proj_ids = nullptr, int32_t proj_u_rows = 0) {
  const int d_u = m.L[0] / 2;
  const bool split_first = group > 0 || proj_ids != nullptr;  // the first layer's user half is Zu
  // the eval case of the split first layer, whose H1 the second layer's producers compute
  const bool proj_in_producer = split_first && t.bits[1] == nullptr && t.Pi != nullptr;
  if (group > 0) {
    const int rc = tc_grouped_first_layer(m, t, users, items, r0, r1, group, users_per_group, st);
    if (rc != MR_OK) return rc;
  }
  for (int l = split_first ? 2 : 1; l < m.n_layers; ++l) {
    TcDenseArgs a{};
    a.gather = (l == 1);
    a.a_dense = (l == 1) ? nullptr : t.H[l - 1];
    a.user_tab = m.user_mlp;
    a.item_tab = m.item_mlp;
    a.users = users;
    a.items = items;
    a.num_users = m.num_users;
    a.num_items = m.num_items;
    a.d_u = d_u;
    a.user_div = user_div;
    a.b_packed = t.pack_f[l];
    a.N = m.L[l];
    a.K = m.L[l - 1];
    a.rows = r1 - r0;
    a.row0 = r0;
    a.epilogue = TC_EPI_BIAS_RELU;
    a.bias = m.b[l];
    a.out = t.H[l];
    a.bits_out = t.bits[l];  // NULL in forward-only runs
    if (proj_in_producer && l == 2) {
      a.a_dense = nullptr;
      a.proj_i = t.Pi;
      a.proj_u = t.Zu;
      a.proj_div = group;
      a.proj_ids = proj_ids;
      a.proj_u_rows = proj_u_rows;
    }
    if (head_dot && l == m.n_layers - 1) {
      a.epilogue = TC_EPI_HEAD_DOT;
      a.head_w = m.w_out + m.mf_dim;
    }
    int rc = launch_tc_dense(a, st);
    if (rc != MR_OK) return rc;
  }
  return MR_OK;
}

// P = E . W1h over a whole table E (rows x K), linear, no bias (pack must hold the packed row block W1h (K x L[1]) of
// W[1]): the item half of the first layer over the item table, or fold-in's other half over the user table.
static int tc_project_table(const MrModel& m, const float* E, int64_t rows, int K, const float* pack, float* P,
                            cudaStream_t st) {
  TcDenseArgs a{};
  a.a_dense = E;
  a.b_packed = pack;
  a.N = m.L[1];
  a.K = K;
  a.rows = rows;
  a.row0 = 0;
  a.epilogue = TC_EPI_BIAS_RELU;
  a.linear = true;
  a.out = P;
  return launch_tc_dense(a, st);
}

// Pu = E_user . W1[user rows] + b1 over the whole user table (pack_fu must hold the packed user rows of W[1]).
static int tc_project_users(const MrModel& m, const TcWs& t, cudaStream_t st) {
  TcDenseArgs a{};
  a.a_dense = m.user_mlp;
  a.b_packed = t.pack_fu;
  a.N = m.L[1];
  a.K = m.L[0] / 2;
  a.rows = m.num_users;
  a.row0 = 0;
  a.epilogue = TC_EPI_BIAS_RELU;
  a.bias = m.b[1];
  a.linear = true;
  a.out = t.Pu;
  return launch_tc_dense(a, st);
}

// Backward of one half of the first layer over its whole table E (rows x d), on the per-row sums S (rows x L1):
// dE = S . W1h^T (pack_b: the packed backward operand of that half of W[1]), and d W1h = E^T . S plus, with db_partial,
// d b1 = colsum(S) into the dense partial rows.  mark_phases: attribute the two launches to their phases on st.
static int tc_table_backward(const MrModel& m, const float* E, const float* S, int64_t rows, int d, const float* pack_b,
                             float* dE, float* dw_partial, float* db_partial, int64_t partial_stride, bool mark_phases,
                             cudaStream_t st) {
  if (mark_phases) prof_mark(MR_PHASE_TC_DENSE_BWD, st);
  TcDenseArgs a{};
  a.a_dense = S;
  a.b_packed = pack_b;
  a.N = d;
  a.K = m.L[1];
  a.rows = rows;
  a.row0 = 0;
  a.epilogue = TC_EPI_BIAS_RELU;
  a.linear = true;
  a.out = dE;
  const int rc = launch_tc_dense(a, st);
  if (rc != MR_OK) return rc;
  if (mark_phases) prof_mark(MR_PHASE_TC_WGRAD, st);
  TcWgradArgs w{};
  w.a_dense = E;
  w.z = S;
  w.Fa = d;
  w.Fb = m.L[1];
  w.rows = rows;
  w.row0 = 0;
  w.dw_partial = dw_partial;
  w.db_partial = db_partial;
  w.partial_stride = partial_stride;
  return launch_tc_wgrad(w, st);
}

struct TrainWs {
  int32_t* flags;
  float* wt;
  float* dense_partial;
  int64_t dense_stride;
  float* loss_partial;
  float* probs;
  float* stage_u;
  float* stage_i;
  int32_t* sorted_keys;    // users (or the users of the groups), sorted
  int32_t* sorted_index;
  int32_t* sorted_keys_i;  // items, sorted
  int32_t* sorted_index_i;
  void* sort_ws;
  size_t sort_ws_bytes;
  void* seg_ws;
  size_t seg_ws_bytes;
  void* seg_ws_u;  // user-side reduction when it runs next to the item-side one
  size_t seg_ws_u_bytes;
  void* tc_ws;
  size_t tc_ws_bytes;
  void* small_ws;  // projected tables and per-item / per-user sums of the default-tower step
  size_t small_ws_bytes;
  int32_t* pos;
  float* rank_partials;
  int32_t* group_users;  // grouped batches: the user of each group
  size_t total;
};

static TrainWs carve_train(const MrModel& m, int64_t B, void* ws) {
  TrainWs t;
  Carver cv(ws);
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u;
  const int cap = max_tile_ctas();
  t.flags = cv.take<int32_t>(64);
  t.wt = cv.take<float>(m.dense_count);
  t.dense_stride = (m.dense_count + 3) & ~(int64_t)3;
  t.dense_partial = cv.take<float>((size_t)cap * t.dense_stride);
  t.loss_partial = cv.take<float>(cap);
  t.probs = cv.take<float>(B);
  t.stage_u = cv.take<float>((size_t)B * (d_u + m.mf_dim));
  // (the fused train kernel's rows are L1 = d_i wide; its dz per row follows them in the same block: TrainStep::plan)
  t.stage_i = cv.take<float>((size_t)B * (d_i + m.mf_dim));
  t.sorted_keys = cv.take<int32_t>(B);
  t.sorted_index = cv.take<int32_t>(B);
  t.sorted_keys_i = cv.take<int32_t>(B);
  t.sorted_index_i = cv.take<int32_t>(B);
  t.sort_ws_bytes = sort_workspace_bytes(B);
  t.sort_ws = cv.take<char>(t.sort_ws_bytes);
  t.seg_ws_bytes = segreduce_workspace_bytes(B, (d_u > d_i ? d_u : d_i) + m.mf_dim);
  t.seg_ws = cv.take<char>(t.seg_ws_bytes);
  t.seg_ws_u_bytes = segreduce_workspace_bytes(B / 2 + 1, d_u + m.mf_dim);
  t.seg_ws_u = cv.take<char>(t.seg_ws_u_bytes);
  t.pos = cv.take<int32_t>(B);
  t.rank_partials = cv.take<float>(rank_partials_count(B));
  t.group_users = cv.take<int32_t>(B / 2 + 1);
  t.tc_ws_bytes = tc_eligible(m) ? carve_tc(m, true, B, nullptr).total : 0;
  t.tc_ws = cv.take<char>(t.tc_ws_bytes);
  t.small_ws_bytes = (!tc_eligible(m) && small_tower_supported(m, 5)) ? carve_small(m, nullptr).total : 0;
  t.small_ws = cv.take<char>(t.small_ws_bytes);
  t.total = cv.off;
  return t;
}

static float adam_lr_t(const MrOptState& o, int64_t t) {
  // legacy Keras Adam folds both bias corrections into the step size (SURVEY App. A-4)
  return (float)((double)o.lr * sqrt(1.0 - pow((double)o.beta_2, (double)t)) / (1.0 - pow((double)o.beta_1, (double)t)));
}

static int check_opt(const MrModel& m, const MrOptState* o, const MrGrads* g) {
  MR_REQUIRE(o != nullptr && g != nullptr, "opt/grads is NULL");
  MR_REQUIRE(o->optimizer == MR_OPT_ADAM || o->optimizer == MR_OPT_SGD, "unknown optimizer %d", o->optimizer);
  MR_REQUIRE(o->table_mode == MR_TABLES_DENSE || o->table_mode == MR_TABLES_SPARSE, "unknown table_mode %d", o->table_mode);
  MR_REQUIRE(g->dense != nullptr, "grads.dense is NULL");
  if (o->optimizer == MR_OPT_ADAM) {
    MR_REQUIRE(o->m_dense && o->v_dense && o->m_user_mlp && o->v_user_mlp && o->m_item_mlp && o->v_item_mlp,
               "Adam state pointers are NULL");
    if (m.mf_dim > 0) MR_REQUIRE(o->m_user_gmf && o->v_user_gmf && o->m_item_gmf && o->v_item_gmf, "Adam GMF state is NULL");
  }
  if (o->table_mode == MR_TABLES_DENSE) {
    MR_REQUIRE(g->user_mlp && g->item_mlp, "dense table mode needs gradient tables");
    if (m.mf_dim > 0) MR_REQUIRE(g->user_gmf && g->item_gmf, "dense table mode needs GMF gradient tables");
  } else {
    MR_REQUIRE(m.l2[0] == 0.f, "layers_l2reg[0] != 0 makes embedding gradients dense; use MR_TABLES_DENSE");
  }
  return MR_OK;
}

// ---- train step ----------------------------------------------------------------------------------------------------
// Every launch-sequence choice of a step, made once by TrainStep::plan.  The tower runs as the projected tensor-core
// tower's fused kernel, the tensor-core sub-batch loop, the default tower's projected step on CUDA cores, or the
// generic tile kernel.
enum { TRAIN_TC_FUSED = 0, TRAIN_TC = 1, TRAIN_SMALL = 2, TRAIN_TILES = 3 };
struct TrainPlan {
  int path;             // TRAIN_*
  bool grouped;         // one user per group: the user side runs once per group (promise checked on the device)
  bool proj, uproj;     // item / user half of the first layer once per item / user (item_proj_ok, user_proj_ok)
  int64_t n_user_rows;  // staged user-gradient rows: one per group or one per row
  // TRAIN_TC_FUSED: dz of every row, behind the item staging rows, which then hold dZ1 only (L1 wide); the item-side
  // reduction forms the GMF item gradient from it (GmfRows).  NULL on the other paths: they stage [dZ1 | d gmf_i].
  float* dz_rows;
  // where the segmented reductions put the MLP part of their rows (dense table mode): the per-user / per-item sums
  // of dZ[1] (L1 wide) on a projected side, the gradient table otherwise
  float *user_sums, *item_sums;
  TcWs tc;              // TRAIN_TC_FUSED, TRAIN_TC: Pi / Si and Pu / Su NULL on a side that is not projected
  SmallWs small;        // TRAIN_SMALL
};

// One train step: the call's arguments, workspace, streams and plan.  Its parts run as prologue, tower, epilogue.
struct TrainStep {
  const MrModel& m;
  const MrOptState& opt;
  const MrGrads& grads;
  const int32_t *users, *items;
  const float* labels;
  int64_t B;
  int group, k, flags;
  float inv_batch;
  float* step_out;
  TrainWs t;
  SideStream* side;  // NULL when it could not be created: its work then runs on st
  cudaStream_t st;
  TrainPlan p;

  TrainPlan plan() const;
  int prologue() const;
  int tower_tc() const;
  int tc_sub_batches() const;
  int tc_grouped_first_layer_backward(int64_t r0, int64_t r1) const;
  template <class UserTables, class ItemTables>
  int projected_backward(UserTables user_tables, ItemTables item_tables) const;
  int tower_small() const;
  int tower_tiles() const;
  int epilogue() const;
};

TrainPlan TrainStep::plan() const {
  const bool dense = opt.table_mode == MR_TABLES_DENSE;
  const bool users_grouped = (flags & MR_TRAIN_USERS_GROUPED) != 0;
  TrainPlan q{};
  if (use_tc(m)) {
    q.grouped = users_grouped && tc_grouped_ok(m, B, group);
    q.proj = q.grouped && dense && item_proj_ok(m, B);
    q.uproj = q.proj && user_proj_ok(m, B, group);
    // The per-row work of the projected step in ONE kernel (tc_fused.cu): H1, the second layer forward, the head,
    // the second layer's weight gradient and backward, the staged rows and their group sums never leave the SM.
    const bool fused = q.uproj && m.fused_train != MR_FUSED_OFF && fused_train_supported(m, group);
    q.path = fused ? TRAIN_TC_FUSED : TRAIN_TC;
    if (fused) q.dz_rows = t.stage_i + (size_t)B * m.L[1];
    q.tc = carve_tc(m, true, B, t.tc_ws);
    if (!q.proj) q.tc.Pi = q.tc.Si = nullptr;
    if (!q.uproj) q.tc.Pu = q.tc.Su = nullptr;
  } else if (users_grouped && dense && small_proj_ok(m, B, group)) {
    // default tower: both projections on CUDA cores, thread per group (small_tower.cu)
    q.path = TRAIN_SMALL;
    q.grouped = q.proj = q.uproj = true;
    q.small = carve_small(m, t.small_ws);
  } else {
    q.path = TRAIN_TILES;
  }
  const bool small = q.path == TRAIN_SMALL;
  q.user_sums = q.uproj ? (small ? q.small.Su : q.tc.Su) : grads.user_mlp;
  q.item_sums = q.proj ? (small ? q.small.Si : q.tc.Si) : grads.item_mlp;
  q.n_user_rows = q.grouped ? B / group : B;
  return q;
}

// The l2 penalty, then on the side stream the clears of what the segmented reductions add into, the group check and
// the stable sorts of the ids (the reductions' keys): they do not depend on the tower, so they run under it (phase
// timing then sees only the launch cost of this block on the caller's stream).
int TrainStep::prologue() const {
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u;
  int rc = MR_OK;
  prof_mark(MR_PHASE_MISC, st);
  MR_CUDA(cudaMemsetAsync(t.flags, 0, 256, st));
  MR_CUDA(cudaMemsetAsync(step_out, 0, MR_STEP_OUT_FLOATS * sizeof(float), st));
  // l2 penalty of the step's weights: first, so that nothing reads the tables after grads->user_tables_ready
  if (any_l2(m)) {
    float* pen = step_out + MR_OUT_L2_PENALTY;
    if (m.l2[0] != 0.f) {
      rc = launch_l2_penalty(m.user_mlp, (int64_t)m.num_users * d_u, m.l2[0], pen, st);
      if (rc == MR_OK) rc = launch_l2_penalty(m.item_mlp, (int64_t)m.num_items * d_i, m.l2[0], pen, st);
      if (rc == MR_OK && m.mf_dim > 0) rc = launch_l2_penalty(m.user_gmf, (int64_t)m.num_users * m.mf_dim, m.l2[0], pen, st);
      if (rc == MR_OK && m.mf_dim > 0) rc = launch_l2_penalty(m.item_gmf, (int64_t)m.num_items * m.mf_dim, m.l2[0], pen, st);
      if (rc != MR_OK) return rc;
    }
    for (int l = 1; l < m.n_layers; ++l)
      if (m.l2[l] != 0.f) {
        rc = launch_l2_penalty(m.W[l], (int64_t)m.L[l - 1] * m.L[l], m.l2[l], pen, st);
        if (rc != MR_OK) return rc;
      }
  }
  cudaStream_t ss = st;
  if (side != nullptr) {
    MR_CUDA(cudaEventRecord(side->fork, st));
    MR_CUDA(cudaStreamWaitEvent(side->stream, side->fork, 0));
    ss = side->stream;
  }
  prof_mark(MR_PHASE_SORT, st);
  if (opt.table_mode == MR_TABLES_DENSE) {  // (on a projected side a GEMM on the sums then writes the MLP table whole)
    MR_CUDA(cudaMemsetAsync(p.user_sums, 0, (size_t)m.num_users * (p.uproj ? m.L[1] : d_u) * sizeof(float), ss));
    MR_CUDA(cudaMemsetAsync(p.item_sums, 0, (size_t)m.num_items * (p.proj ? m.L[1] : d_i) * sizeof(float), ss));
    if (m.mf_dim > 0) {
      MR_CUDA(cudaMemsetAsync(grads.user_gmf, 0, (size_t)m.num_users * m.mf_dim * sizeof(float), ss));
      MR_CUDA(cudaMemsetAsync(grads.item_gmf, 0, (size_t)m.num_items * m.mf_dim * sizeof(float), ss));
    }
  }
  if (p.grouped) {
    rc = launch_check_grouped(users, B, group, t.flags + 1, ss);
    if (rc == MR_OK) rc = launch_group_heads(users, B / group, group, t.group_users, ss);
    if (rc != MR_OK) return rc;
  }
  rc = sort_row_ids(p.grouped ? t.group_users : users, p.n_user_rows, m.num_users, t.sorted_keys, t.sorted_index,
                    t.sort_ws, t.sort_ws_bytes, ss);
  if (rc == MR_OK)
    rc = sort_row_ids(items, B, m.num_items, t.sorted_keys_i, t.sorted_index_i, t.sort_ws, t.sort_ws_bytes, ss);
  if (rc != MR_OK) return rc;
  if (side != nullptr) MR_CUDA(cudaEventRecord(side->join, ss));
  prof_mark(MR_PHASE_MISC, st);
  return MR_OK;
}

// Backward of the projected first layer after the tower's per-row work: segment sums of the staged rows [dZ1 | GMF row
// gradient] per item (the GMF part straight into its gradient table), then the tower's GEMMs over the item table on
// them (item_tables, caller's stream); the same per user when the user half is projected (user_tables).  The two
// chains are independent (disjoint buffers and columns of the dense partial rows): the user chain runs on the side
// stream, so the latency-bound upper levels of one run under the other, and the user-side gradient tables (83 % of the table-gradient bytes at the ML-20M shape) are final while
// the item side is still being reduced: a data-parallel caller starts their all-reduce on grads->user_tables_ready.
// A data-parallel caller may also update the user tables from those events on, so they wait for the step's last read
// of the user GMF table: with GmfRows (TRAIN_TC_FUSED) that is the item-side reduction's level 0.
template <class UserTables, class ItemTables>
int TrainStep::projected_backward(UserTables user_tables, ItemTables item_tables) const {
  if (side != nullptr) MR_CUDA(cudaStreamWaitEvent(st, side->join, 0));  // sorted keys, cleared sums and GMF tables
  const bool gmf_formed = p.dz_rows != nullptr;
  const GmfRows gmf{p.dz_rows, t.group_users, group, m.num_users, m.w_out, m.user_gmf};
  const cudaEvent_t gmf_ready = (cudaEvent_t)grads.user_gmf_ready, tables_ready = (cudaEvent_t)grads.user_tables_ready;
  RowUpdate u{};
  u.mode = MR_TABLES_DENSE;
  u.optimizer = opt.optimizer;
  u.d0 = m.L[1];
  u.d1 = m.mf_dim;
  cudaStream_t su = st;
  if (p.uproj) {
    if (side != nullptr) {
      MR_CUDA(cudaEventRecord(side->fork2, st));
      MR_CUDA(cudaStreamWaitEvent(side->stream, side->fork2, 0));
      su = side->stream;
    }
    u.num_rows = m.num_users;
    u.g0 = p.user_sums;
    u.g1 = grads.user_gmf;
    int rc = launch_segreduce(t.sorted_keys, t.sorted_index, p.n_user_rows, t.stage_u, u, t.seg_ws_u, t.seg_ws_u_bytes, su);
    if (rc != MR_OK) return rc;
    // user_gmf: gradients final, table last read by the tower (or by the item side's level 0 below)
    if (gmf_ready != nullptr) {
      if (!gmf_formed) MR_CUDA(cudaEventRecord(gmf_ready, su));
      else if (side != nullptr) MR_CUDA(cudaEventRecord(side->user_sums, su));
    }
  }
  prof_mark(MR_PHASE_SEGREDUCE, st);
  u.num_rows = m.num_items;
  u.g0 = p.item_sums;
  u.g1 = grads.item_gmf;
  int rc = launch_segreduce(t.sorted_keys_i, t.sorted_index_i, B, t.stage_i, u, t.seg_ws, t.seg_ws_bytes, st,
                            gmf_formed ? &gmf : nullptr, [&]() -> int {
                              if (!gmf_formed) return MR_OK;
                              if (gmf_ready != nullptr) {
                                if (side != nullptr) MR_CUDA(cudaStreamWaitEvent(st, side->user_sums, 0));
                                MR_CUDA(cudaEventRecord(gmf_ready, st));
                              }
                              if (tables_ready != nullptr && side != nullptr) MR_CUDA(cudaEventRecord(side->gmf_read, st));
                              return MR_OK;
                            });
  if (rc != MR_OK) return rc;
  if (p.uproj) {
    rc = user_tables(su);  // the step's last read of the user table, so it goes before the event
    if (rc != MR_OK) return rc;
    if (tables_ready != nullptr) {
      if (gmf_formed && side != nullptr) MR_CUDA(cudaStreamWaitEvent(su, side->gmf_read, 0));
      MR_CUDA(cudaEventRecord(tables_ready, su));
    }
    if (side != nullptr) MR_CUDA(cudaEventRecord(side->join2, su));
  }
  rc = item_tables();
  if (rc != MR_OK) return rc;
  if (p.uproj && side != nullptr) MR_CUDA(cudaStreamWaitEvent(st, side->join2, 0));
  return MR_OK;
}

// First layer's backward of a grouped sub-batch, rows [r0, r1): the item half per row, the user half per group on
// S1 = the group sums of dZ[1].  A projected half only stages its rows here; it runs on the per-item / per-user sums.
int TrainStep::tc_grouped_first_layer_backward(int64_t r0, int64_t r1) const {
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u, f = m.mf_dim;
  const TcWs& tw = p.tc;
  const int64_t ng = (r1 - r0) / group, g0 = r0 / group;
  int rc = MR_OK;
  prof_mark(MR_PHASE_MISC, st);
  if (p.uproj)
    rc = launch_group_sum_rows(t.stage_i + (size_t)r0 * (d_i + f), ng, group, m.L[1],
                               t.stage_u + (size_t)g0 * (d_u + f), st, d_i + f, d_u + f);
  else if (p.proj)  // (columns [0, L1) of the item staging rows, stride d_i + f)
    rc = launch_group_sum_rows(t.stage_i + (size_t)r0 * (d_i + f), ng, group, m.L[1], tw.S1, st, d_i + f);
  else
    rc = launch_group_sum_rows(tw.dZ[1], ng, group, m.L[1], tw.S1, st);
  if (rc != MR_OK) return rc;
  prof_mark(MR_PHASE_TC_WGRAD, st);
  if (!p.proj) {
    TcWgradArgs wi{};
    wi.gather = true;
    wi.item_tab = m.item_mlp;
    wi.items = items;
    wi.num_users = m.num_users;
    wi.num_items = m.num_items;
    wi.d_u = 0;
    wi.z = tw.dZ[1];
    wi.Fa = d_i;
    wi.Fb = m.L[1];
    wi.rows = r1 - r0;
    wi.row0 = r0;
    wi.dw_partial = t.dense_partial + (m.W[1] - m.dense) + (size_t)d_u * m.L[1];
    wi.db_partial = t.dense_partial + (m.b[1] - m.dense);
    wi.partial_stride = t.dense_stride;
    rc = launch_tc_wgrad(wi, st);
    if (rc != MR_OK) return rc;
  }
  if (p.uproj) return MR_OK;
  TcWgradArgs wu{};
  wu.gather = true;
  wu.user_tab = m.user_mlp;
  wu.users = users;
  wu.num_users = m.num_users;
  wu.num_items = m.num_items;
  wu.d_u = d_u;
  wu.user_mul = group;
  wu.z = tw.S1;
  wu.Fa = d_u;
  wu.Fb = m.L[1];
  wu.rows = ng;
  wu.row0 = g0;
  wu.dw_partial = t.dense_partial + (m.W[1] - m.dense);
  // the bias gradient (column sums of dZ[1]) comes with the item half, or from the group sums when the item half runs
  // per item
  wu.db_partial = p.proj ? t.dense_partial + (m.b[1] - m.dense) : nullptr;
  wu.partial_stride = t.dense_stride;
  rc = launch_tc_wgrad(wu, st);
  if (rc != MR_OK) return rc;
  prof_mark(MR_PHASE_TC_DENSE_BWD, st);
  if (!p.proj) {
    TcDenseArgs bi{};
    bi.a_dense = tw.dZ[1];
    bi.d_u = 0;  // every output column belongs to the item row
    bi.b_packed = tw.pack_bi;
    bi.N = d_i;
    bi.K = m.L[1];
    bi.rows = r1 - r0;
    bi.row0 = r0;
    bi.epilogue = TC_EPI_STAGE;
    bi.stage_u = t.stage_u;
    bi.stage_i = t.stage_i;
    bi.su = d_u + f;
    bi.si = d_i + f;
    rc = launch_tc_dense(bi, st);
    if (rc != MR_OK) return rc;
  }
  TcDenseArgs bu{};
  bu.a_dense = tw.S1;
  bu.d_u = d_u;  // every output column belongs to the user row of the group
  bu.b_packed = tw.pack_bu;
  bu.N = d_u;
  bu.K = m.L[1];
  bu.rows = ng;
  bu.row0 = g0;
  bu.epilogue = TC_EPI_STAGE;
  bu.stage_u = t.stage_u;
  bu.stage_i = t.stage_i;
  bu.su = d_u + f;
  bu.si = d_i + f;
  return launch_tc_dense(bu, st);
}

// Per sub-batch: forward layers -> head -> per layer weight gradient + backward.
int TrainStep::tc_sub_batches() const {
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u, n = m.n_layers, f = m.mf_dim;
  const TcWs& tw = p.tc;
  const int gdiv = p.grouped ? group : 0;
  const int64_t sb = tc_sub_batch(B);
  for (int64_t r0 = 0; r0 < B; r0 += sb) {
    const int64_t r1 = r0 + sb < B ? r0 + sb : B;
    prof_mark(MR_PHASE_TC_DENSE_FWD, st);
    int rc = tc_forward_rows(m, tw, users, items, 1, r0, r1, st, gdiv);
    if (rc != MR_OK) return rc;
    prof_mark(MR_PHASE_HEAD, st);
    HeadArgs h{};
    h.model = &m;
    h.h_last = tw.H[n - 1];
    h.users = users;
    h.items = items;
    h.labels = labels;
    h.rows = r1 - r0;
    h.row0 = r0;
    h.user_div = 1;
    h.group = gdiv;
    h.inv_batch = inv_batch;
    h.probs = t.probs;
    h.dz_last = tw.dZ[n - 1];
    h.stage_u = t.stage_u;
    h.stage_i = t.stage_i;
    h.head_partial = tw.head_partial;
    h.flags = t.flags;
    rc = launch_head(h, st);
    if (rc != MR_OK) return rc;
    for (int l = n - 1; l >= (p.grouped ? 2 : 1); --l) {
      prof_mark(MR_PHASE_TC_WGRAD, st);
      TcWgradArgs w{};
      w.gather = (l == 1);
      w.a_dense = (l == 1) ? nullptr : tw.H[l - 1];
      w.user_tab = m.user_mlp;
      w.item_tab = m.item_mlp;
      w.users = users;
      w.items = items;
      w.num_users = m.num_users;
      w.num_items = m.num_items;
      w.d_u = d_u;
      w.z = tw.dZ[l];
      w.Fa = m.L[l - 1];
      w.Fb = m.L[l];
      w.rows = r1 - r0;
      w.row0 = r0;
      w.dw_partial = t.dense_partial + (m.W[l] - m.dense);
      w.db_partial = t.dense_partial + (m.b[l] - m.dense);
      w.partial_stride = t.dense_stride;
      rc = launch_tc_wgrad(w, st);
      if (rc != MR_OK) return rc;
      prof_mark(MR_PHASE_TC_DENSE_BWD, st);
      TcDenseArgs a{};
      a.gather = false;
      a.a_dense = tw.dZ[l];
      a.d_u = d_u;
      a.b_packed = tw.pack_b[l];
      a.N = m.L[l - 1];
      a.K = m.L[l];
      a.rows = r1 - r0;
      a.row0 = r0;
      if (l - 1 >= 1) {
        a.epilogue = TC_EPI_MASK;
        a.mask_bits = tw.bits[l - 1];
        a.out = tw.dZ[l - 1];
        if (p.proj && l - 1 == 1) {  // dZ[1] goes straight into the item staging rows: the keys of its per-item sums
          a.out = t.stage_i + (size_t)r0 * (d_i + f);
          a.out_ld = d_i + f;
        }
      } else {
        a.epilogue = TC_EPI_STAGE;
        a.stage_u = t.stage_u;
        a.stage_i = t.stage_i;
        a.su = d_u + f;
        a.si = d_i + f;
      }
      rc = launch_tc_dense(a, st);
      if (rc != MR_OK) return rc;
    }
    if (p.grouped) {
      rc = tc_grouped_first_layer_backward(r0, r1);
      if (rc != MR_OK) return rc;
    }
  }
  return MR_OK;
}

// ---- tensor-core tower: the fused kernel or the sub-batch loop, then the projected first layer's backward on its
// per-item / per-user sums and the reductions of the dense partial rows
int TrainStep::tower_tc() const {
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u, n = m.n_layers, f = m.mf_dim;
  const TcWs& tw = p.tc;
  const bool fused = p.path == TRAIN_TC_FUSED;
  const int P = sm_count();  // rows of the partial buffer = CTAs of the weight-gradient kernel
  int rc = MR_OK;
  MR_CUDA(cudaMemsetAsync(t.dense_partial, 0, (size_t)P * t.dense_stride * sizeof(float), st));
  if (!fused) {  // (the fused kernel packs its own operand image of W[2] and keeps the head's sums itself)
    MR_CUDA(cudaMemsetAsync(tw.head_partial, 0, head_partial_floats(m) * sizeof(float), st));
    for (int l = p.grouped ? 2 : 1; l < n; ++l) {
      rc = launch_pack_weights(m.W[l], m.L[l - 1], m.L[l], 0, tw.pack_f[l], st);
      if (rc == MR_OK) rc = launch_pack_weights(m.W[l], m.L[l - 1], m.L[l], 1, tw.pack_b[l], st);
      if (rc != MR_OK) return rc;
    }
  }
  if (p.grouped) {  // W[1] is (L0, L1) row-major: rows [0, d_u) multiply the user row, rows [d_u, L0) the item row
    const float* Wu = m.W[1];
    const float* Wi = m.W[1] + (size_t)d_u * m.L[1];
    rc = launch_pack_weights(Wu, d_u, m.L[1], 0, tw.pack_fu, st);
    if (rc == MR_OK) rc = launch_pack_weights(Wi, d_i, m.L[1], 0, tw.pack_fi, st);
    if (rc == MR_OK) rc = launch_pack_weights(Wu, d_u, m.L[1], 1, tw.pack_bu, st);
    if (rc == MR_OK) rc = launch_pack_weights(Wi, d_i, m.L[1], 1, tw.pack_bi, st);
    if (rc != MR_OK) return rc;
  }
  if (p.proj) {
    prof_mark(MR_PHASE_TC_DENSE_FWD, st);
    rc = tc_project_table(m, m.item_mlp, m.num_items, d_i, tw.pack_fi, tw.Pi, st);
    if (rc == MR_OK && p.uproj) rc = tc_project_users(m, tw, st);
    if (rc != MR_OK) return rc;
  }
  int fused_grid = 0;
  if (fused) {
    prof_mark(MR_PHASE_FUSED_TILE, st);
    FusedTrainArgs fa{};
    fa.Pi = tw.Pi;
    fa.Pu = tw.Pu;
    fa.user_gmf = m.user_gmf;
    fa.item_gmf = m.item_gmf;
    fa.users = users;
    fa.items = items;
    fa.labels = labels;
    fa.num_users = m.num_users;
    fa.num_items = m.num_items;
    fa.rows = B;
    fa.group = group;
    fa.W2 = m.W[2];
    fa.w2_image = tw.w2_image;
    fa.b2 = m.b[2];
    fa.w_out = m.w_out;
    fa.b_out = m.b_out;
    fa.inv_batch = inv_batch;
    fa.probs = t.probs;
    fa.stage_i = t.stage_i;
    fa.dz_rows = p.dz_rows;
    fa.stage_u = t.stage_u;
    fa.si = m.L[1];  // dZ1 only (p.dz_rows)
    fa.su = d_u + f;
    fa.partial = t.dense_partial;
    fa.partial_stride = t.dense_stride;
    fa.off_w2 = m.W[2] - m.dense;
    fa.off_b2 = m.b[2] - m.dense;
    fa.off_wout = m.w_out - m.dense;
    fa.off_bout = m.b_out - m.dense;
    fa.loss_partial = t.loss_partial;
    fa.flags = t.flags;
    rc = launch_fused_train(fa, st, &fused_grid);
  } else {
    rc = tc_sub_batches();
  }
  if (rc != MR_OK) return rc;
  if (p.proj) {
    float* dw1 = t.dense_partial + (m.W[1] - m.dense);
    rc = projected_backward(
        [&](cudaStream_t su) {
          return tc_table_backward(m, m.user_mlp, tw.Su, m.num_users, d_u, tw.pack_bu, grads.user_mlp, dw1,
                                   t.dense_partial + (m.b[1] - m.dense), t.dense_stride, false, su);
        },
        [&] {
          return tc_table_backward(m, m.item_mlp, tw.Si, m.num_items, d_i, tw.pack_bi, grads.item_mlp,
                                   dw1 + (size_t)d_u * m.L[1], nullptr, t.dense_stride, true, st);
        });
    if (rc != MR_OK) return rc;
  }
  prof_mark(MR_PHASE_MISC, st);
  if (fused)  // (its d w_out / d b_out partials sit in the CTAs' rows of the dense partial buffer already)
    rc = launch_sum_partials(t.loss_partial, fused_grid, step_out + MR_OUT_LOSS_SUM, st);
  else
    rc = launch_head_reduce(m, tw.head_partial, t.dense_partial + (m.w_out - m.dense),
                            t.dense_partial + (m.b_out - m.dense), step_out + MR_OUT_LOSS_SUM, st);
  if (rc != MR_OK) return rc;
  return launch_dense_reduce(m, t.dense_partial, t.dense_stride, P, grads.dense, st, !(flags & MR_TRAIN_NO_DENSE_L2));
}

// ---- default tower, projected: Pi / Pu over the tables, one thread-per-group kernel for everything per row,
// segment sums of the staged rows per item / per user, then the first layer's backward on the sums
int TrainStep::tower_small() const {
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u, L1 = m.L[1], cap = max_tile_ctas();
  const SmallWs& w = p.small;
  const float* W1u = m.W[1];
  const float* W1i = m.W[1] + (size_t)d_u * L1;
  MR_CUDA(cudaMemsetAsync(t.dense_partial, 0, (size_t)cap * t.dense_stride * sizeof(float), st));
  prof_mark(MR_PHASE_TC_DENSE_FWD, st);
  int rc = launch_small_rows_gemm(m.item_mlp, m.num_items, d_i, W1i, L1, L1, false, nullptr, w.Pi, st);
  if (rc == MR_OK) rc = launch_small_rows_gemm(m.user_mlp, m.num_users, d_u, W1u, L1, L1, false, m.b[1], w.Pu, st);
  if (rc != MR_OK) return rc;
  SmallTowerArgs a{};
  a.model = &m;
  a.Pi = w.Pi;
  a.Pu = w.Pu;
  a.users = users;
  a.items = items;
  a.labels = labels;
  a.B = B;
  a.inv_batch = inv_batch;
  a.probs = t.probs;
  a.stage_i = t.stage_i;
  a.stage_u = t.stage_u;
  a.dense_partial = t.dense_partial;
  a.dense_stride = t.dense_stride;
  a.loss_partial = t.loss_partial;
  a.flags = t.flags;
  a.max_ctas = cap;
  int grid = 0, grid_i = 0, grid_u = 0;
  prof_mark(MR_PHASE_FUSED_TILE, st);
  rc = launch_small_tower_train(a, st, &grid);
  if (rc != MR_OK) return rc;
  rc = projected_backward(
      [&](cudaStream_t su) {  // d E_user = Su . W1u^T, d W1u = E_user^T . Su, d b1 = colsum(Su)
        int r = launch_small_rows_gemm(w.Su, m.num_users, L1, W1u, L1, d_u, true, nullptr, grads.user_mlp, su);
        if (r == MR_OK)
          r = launch_small_table_wgrad(m.user_mlp, w.Su, m.num_users, t.dense_partial + (W1u - m.dense),
                                       t.dense_partial + (m.b[1] - m.dense), t.dense_stride, cap, su, &grid_u);
        return r;
      },
      [&] {
        prof_mark(MR_PHASE_TC_DENSE_BWD, st);  // d E_item = Si . W1i^T over the table
        int r = launch_small_rows_gemm(w.Si, m.num_items, L1, W1i, L1, d_i, true, nullptr, grads.item_mlp, st);
        if (r != MR_OK) return r;
        prof_mark(MR_PHASE_TC_WGRAD, st);  // d W1i = E_item^T . Si
        return launch_small_table_wgrad(m.item_mlp, w.Si, m.num_items, t.dense_partial + (W1i - m.dense), nullptr,
                                        t.dense_stride, cap, st, &grid_i);
      });
  if (rc != MR_OK) return rc;
  prof_mark(MR_PHASE_MISC, st);
  const int nrows = grid > grid_i ? (grid > grid_u ? grid : grid_u) : (grid_i > grid_u ? grid_i : grid_u);
  rc = launch_dense_reduce(m, t.dense_partial, t.dense_stride, nrows, grads.dense, st, !(flags & MR_TRAIN_NO_DENSE_L2));
  if (rc != MR_OK) return rc;
  return launch_sum_partials(t.loss_partial, grid, step_out + MR_OUT_LOSS_SUM, st);
}

// ---- generic tile kernel: the whole per-row step on CUDA cores
int TrainStep::tower_tiles() const {
  int rc = launch_transpose_kernels(m, t.wt, st);
  if (rc != MR_OK) return rc;
  TileLaunch a{};
  a.model = &m;
  a.train = true;
  a.wt = t.wt;
  a.users = users;
  a.items = items;
  a.labels = labels;
  a.B = B;
  a.user_div = 1;
  a.inv_batch = inv_batch;
  a.probs = t.probs;
  a.loss_partial = t.loss_partial;
  a.dense_partial = t.dense_partial;
  a.dense_stride = t.dense_stride;
  a.stage_u = t.stage_u;
  a.stage_i = t.stage_i;
  a.flags = t.flags;
  int grid = 0;
  prof_mark(MR_PHASE_TILE_TRAIN, st);
  rc = launch_neumf_tiles(a, st, &grid);
  prof_mark(MR_PHASE_MISC, st);
  if (rc != MR_OK) return rc;
  rc = launch_dense_reduce(m, t.dense_partial, t.dense_stride, grid, grads.dense, st, !(flags & MR_TRAIN_NO_DENSE_L2));
  if (rc != MR_OK) return rc;
  return launch_sum_partials(t.loss_partial, grid, step_out + MR_OUT_LOSS_SUM, st);
}

// The bad-id flag, the ranking of grouped batches, the embedding rows of the sides not projected (stable sort by row
// id, segmented reduce in batch order, row update) and, unless a projected user side recorded them, the events.
int TrainStep::epilogue() const {
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u;
  int rc = MR_OK;
  if (side != nullptr) MR_CUDA(cudaStreamWaitEvent(st, side->join, 0));  // sorts and the group check are done
  flag_to_float_kernel<<<1, 1, 0, st>>>(t.flags, step_out + MR_OUT_BAD_IDS);
  MR_LAUNCH_CHECK("flag_to_float_kernel");

  if (group > 0) {
    prof_mark(MR_PHASE_RANK, st);
    // label column = argmax of the group's labels (model.py:447-448): any layout of the positive is ranked right
    rc = launch_rank_scores(t.probs, B / group, group, k, nullptr, nullptr, t.pos, step_out + MR_OUT_HIT_SUM,
                            t.rank_partials, st, labels);
    if (rc != MR_OK) return rc;
  }
  prof_mark(MR_PHASE_MISC, st);

  RowUpdate u{};
  u.mode = opt.table_mode;
  u.optimizer = opt.optimizer;
  u.lr = opt.lr;
  u.lr_t = opt.optimizer == MR_OPT_ADAM ? adam_lr_t(opt, opt.iterations + 1) : opt.lr;
  u.beta_1 = opt.beta_1;
  u.beta_2 = opt.beta_2;
  u.epsilon = opt.epsilon;
  // users
  u.d0 = d_u;
  u.d1 = m.mf_dim;
  u.num_rows = m.num_users;
  u.p0 = m.user_mlp; u.m0 = opt.m_user_mlp; u.v0 = opt.v_user_mlp; u.g0 = grads.user_mlp;
  u.p1 = m.user_gmf; u.m1 = opt.m_user_gmf; u.v1 = opt.v_user_gmf; u.g1 = grads.user_gmf;
  if (!p.uproj) {
    prof_mark(MR_PHASE_SEGREDUCE, st);
    rc = launch_segreduce(t.sorted_keys, t.sorted_index, p.n_user_rows, t.stage_u, u, t.seg_ws, t.seg_ws_bytes, st);
    if (rc != MR_OK) return rc;
  }
  // items
  u.d0 = d_i;
  u.num_rows = m.num_items;
  u.p0 = m.item_mlp; u.m0 = opt.m_item_mlp; u.v0 = opt.v_item_mlp; u.g0 = grads.item_mlp;
  u.p1 = m.item_gmf; u.m1 = opt.m_item_gmf; u.v1 = opt.v_item_gmf; u.g1 = grads.item_gmf;
  if (!p.proj) {
    prof_mark(MR_PHASE_SEGREDUCE, st);
    rc = launch_segreduce(t.sorted_keys_i, t.sorted_index_i, B, t.stage_i, u, t.seg_ws, t.seg_ws_bytes, st);
  }
  if (!p.uproj) {  // the user side's gradients are final only now
    if (grads.user_gmf_ready != nullptr) MR_CUDA(cudaEventRecord((cudaEvent_t)grads.user_gmf_ready, st));
    if (grads.user_tables_ready != nullptr) MR_CUDA(cudaEventRecord((cudaEvent_t)grads.user_tables_ready, st));
  }
  prof_mark(-1, st);
  return rc;
}

// ---- evaluation: one plan per scoring call ---------------------------------------------------------------
// Rows per launch of mr_rank_eval's tensor-core tower: whole groups and whole 128-row tiles, at most 2^22 rows (the
// ML-20M sweep of 13.8 M rows: 14 launches of 2^20 rows 4.60 ms, 7 of 2^21 4.41 ms, 4 of 2^22 4.33 ms).
static int64_t eval_sub_batch(int group) {
  int64_t a = 128, b = group;
  while (b) { const int64_t t = a % b; a = b; b = t; }
  const int64_t l = (int64_t)128 / a * group;  // lcm(128, group)
  const int64_t cap = kEvalSubBatchCap;
  return l > cap ? 0 : cap / l * l;
}

static bool eval_fused_ok(const MrModel& m, int group) {
  return use_tc(m) && (head_rank_supported(m) || (m.n_layers >= 3 && head_rank_takes_dot(m, group))) && m.n_layers >= 2 &&
         group >= 2 && group <= 256 && eval_sub_batch(group) > 0;
}

// Catalogue calls score in chunks of whole users: about kEvalSubBatchCap rows (the ranking eval's launch size), at
// least one user, and at most kCatalogueMaxChunkUsers so that the selection's per-slice lists stay bounded when the
// catalogue is tiny.
constexpr int64_t kCatalogueMaxChunkUsers = 16384;

static int64_t catalogue_chunk_users(int32_t N) {
  int64_t c = kEvalSubBatchCap / (N < 1 ? 1 : N);
  if (c > kCatalogueMaxChunkUsers) c = kCatalogueMaxChunkUsers;
  return c < 1 ? 1 : c;
}

// The tower an eval call scores with: the tensor-core tower with the first layer split into its user half Zu and its
// item half (Pi, or the gathered item rows), the default tower's projected tables on CUDA cores (small_tower.cu), or
// the plain forward (mr_neumf_forward).
enum { EVAL_TC = 0, EVAL_SMALL = 1, EVAL_FORWARD = 2 };
// The shape of the call: G groups of `group` rows with one user each (mr_rank_eval), chunks of C users against the
// whole catalogue (catalogue calls, group = num_items), or U ragged lists of nnz rows in all (mr_rank_lists).
enum { SCORE_GROUPS = 0, SCORE_CATALOGUE = 1, SCORE_LISTS = 2 };
struct EvalPlan {
  int tower;           // EVAL_*
  bool proj;           // Pi = E_item . W1[item rows] over the item table (always on EVAL_SMALL)
  bool head_dot;       // EVAL_TC: the last hidden layer ends in its dot with w_out[MLP columns] (one float per row) and
                       // the head adds the GMF term; else the head reads the last layer whole
  bool call_users;     // the user half once per call over the call's users (SCORE_LISTS: Zu, or Pu of the gathered
                       // rows); else Zu per launch, one row per group, or Pu over the user table
  int64_t user_rows;   // rows of Zu (EVAL_TC) or Pu (EVAL_SMALL)
  int64_t sb;          // rows per scoring launch (EVAL_TC; SCORE_LISTS); EVAL_FORWARD: rows per forward call
};

// Every launch-sequence choice of an eval call, made once.  users / group / rows: G, group, G * group (SCORE_GROUPS);
// C, num_items, C * num_items (SCORE_CATALOGUE); U, -, nnz (SCORE_LISTS).  fused_head: mr_rank_eval's tensor-core
// tower ends in the fused score + position head, which writes no ranks.  AUTO's row-count rules judge the call's rows,
// the catalogue's full chunk (so that the choice does not depend on how many users a call has), or for lists nothing:
// their sequence is a function of the model alone, so that a list's outputs do not depend on the other lists.
static EvalPlan eval_plan(const MrModel& m, int shape, int64_t users, int group, int64_t rows, bool fused_head = true) {
  const bool lists = shape == SCORE_LISTS;
  const int64_t auto_rows = shape == SCORE_CATALOGUE ? catalogue_chunk_users(m.num_items) * m.num_items : rows;
  EvalPlan p{};
  p.call_users = lists;
  const bool tc = shape == SCORE_GROUPS
                      ? fused_head && eval_fused_ok(m, group)
                      : m.n_layers >= 3 && catalogue_head_supported(m) && (lists ? item_proj_ok(m, 0, true) : use_tc(m));
  if (tc) {
    p.tower = EVAL_TC;
    // the catalogue's tower without Pi runs the unprojected grouped first layer
    p.proj = item_proj_ok(m, auto_rows, lists);
    p.head_dot = shape != SCORE_GROUPS || (m.n_layers >= 3 && head_rank_takes_dot(m, group));
  } else {
    p.tower = small_eval_ok(m, auto_rows, lists) ? EVAL_SMALL : EVAL_FORWARD;
    p.proj = p.tower == EVAL_SMALL;
  }
  const int64_t tiles = (rows + 127) / 128 * 128;
  if (lists) {  // the call's rows in whole tiles, up to the ranking eval's 2^22 -- or the forward's own 2^21
    const int64_t cap = p.tower == EVAL_FORWARD ? kTcSubBatchCap : kEvalSubBatchCap;
    p.sb = tiles < 128 ? 128 : (tiles < cap ? tiles : cap);
  } else if (shape == SCORE_GROUPS && tc) {
    p.sb = eval_sub_batch(group) < tiles ? eval_sub_batch(group) : tiles;
  } else {
    p.sb = rows;
  }
  if (lists) p.user_rows = users < 1 ? 1 : users;
  else p.user_rows = tc ? p.sb / group + 1 : m.num_users;
  return p;
}

struct EvalWs {
  TcWs t;            // EVAL_TC: the packed weights, Zu and H; Pi (proj); EVAL_SMALL: Pu
  float* Eu;         // EVAL_SMALL with call_users: the call's users' MLP rows
  void* fwd;         // EVAL_FORWARD: mr_neumf_forward's workspace
  size_t fwd_bytes;
  size_t total;
};

// The scoring workspace of a plan; the workspace queries take its size from here (ws = NULL).  H[1] exists only when
// the first layer writes it (with Pi the second layer's producers compute it), and H[n-1] holds one float per row when
// the plan ends in head_dot.
static EvalWs eval_carve(const MrModel& m, const EvalPlan& p, void* ws) {
  EvalWs w{};
  Carver cv(ws);
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u, L1 = m.L[1];
  if (p.tower == EVAL_TC) {
    w.t.pack_fu = cv.take<float>((size_t)2 * d_u * L1);
    w.t.pack_fi = cv.take<float>((size_t)2 * d_i * L1);
    for (int l = 2; l < m.n_layers; ++l) w.t.pack_f[l] = cv.take<float>((size_t)2 * m.L[l - 1] * m.L[l]);
    w.t.Zu = cv.take<float>((size_t)p.user_rows * L1);
    for (int l = p.proj ? 2 : 1; l < m.n_layers; ++l)
      w.t.H[l] = cv.take<float>((size_t)p.sb * (p.head_dot && l == m.n_layers - 1 ? 1 : m.L[l]));
  }
  if (p.proj) w.t.Pi = cv.take<float>((size_t)m.num_items * L1);
  if (p.tower == EVAL_SMALL) {
    if (p.call_users) w.Eu = cv.take<float>((size_t)p.user_rows * d_u);
    w.t.Pu = cv.take<float>((size_t)p.user_rows * L1);
  }
  if (p.tower == EVAL_FORWARD) {
    w.fwd_bytes = mr_forward_workspace_bytes(&m, p.sb);
    w.fwd = cv.take<char>(w.fwd_bytes);
  }
  w.total = cv.off;
  return w;
}

// Once per call, what the plan's tower reads besides the tables: the packed weights (EVAL_TC), Pi, then the user half
// that is not per launch -- Pu over the user table or over the call's users (EVAL_SMALL), Zu of the call's users
// (EVAL_TC with call_users).  users: the call's users, p.user_rows of them when p.call_users.
static int eval_prepare(const MrModel& m, const EvalPlan& p, const EvalWs& w, const int32_t* users, cudaStream_t st) {
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u, L1 = m.L[1];
  const bool tc = p.tower == EVAL_TC;
  int rc = MR_OK;
  if (tc) {
    rc = launch_pack_weights(m.W[1], d_u, L1, 0, w.t.pack_fu, st);
    if (rc == MR_OK) rc = launch_pack_weights(m.W[1] + (size_t)d_u * L1, d_i, L1, 0, w.t.pack_fi, st);
    for (int l = 2; rc == MR_OK && l < m.n_layers; ++l) rc = launch_pack_weights(m.W[l], m.L[l - 1], m.L[l], 0, w.t.pack_f[l], st);
  }
  if (rc == MR_OK && p.proj) {
    prof_mark(MR_PHASE_TC_DENSE_FWD, st);
    rc = tc ? tc_project_table(m, m.item_mlp, m.num_items, d_i, w.t.pack_fi, w.t.Pi, st)
            : launch_small_rows_gemm(m.item_mlp, m.num_items, d_i, m.W[1] + (size_t)d_u * L1, L1, L1, false, nullptr,
                                     w.t.Pi, st);
  }
  if (rc != MR_OK) return rc;
  if (tc && p.call_users) return tc_user_half(m, w.t, users, 1, 0, p.user_rows, st);
  if (p.tower != EVAL_SMALL) return MR_OK;
  if (!p.call_users) return launch_small_rows_gemm(m.user_mlp, m.num_users, d_u, m.W[1], L1, L1, false, m.b[1], w.t.Pu, st);
  rc = launch_gather_rows(m.user_mlp, m.num_users, d_u, users, p.user_rows, w.Eu, st);  // NaN rows: bad users
  if (rc == MR_OK) rc = launch_small_rows_gemm(w.Eu, p.user_rows, d_u, m.W[1], L1, L1, false, m.b[1], w.t.Pu, st);
  return rc;
}

// ---- catalogue calls: every user against every item, in chunks of whole users --------------------------------
static int64_t clamp_users(int64_t U, int64_t C) { return U < 1 ? 1 : (U < C ? U : C); }

// Chunks of C users x M items (M = num_items: the catalogue).  The tower choices judge the catalogue's full chunk
// whatever M is (eval_plan), so an audience scores a pair with the launch sequence mr_catalogue_topk takes.
static EvalPlan catalogue_plan(const MrModel& m, int64_t C, int32_t M) {
  return eval_plan(m, SCORE_CATALOGUE, C, M, C * M);
}

// The sweep's workspace (chunks of C users x M items): the item of every row of a chunk, the chunk's probabilities, the
// chunk's user ids when the caller gives none (own_users), the scoring.
static size_t catalogue_sweep_bytes(const MrModel& m, int64_t C, int32_t M, bool own_users = false) {
  const size_t rows = (size_t)C * M;
  return align_up(rows * sizeof(int32_t), 256) + align_up(rows * sizeof(float), 256) +
         (own_users ? align_up((size_t)C * sizeof(int32_t), 256) : 0) +
         eval_carve(m, catalogue_plan(m, C, M), nullptr).total;
}

static int topk_check(int64_t U, int32_t N, int32_t k, int32_t excl_rows, const int64_t* excl_rowptr,
                      const int32_t* excl_items, const int32_t* targets, const int32_t* pos, const float* sums) {
  MR_REQUIRE(U >= 0 && N >= 1, "topk: bad U=%lld N=%d", (long long)U, N);
  MR_REQUIRE(k >= 1 && k <= MR_MAX_TOPK, "topk: k=%d out of [1,%d]", k, MR_MAX_TOPK);
  MR_REQUIRE(excl_rows >= 0 && (excl_rowptr == nullptr || excl_items != nullptr), "topk: bad exclusion lists");
  MR_REQUIRE(targets != nullptr || (pos == nullptr && sums == nullptr), "topk: pos / sums need targets");
  return MR_OK;
}

// The chunk loop of every serving query over users: per chunk of C users, select(u0, users in the chunk, the chunk's
// scores).  model == NULL: the scores are the caller's U x N matrix, read at scores + u0 * N under MR_PHASE_RANK.
// Otherwise they are the model's probabilities of every (user, item) pair through the plan's tower, each chunk's
// selection under MR_PHASE_RANK.  The items are the catalogue (N = num_items), or with `items` the list items[0, N)
// (chunk row r pairs user r / N with items[r % N]; the item half of the first layer is still projected once over the
// whole table).  users == NULL: user u is id u.  The probabilities go to scores + u0 * N when scores is given, else to
// the sweep's buffer (C x N).  ws: catalogue_sweep_bytes(m, C, N, users == NULL) bytes.  Every model query scores
// through here, so a pair's probability is the same in all of them by construction.
template <class Select>
static int catalogue_sweep(const MrModel* model, const int32_t* users, int64_t U, int64_t C, int32_t N, float* scores,
                           void* ws, cudaStream_t st, Select select, const int32_t* items = nullptr) {
  int rc = MR_OK;
  if (model == nullptr) {
    prof_mark(MR_PHASE_RANK, st);
    for (int64_t u0 = 0; u0 < U && rc == MR_OK; u0 += C) rc = select(u0, U - u0 < C ? U - u0 : C, scores + u0 * N);
    return rc;
  }
  const MrModel& m = *model;
  const EvalPlan p = catalogue_plan(m, C, N);
  Carver cv(ws);
  int32_t* iota = cv.take<int32_t>((size_t)C * N);
  float* probs_buf = cv.take<float>((size_t)C * N);
  int32_t* own_users = users == nullptr ? cv.take<int32_t>((size_t)C) : nullptr;
  const EvalWs w = eval_carve(m, p, static_cast<char*>(ws) + cv.off);
  prof_mark(MR_PHASE_MISC, st);
  rc = items != nullptr ? launch_tile_list(iota, C * N, items, N, st) : launch_tile_iota(iota, C * N, N, st);
  if (rc == MR_OK) rc = eval_prepare(m, p, w, users, st);
  for (int64_t u0 = 0; u0 < U && rc == MR_OK; u0 += C) {
    const int64_t c = U - u0 < C ? U - u0 : C;
    const int64_t rows = c * N;
    float* out = scores != nullptr ? scores + u0 * N : probs_buf;
    const int32_t* cu = users != nullptr ? users + u0 : own_users;
    if (own_users != nullptr) rc = launch_iota(own_users, c, u0, st);
    if (rc != MR_OK) break;
    if (p.tower == EVAL_TC) {
      // each chunk starts at row 0 of its own users: one group = one user, Zu once per user
      prof_mark(MR_PHASE_TC_DENSE_FWD, st);
      rc = tc_forward_rows(m, w.t, cu, iota, 1, 0, rows, st, N, true, p.head_dot);
      if (rc == MR_OK) {
        prof_mark(MR_PHASE_HEAD, st);
        rc = launch_catalogue_head(m, w.t.H[m.n_layers - 1], cu, rows, N, out, st, nullptr,
                                   items != nullptr ? iota : nullptr);
      }
    } else if (p.tower == EVAL_SMALL) {
      prof_mark(MR_PHASE_FUSED_TILE, st);
      rc = launch_small_tower_forward(m, w.t.Pi, w.t.Pu, cu, iota, rows, N, out, st);
    } else {
      rc = mr_neumf_forward(&m, cu, iota, rows, N, nullptr, out, nullptr, nullptr, w.fwd, w.fwd_bytes, st);
    }
    if (rc != MR_OK) break;
    prof_mark(MR_PHASE_RANK, st);
    rc = select(u0, c, out);
  }
  return rc;
}

static int targets_check(int64_t U, int32_t N, int32_t excl_rows, const int64_t* excl_rowptr, const int32_t* excl_items,
                         const int64_t* tgt_rowptr, const int32_t* tgt_items, int64_t nnz_t, const int32_t* ks,
                         int32_t n_ks, const int32_t* tpos, const float* sums, TargetCutoffs& cut) {
  MR_REQUIRE(U >= 0 && U <= INT32_MAX && N >= 1 && nnz_t >= 0 && nnz_t <= INT32_MAX, "targets: bad U=%lld N=%d nnz_t=%lld",
             (long long)U, N, (long long)nnz_t);
  MR_REQUIRE(U > 0 || nnz_t == 0, "targets: nnz_t=%lld targets in no list", (long long)nnz_t);
  MR_REQUIRE(ks != nullptr && n_ks >= 1 && n_ks <= MR_MAX_CUTOFFS, "targets: n_ks=%d out of [1,%d]", n_ks, MR_MAX_CUTOFFS);
  for (int c = 0; c < n_ks; ++c) {
    MR_REQUIRE(ks[c] >= 1, "targets: cutoff ks[%d]=%d < 1", c, ks[c]);
    cut.k[c] = ks[c];
  }
  cut.n = n_ks;
  MR_REQUIRE(excl_rows >= 0 && (excl_rowptr == nullptr || excl_items != nullptr), "targets: bad exclusion lists");
  MR_REQUIRE(nnz_t == 0 || (tgt_rowptr != nullptr && tgt_items != nullptr), "targets: tgt_rowptr / tgt_items is NULL");
  MR_REQUIRE(tpos != nullptr || sums != nullptr, "targets: tpos and sums are both NULL");
  return MR_OK;
}

static int audience_check(int64_t U, int32_t M, int32_t k, int32_t excl_rows, const int64_t* excl_rowptr,
                          const int32_t* excl_users, const int32_t* targets, const int32_t* pos, const float* sums) {
  MR_REQUIRE(U >= 0 && U <= INT32_MAX && M >= 0, "audience: bad U=%lld M=%d", (long long)U, M);
  MR_REQUIRE(k >= 1 && k <= MR_MAX_TOPK, "audience: k=%d out of [1,%d]", k, MR_MAX_TOPK);
  MR_REQUIRE(excl_rows >= 0 && (excl_rowptr == nullptr || excl_users != nullptr), "audience: bad exclusion lists");
  MR_REQUIRE(targets != nullptr || (pos == nullptr && sums == nullptr), "audience: pos / sums need targets");
  return MR_OK;
}

// ---- ragged candidate lists: list u pairs users[u] with items[rowptr[u] .. rowptr[u+1]) ------------------------------
static int lists_check(int64_t U, const int64_t* rowptr, int64_t nnz, int32_t k, const int32_t* targets,
                       const int32_t* pos, const float* sums) {
  MR_REQUIRE(U >= 0 && U <= INT32_MAX && nnz >= 0 && nnz <= INT32_MAX, "lists: bad U=%lld nnz=%lld", (long long)U,
             (long long)nnz);
  MR_REQUIRE(U > 0 || nnz == 0, "lists: nnz=%lld rows in no list", (long long)nnz);
  MR_REQUIRE(k >= 1 && k <= MR_MAX_TOPK, "lists: k=%d out of [1,%d]", k, MR_MAX_TOPK);
  MR_REQUIRE(targets != nullptr || (pos == nullptr && sums == nullptr), "lists: pos / sums need targets");
  MR_REQUIRE(U == 0 || rowptr != nullptr, "lists: rowptr is NULL");
  return MR_OK;
}


// ---- serving queries: one body per query --------------------------------------------------------------------------
// Each query runs on the caller's scores (model == NULL: mr_topk_scores, mr_targets_scores, mr_audience_scores,
// mr_topk_lists) or on the model's probabilities (mr_catalogue_topk, mr_catalogue_targets, mr_catalogue_audience,
// mr_rank_lists); catalogue_sweep is the one chunk loop of both.  `fn` names the call in error messages.  A model
// call's workspace adds the scoring's and 512 bytes of carving slack to the selection's; a matrix call's adds 256.

static int workspace_check(const char* fn, size_t ws_bytes, size_t need) {
  if (ws_bytes >= need) return MR_OK;
  set_error("%s workspace too small: %zu < %zu", fn, ws_bytes, need);
  return MR_ERR_WORKSPACE;
}

// What a model's workspace query needs of it (0 bytes otherwise); lists and targets also need a first layer to split.
static bool serving_model_ok(const MrModel* model, bool split_first_layer) {
  return model != nullptr && model->n_layers >= 1 && model->n_layers <= MR_MAX_LAYERS && model->num_items >= 1 &&
         model->num_users >= 1 && (!split_first_layer || model->L[0] >= 2);
}

static size_t topk_bytes(const MrModel* model, int64_t U, int32_t N, int32_t k) {
  if (U < 0 || N < 1 || k < 1 || k > MR_MAX_TOPK) return 0;
  const int64_t C = clamp_users(U, catalogue_chunk_users(N));
  if (model == nullptr) return topk_workspace_bytes(C, N, k) + 256;
  return align_up(topk_workspace_bytes(C, N, k), 256) + catalogue_sweep_bytes(*model, C, N) + 512;
}

// Top-k per row: row u is users[u] against the catalogue (model) or row u of the matrix; exclusion list excl_ids[u].
static int topk_query(const char* fn, const MrModel* model, float* scores, int32_t N, const int32_t* users,
                      int32_t num_users, int64_t U, int32_t k, const int32_t* excl_ids, int32_t excl_rows,
                      const int64_t* excl_rowptr, const int32_t* excl_items, const int32_t* targets, int32_t* top_items,
                      float* top_scores, int32_t* pos, float* sums, void* ws, size_t ws_bytes, cudaStream_t st) {
  int rc = topk_check(U, N, k, excl_rows, excl_rowptr, excl_items, targets, pos, sums);
  if (rc != MR_OK) return rc;
  if (U == 0) {
    if (sums != nullptr) MR_CUDA(cudaMemsetAsync(sums, 0, 2 * sizeof(float), st));
    return MR_OK;
  }
  MR_REQUIRE((model != nullptr ? users != nullptr : scores != nullptr) && ws != nullptr, "%s: %s / ws is NULL", fn,
             model != nullptr ? "users" : "scores");
  rc = workspace_check(fn, ws_bytes, topk_bytes(model, U, N, k));
  if (rc != MR_OK) return rc;
  const int64_t C = clamp_users(U, catalogue_chunk_users(N));
  Carver cv(ws);
  void* sel_ws = cv.take<char>(topk_workspace_bytes(C, N, k));
  TopkArgs a{};
  a.N = N;
  a.k = k;
  a.excl_ids = excl_ids;
  a.excl_rows = excl_rows;
  a.excl_rowptr = excl_rowptr;
  a.excl_items = excl_items;
  a.targets = targets;
  a.users = users;
  a.num_users = num_users;
  a.top_items = top_items;
  a.top_scores = top_scores;
  a.pos = pos;
  rc = catalogue_sweep(model, users, U, C, N, scores, static_cast<char*>(ws) + cv.off, st,
                       [&](int64_t u0, int64_t c, const float* out) {
                         a.u0 = u0;
                         a.U = c;
                         a.scores = out;
                         return launch_topk(a, sel_ws, st);
                       });
  if (rc == MR_OK) {
    prof_mark(MR_PHASE_RANK, st);
    rc = launch_topk_metrics(pos, U, k, sums, st);
  }
  prof_mark(-1, st);
  return rc;
}

static size_t targets_bytes(const MrModel* model, int64_t U, int32_t N, int64_t nnz_t) {
  if (U < 0 || U > INT32_MAX || N < 1 || nnz_t < 0 || nnz_t > INT32_MAX) return 0;
  const int64_t C = clamp_users(U, catalogue_chunk_users(N));
  const size_t sel = targets_workspace_bytes(C, nnz_t) + 256;
  return model == nullptr ? sel : align_up(sel, 256) + catalogue_sweep_bytes(*model, C, N) + 512;
}

// Places of many targets per row; rows and exclusion lists as topk_query.
static int targets_query(const char* fn, const MrModel* model, float* scores, int32_t N, const int32_t* users,
                         int32_t num_users, int64_t U, const int32_t* excl_ids, int32_t excl_rows,
                         const int64_t* excl_rowptr, const int32_t* excl_items, const int64_t* tgt_rowptr,
                         const int32_t* tgt_items, int64_t nnz_t, const int32_t* ks, int32_t n_ks, int32_t* tpos,
                         float* sums, void* ws, size_t ws_bytes, cudaStream_t st) {
  TargetCutoffs cut{};
  int rc = targets_check(U, N, excl_rows, excl_rowptr, excl_items, tgt_rowptr, tgt_items, nnz_t, ks, n_ks, tpos, sums,
                         cut);
  if (rc != MR_OK) return rc;
  // A model call without users needs no users or workspace; a matrix call without rows still wants its workspace and
  // zeroes the sums in launch_targets_metrics.
  if (model != nullptr && U == 0) {
    if (sums != nullptr) MR_CUDA(cudaMemsetAsync(sums, 0, (MR_TGT_CUTOFF0 + MR_TGT_PER_CUTOFF * n_ks) * sizeof(float), st));
    return MR_OK;
  }
  MR_REQUIRE(U == 0 || (model != nullptr ? users != nullptr : scores != nullptr), "%s: %s is NULL", fn,
             model != nullptr ? "users" : "scores");
  MR_REQUIRE(ws != nullptr, "%s: workspace is NULL", fn);
  rc = workspace_check(fn, ws_bytes, targets_bytes(model, U, N, nnz_t));
  if (rc != MR_OK) return rc;
  const int64_t C = clamp_users(U, catalogue_chunk_users(N));
  Carver cv(ws);
  const TargetsWs w = carve_targets(cv.take<char>(targets_bytes(nullptr, U, N, nnz_t)), C, nnz_t);
  TargetsArgs a{};
  a.N = N;
  a.excl_ids = excl_ids;
  a.excl_rows = excl_rows;
  a.excl_rowptr = excl_rowptr;
  a.excl_items = excl_items;
  a.tgt_rowptr = tgt_rowptr;
  a.tgt_items = tgt_items;
  a.nnz_t = nnz_t;
  a.users = users;
  a.num_users = num_users;
  a.tpos = tpos;
  rc = catalogue_sweep(model, users, U, C, N, scores, static_cast<char*>(ws) + cv.off, st,
                       [&](int64_t u0, int64_t c, const float* out) {
                         a.u0 = u0;
                         a.U = c;
                         a.scores = out;
                         return launch_targets_chunk(a, w, st);
                       });
  if (rc == MR_OK) {
    prof_mark(MR_PHASE_RANK, st);
    rc = launch_targets_metrics(tgt_rowptr, U, nnz_t, w.spos, cut, sums, w.partials, st);
  }
  prof_mark(-1, st);
  return rc;
}

static size_t audience_bytes(const MrModel* model, int64_t U, int32_t M, int32_t k) {
  if (U < 0 || U > INT32_MAX || M < 0 || k < 1 || k > MR_MAX_TOPK) return 0;
  const int64_t C = clamp_users(U, catalogue_chunk_users(M));
  const size_t sel = carve_audience(nullptr, C, M, k).total;  // the running lists of every item
  if (model == nullptr) return sel + 256;
  return align_up(sel, 256) + catalogue_sweep_bytes(*model, C, M < 1 ? 1 : M, true) + 512;
}

// Audiences: the k best of U pool users (users, NULL = ids 0 .. U-1) for each of M columns: the matrix's columns, or
// the model's items[0, M) (which also index the exclusion lists).
static int audience_query(const char* fn, const MrModel* model, float* scores, const int32_t* items, int32_t M,
                          int32_t k, const int32_t* users, int32_t num_users, int64_t U, const int32_t* excl_ids,
                          int32_t excl_rows, const int64_t* excl_rowptr, const int32_t* excl_users,
                          const int32_t* targets, int32_t* top_users, float* top_scores, int32_t* pos, float* sums,
                          void* ws, size_t ws_bytes, cudaStream_t st) {
  int rc = audience_check(U, M, k, excl_rows, excl_rowptr, excl_users, targets, pos, sums);
  if (rc != MR_OK) return rc;
  if (model != nullptr) {
    MR_REQUIRE(users != nullptr || U == model->num_users, "%s: without a pool U must be num_users (%d), got %lld", fn,
               model->num_users, (long long)U);
    MR_REQUIRE((M == 0 || items != nullptr) && ws != nullptr, "%s: items / ws is NULL", fn);
  } else {
    MR_REQUIRE((U == 0 || M == 0 || scores != nullptr) && ws != nullptr, "%s: scores / ws is NULL", fn);
  }
  rc = workspace_check(fn, ws_bytes, audience_bytes(model, U, M, k));
  if (rc != MR_OK) return rc;
  const int64_t C = clamp_users(U, catalogue_chunk_users(M));
  Carver cv(ws);
  const AudienceState w = carve_audience(cv.take<char>(carve_audience(nullptr, C, M, k).total), C, M, k);
  AudienceArgs a{};
  a.M = M;
  a.k = k;
  a.users = users;
  a.num_users = num_users;
  a.excl_ids = excl_ids;
  a.excl_rows = excl_rows;
  a.excl_rowptr = excl_rowptr;
  a.excl_users = excl_users;
  a.targets = targets;
  if (M > 0) {
    rc = launch_audience_init(a, w, st);
    if (rc == MR_OK)
      rc = catalogue_sweep(model, users, U, C, M, scores, static_cast<char*>(ws) + cv.off, st,
                           [&](int64_t u0, int64_t c, const float* out) {
                             a.u0 = u0;
                             a.U = c;
                             a.scores = out;
                             return launch_audience_chunk(a, w, st);
                           },
                           items);
  }
  if (rc == MR_OK) {
    prof_mark(MR_PHASE_RANK, st);
    rc = launch_audience_final(a, w, items, model != nullptr ? model->num_items : 0, top_users, top_scores, pos, sums,
                               st);
  }
  prof_mark(-1, st);
  return rc;
}

static size_t lists_bytes(const MrModel* model, int64_t U, int64_t nnz, int32_t k) {
  if (U < 0 || U > INT32_MAX || nnz < 0 || nnz > INT32_MAX || k < 1 || k > MR_MAX_TOPK) return 0;
  const size_t sel = topk_lists_workspace_bytes(U, nnz, k) + 256;
  if (model == nullptr) return sel;
  return sel + align_up((size_t)nnz * sizeof(int32_t), 256) + align_up((size_t)nnz * sizeof(float), 256) +
         eval_carve(*model, eval_plan(*model, SCORE_LISTS, U, 0, nnz), nullptr).total + 256;
}

// Top-k of ragged lists: list u is rows rowptr[u] .. rowptr[u+1] of the caller's scores (model == NULL), or pairs
// users[u] with items[rowptr[u] .. rowptr[u+1]) and is scored first (into scores when given).
static int lists_query(const char* fn, const MrModel* model, float* scores, const int32_t* users, int64_t U,
                       const int64_t* rowptr, const int32_t* items, int64_t nnz, int32_t k, const int32_t* targets,
                       int32_t* top_pos, int32_t* top_items, float* top_scores, int32_t* pos, float* sums, void* ws,
                       size_t ws_bytes, cudaStream_t st) {
  int rc = lists_check(U, rowptr, nnz, k, targets, pos, sums);
  if (rc != MR_OK) return rc;
  if (model != nullptr) MR_REQUIRE(U == 0 || users != nullptr, "%s: users is NULL", fn);
  MR_REQUIRE(nnz == 0 || (model != nullptr ? items != nullptr : scores != nullptr), "%s: %s is NULL", fn,
             model != nullptr ? "items" : "scores");
  MR_REQUIRE(ws != nullptr, "%s: workspace is NULL", fn);
  rc = workspace_check(fn, ws_bytes, lists_bytes(model, U, nnz, k));
  if (rc != MR_OK) return rc;
  Carver cv(ws);
  void* sel_ws = cv.take<char>(topk_lists_workspace_bytes(U, nnz, k));
  if (model != nullptr) {
    const MrModel& m = *model;
    int32_t* seg = cv.take<int32_t>((size_t)nnz);
    float* probs_buf = cv.take<float>((size_t)nnz);
    if (scores == nullptr) scores = probs_buf;
    const EvalPlan p = eval_plan(m, SCORE_LISTS, U, 0, nnz);
    const EvalWs w = eval_carve(m, p, static_cast<char*>(ws) + cv.off);
    if (nnz > 0) {
      prof_mark(MR_PHASE_MISC, st);
      // seg: the list of each row, or the user of each row (plain forward)
      rc = launch_list_rows(rowptr, U, nnz, p.tower == EVAL_FORWARD ? users : nullptr, seg, st);
      if (rc == MR_OK) rc = eval_prepare(m, p, w, users, st);
      if (rc == MR_OK && p.tower == EVAL_SMALL) prof_mark(MR_PHASE_FUSED_TILE, st);
      for (int64_t r0 = 0; r0 < nnz && rc == MR_OK; r0 += p.sb) {
        const int64_t r1 = r0 + p.sb < nnz ? r0 + p.sb : nnz;
        if (p.tower == EVAL_TC) {  // the second layer's producers compute relu(Pi[items[row]] + Zu[seg[row]])
          prof_mark(MR_PHASE_TC_DENSE_FWD, st);
          rc = tc_forward_rows(m, w.t, users, items, 1, r0, r1, st, 0, false, p.head_dot, seg, (int32_t)U);
          if (rc != MR_OK) break;
          prof_mark(MR_PHASE_HEAD, st);
          rc = launch_catalogue_head(m, w.t.H[m.n_layers - 1], users, r1 - r0, 1, scores, st, seg, items, r0, U);
        } else if (p.tower == EVAL_SMALL) {
          rc = launch_small_tower_forward(m, w.t.Pi, w.t.Pu, users, items + r0, r1 - r0, 1, scores + r0, st, seg + r0,
                                          U);
        } else {
          rc = mr_neumf_forward(model, seg + r0, items + r0, r1 - r0, 1, nullptr, scores + r0, nullptr, nullptr, w.fwd,
                                w.fwd_bytes, st);
        }
      }
      if (rc != MR_OK) return rc;
    }
  }
  TopkListsArgs a{};
  a.scores = scores;
  a.rowptr = rowptr;
  a.U = U;
  a.nnz = nnz;
  a.k = k;
  a.targets = targets;
  a.users = users;
  a.num_users = model != nullptr ? model->num_users : 0;
  a.items = items;
  a.top_pos = top_pos;
  a.top_items = top_items;
  a.top_scores = top_scores;
  a.pos = pos;
  prof_mark(MR_PHASE_RANK, st);
  rc = launch_topk_lists(a, sums, sel_ws, st);
  prof_mark(-1, st);
  return rc;
}

}  // namespace mr

using namespace mr;

extern "C" {

int mr_version(void) { return MR_VERSION; }

const char* mr_last_error(void) { return g_err; }

int mr_device_sm_count(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    cuda_fail(cudaGetLastError(), "cudaGetDevice");
    return MR_ERR_NO_DEVICE;
  }
  return sm_count();
}

int mr_gather_rows(const float* table, int64_t rows, int32_t dim, const int32_t* idx, int64_t n, float* out,
                   void* stream) {
  if (n == 0) return MR_OK;  // empty batch: nothing to read or write (pointers may be NULL)
  MR_REQUIRE(table && idx && out, "gather: NULL pointer");
  MR_REQUIRE(rows > 0 && dim > 0 && n >= 0, "gather: bad sizes rows=%lld dim=%d n=%lld", (long long)rows, dim, (long long)n);
  return launch_gather_rows(table, rows, dim, idx, n, out, (cudaStream_t)stream);
}

int mr_gather_rows_sharded(const float* const* shards, int32_t world, int64_t total_rows, int32_t dim,
                           const int32_t* ids, int64_t n, float* out, void* stream) {
  if (n == 0) return MR_OK;
  MR_REQUIRE(shards && ids && out, "gather_rows_sharded: NULL pointer");
  MR_REQUIRE(world >= 1 && total_rows > 0 && dim > 0 && n >= 0, "gather_rows_sharded: bad sizes");
  return launch_gather_rows_sharded(shards, world, total_rows, dim, ids, n, out, (cudaStream_t)stream);
}

size_t mr_forward_workspace_bytes(const MrModel* model, int64_t B) {
  (void)B;
  size_t n = 256 + align_up((size_t)max_tile_ctas() * sizeof(float), 256);
  if (model != nullptr && model->n_layers >= 1 && model->n_layers <= MR_MAX_LAYERS && tc_eligible(*model))
    n += carve_tc(*model, false, B, nullptr).total;
  return n;
}

int mr_neumf_forward(const MrModel* model, const int32_t* users, const int32_t* items, int64_t B, int32_t user_div,
                     float* logits, float* probs, const float* labels, float* loss_sum, void* ws, size_t ws_bytes,
                     void* stream) {
  int rc = check_model(model);
  if (rc != MR_OK) return rc;
  MR_REQUIRE(B >= 0, "forward: negative B");
  if (B == 0) {  // empty batch (pointers may be NULL): only the loss sum is defined
    if (loss_sum != nullptr) MR_CUDA(cudaMemsetAsync(loss_sum, 0, sizeof(float), (cudaStream_t)stream));
    return MR_OK;
  }
  MR_REQUIRE(users && items, "forward: NULL ids");
  MR_REQUIRE(user_div >= 1, "forward: user_div must be >= 1");
  MR_REQUIRE(ws != nullptr, "forward: workspace is NULL");
  if (ws_bytes < mr_forward_workspace_bytes(model, B)) {
    set_error("forward workspace too small: %zu < %zu", ws_bytes, mr_forward_workspace_bytes(model, B));
    return MR_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  Carver cv(ws);
  int32_t* flags = cv.take<int32_t>(64);
  float* loss_partial = cv.take<float>(max_tile_ctas());
  MR_CUDA(cudaMemsetAsync(flags, 0, 256, st));
  if (use_tc(*model) && labels == nullptr) {  // forward with a loss request is served by the SIMT kernel
    const MrModel& m = *model;
    TcWs t = carve_tc(m, false, B, static_cast<char*>(ws) + cv.off);
    prof_mark(MR_PHASE_MISC, st);
    for (int l = 1; l < m.n_layers; ++l) {
      rc = launch_pack_weights(m.W[l], m.L[l - 1], m.L[l], 0, t.pack_f[l], st);
      if (rc != MR_OK) return rc;
    }
    const int64_t sb = tc_sub_batch(B);
    for (int64_t r0 = 0; r0 < B; r0 += sb) {
      const int64_t r1 = r0 + sb < B ? r0 + sb : B;
      prof_mark(MR_PHASE_TC_DENSE_FWD, st);
      rc = tc_forward_rows(m, t, users, items, user_div, r0, r1, st);
      if (rc != MR_OK) return rc;
      prof_mark(MR_PHASE_HEAD, st);
      HeadArgs h{};
      h.model = model;
      h.h_last = t.H[m.n_layers - 1];
      h.users = users;
      h.items = items;
      h.rows = r1 - r0;
      h.row0 = r0;
      h.user_div = user_div;
      h.logits = logits;
      h.probs = probs;
      h.flags = flags;
      rc = launch_head(h, st);
      if (rc != MR_OK) return rc;
    }
    prof_mark(-1, st);
    return MR_OK;
  }
  TileLaunch a{};
  a.model = model;
  a.train = false;
  a.users = users;
  a.items = items;
  a.labels = labels;
  a.B = B;
  a.user_div = user_div;
  a.inv_batch = 0.f;
  a.logits = logits;
  a.probs = probs;
  a.loss_partial = loss_partial;
  a.flags = flags;
  int grid = 0;
  prof_mark(MR_PHASE_TILE_FORWARD, st);
  rc = launch_neumf_tiles(a, st, &grid);
  prof_mark(MR_PHASE_MISC, st);
  if (rc == MR_OK && loss_sum != nullptr) rc = launch_sum_partials(loss_partial, grid, loss_sum, st);
  prof_mark(-1, st);
  return rc;
}

size_t mr_train_workspace_bytes(const MrModel* model, int64_t B) {
  if (model == nullptr || B < 0 || model->n_layers < 1 || model->n_layers > MR_MAX_LAYERS) return 0;
  return carve_train(*model, B, nullptr).total + 256;
}

int mr_neumf_train_grads(MrModel* model, MrOptState* opt, MrGrads* grads, const int32_t* users, const int32_t* items,
                         const float* labels, int64_t B, int32_t group, int32_t k, int32_t flags,
                         float inv_global_batch, float* step_out, void* ws, size_t ws_bytes, void* stream) {
  int rc = check_model(model);
  if (rc != MR_OK) return rc;
  rc = check_opt(*model, opt, grads);
  if (rc != MR_OK) return rc;
  MR_REQUIRE(users && items && labels && step_out && ws, "train: NULL pointer");
  MR_REQUIRE(B > 0 && B < ((int64_t)1 << 31), "train: B=%lld out of range", (long long)B);
  MR_REQUIRE(group >= 0 && (group == 0 || B % group == 0), "train: B=%lld not divisible by group=%d", (long long)B, group);
  if (ws_bytes < mr_train_workspace_bytes(model, B)) {
    set_error("train workspace too small: %zu < %zu", ws_bytes, mr_train_workspace_bytes(model, B));
    return MR_ERR_WORKSPACE;
  }
  TrainStep s{*model, *opt, *grads, users, items, labels, B, group, k, flags, inv_global_batch, step_out,
               carve_train(*model, B, ws), side_stream(), (cudaStream_t)stream};
  s.p = s.plan();
  rc = s.prologue();
  if (rc != MR_OK) return rc;
  switch (s.p.path) {
    case TRAIN_SMALL: rc = s.tower_small(); break;
    case TRAIN_TILES: rc = s.tower_tiles(); break;
    default: rc = s.tower_tc(); break;
  }
  if (rc != MR_OK) return rc;
  return s.epilogue();
}

int mr_neumf_apply(MrModel* model, MrOptState* opt, const MrGrads* grads, void* stream) {
  int rc = check_model(model);
  if (rc != MR_OK) return rc;
  rc = check_opt(*model, opt, grads);
  if (rc != MR_OK) return rc;
  const MrModel& m = *model;
  cudaStream_t st = (cudaStream_t)stream;
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u;
  const bool adam = opt->optimizer == MR_OPT_ADAM;
  const float lr_t = adam ? adam_lr_t(*opt, opt->iterations + 1) : opt->lr;
  prof_mark(MR_PHASE_OPTIMIZER, st);
  OptRegions r{};
  auto add = [&](float* p, const float* g, float* mm, float* vv, int64_t n, float l2) {
    r.p[r.count] = p; r.g[r.count] = g; r.m[r.count] = mm; r.v[r.count] = vv; r.n[r.count] = n; r.l2[r.count] = l2;
    ++r.count;
  };
  add(m.dense, grads->dense, opt->m_dense, opt->v_dense, m.dense_count, 0.f);
  if (opt->table_mode == MR_TABLES_DENSE) {
    const float l2 = m.l2[0];
    add(m.user_mlp, grads->user_mlp, opt->m_user_mlp, opt->v_user_mlp, (int64_t)m.num_users * d_u, l2);
    add(m.item_mlp, grads->item_mlp, opt->m_item_mlp, opt->v_item_mlp, (int64_t)m.num_items * d_i, l2);
    if (m.mf_dim > 0) {
      add(m.user_gmf, grads->user_gmf, opt->m_user_gmf, opt->v_user_gmf, (int64_t)m.num_users * m.mf_dim, l2);
      add(m.item_gmf, grads->item_gmf, opt->m_item_gmf, opt->v_item_gmf, (int64_t)m.num_items * m.mf_dim, l2);
    }
  }
  rc = launch_optimizer_regions(r, opt->optimizer, lr_t, opt->beta_1, opt->beta_2, opt->epsilon, st);
  if (rc != MR_OK) return rc;
  prof_mark(-1, st);
  opt->iterations += 1;
  return MR_OK;
}

int mr_neumf_train_step(MrModel* model, MrOptState* opt, MrGrads* grads, const int32_t* users, const int32_t* items,
                        const float* labels, int64_t B, int32_t group, int32_t k, int32_t flags, float inv_global_batch,
                        float* step_out, void* ws, size_t ws_bytes, void* stream) {
  int rc = mr_neumf_train_grads(model, opt, grads, users, items, labels, B, group, k, flags, inv_global_batch, step_out,
                                ws, ws_bytes, stream);
  if (rc != MR_OK) return rc;
  return mr_neumf_apply(model, opt, grads, stream);
}

// [flags 256 B][partials][probabilities, unless the fused head writes them][scoring]: the larger of the plans with and
// without ranks
size_t mr_rank_eval_workspace_bytes(const MrModel* model, int64_t G, int32_t group) {
  if (model == nullptr || model->n_layers < 1 || model->n_layers > MR_MAX_LAYERS || G < 0 || group < 1) return 0;
  size_t scoring = 0;
  for (const bool ranks : {false, true}) {
    const EvalPlan p = eval_plan(*model, SCORE_GROUPS, G, group, G * group, !ranks);
    const size_t probs = p.tower == EVAL_TC ? 0 : align_up((size_t)G * group * sizeof(float), 256);
    const size_t n = probs + eval_carve(*model, p, nullptr).total;
    if (n > scoring) scoring = n;
  }
  return 256 + align_up(rank_partials_count(G) * sizeof(float), 256) + scoring;
}

int mr_rank_eval(const MrModel* model, const int32_t* users, const int32_t* items, int64_t G, int32_t group, int32_t k,
                 int32_t* rank, int32_t* pos, float* probs, float* sums, void* ws, size_t ws_bytes, void* stream) {
  MR_REQUIRE(G >= 0 && group >= 2 && group <= MR_MAX_NEGS + 1, "rank_eval: bad G=%lld group=%d", (long long)G, group);
  MR_REQUIRE(pos != nullptr && ws != nullptr, "rank_eval: pos/ws is NULL");
  if (ws_bytes < mr_rank_eval_workspace_bytes(model, G, group)) {
    set_error("rank_eval workspace too small: %zu < %zu", ws_bytes, mr_rank_eval_workspace_bytes(model, G, group));
    return MR_ERR_WORKSPACE;
  }
  if (G == 0) {
    if (sums != nullptr) MR_CUDA(cudaMemsetAsync(sums, 0, 2 * sizeof(float), (cudaStream_t)stream));
    return MR_OK;
  }
  {
    int rc0 = check_model(model);
    if (rc0 != MR_OK) return rc0;
  }
  MR_REQUIRE(users && items, "rank_eval: NULL ids");
  const MrModel& m = *model;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t rows = G * group;
  const EvalPlan p = eval_plan(m, SCORE_GROUPS, G, group, rows, rank == nullptr);
  Carver cv(ws);
  int32_t* flags = cv.take<int32_t>(64);
  float* partials = cv.take<float>(rank_partials_count(G));
  float* probs_buf = p.tower == EVAL_TC ? nullptr : cv.take<float>((size_t)rows);
  const EvalWs w = eval_carve(m, p, static_cast<char*>(ws) + cv.off);
  int rc;
  if (p.tower == EVAL_TC) {  // forward with the user half of the first layer once per group, then the fused head
    prof_mark(MR_PHASE_MISC, st);
    MR_CUDA(cudaMemsetAsync(flags, 0, 256, st));
    rc = eval_prepare(m, p, w, users, st);
    for (int64_t r0 = 0; r0 < rows && rc == MR_OK; r0 += p.sb) {
      const int64_t r1 = r0 + p.sb < rows ? r0 + p.sb : rows;
      prof_mark(MR_PHASE_TC_DENSE_FWD, st);
      rc = tc_forward_rows(m, w.t, users, items, 1, r0, r1, st, group, true, p.head_dot);
      if (rc != MR_OK) break;
      prof_mark(MR_PHASE_HEAD, st);
      HeadArgs h{};
      h.model = &m;
      h.h_is_dot = p.head_dot;
      h.h_last = w.t.H[m.n_layers - 1];
      h.users = users;
      h.items = items;
      h.rows = r1 - r0;
      h.row0 = r0;
      h.flags = flags;
      rc = launch_head_rank(h, group, pos, probs, st);
    }
    if (rc != MR_OK) return rc;
    prof_mark(MR_PHASE_RANK, st);
    rc = launch_rank_metrics(pos, G, k, sums, partials, st);
  } else {
    float* pr = probs != nullptr ? probs : probs_buf;
    if (p.tower == EVAL_SMALL) {  // thread-per-row forward on the projected tables (small_tower.cu)
      rc = eval_prepare(m, p, w, users, st);
      prof_mark(MR_PHASE_FUSED_TILE, st);
      if (rc == MR_OK) rc = launch_small_tower_forward(m, w.t.Pi, w.t.Pu, users, items, rows, group, pr, st);
    } else {
      rc = mr_neumf_forward(model, users, items, rows, group, nullptr, pr, nullptr, nullptr, w.fwd, w.fwd_bytes, stream);
    }
    if (rc != MR_OK) return rc;
    prof_mark(MR_PHASE_RANK, st);
    rc = launch_rank_scores(pr, G, group, k, nullptr, rank, pos, sums, partials, st);
  }
  prof_mark(-1, st);
  return rc;
}

size_t mr_rank_scores_workspace_bytes(int64_t G) { return align_up(rank_partials_count(G < 0 ? 0 : G) * sizeof(float), 256); }

int mr_rank_scores(const float* scores, int64_t G, int32_t group, int32_t k, const int32_t* label_col,
                   const float* labels, int32_t* rank, int32_t* pos, float* sums, void* ws, size_t ws_bytes,
                   void* stream) {
  MR_REQUIRE(scores && pos, "rank_scores: NULL pointer");
  MR_REQUIRE(G >= 0 && group >= 1 && group <= MR_MAX_NEGS + 1, "rank_scores: bad G=%lld group=%d", (long long)G, group);
  if (sums != nullptr) {
    MR_REQUIRE(ws != nullptr, "rank_scores: workspace is NULL");
    if (ws_bytes < mr_rank_scores_workspace_bytes(G)) {
      set_error("rank_scores workspace too small");
      return MR_ERR_WORKSPACE;
    }
  }
  return launch_rank_scores(scores, G, group, k, label_col, rank, pos, sums, static_cast<float*>(ws), (cudaStream_t)stream,
                            labels);
}

// The matrix calls only read `scores`; the bodies take it writable for the model calls' optional full-score output.
size_t mr_topk_scores_workspace_bytes(int64_t U, int32_t N, int32_t k) { return topk_bytes(nullptr, U, N, k); }

int mr_topk_scores(const float* scores, int64_t U, int32_t N, int32_t k, const int32_t* excl_ids, int32_t excl_rows,
                   const int64_t* excl_rowptr, const int32_t* excl_items, const int32_t* targets, int32_t* top_items,
                   float* top_scores, int32_t* pos, float* sums, void* ws, size_t ws_bytes, void* stream) {
  return topk_query("topk_scores", nullptr, const_cast<float*>(scores), N, nullptr, 0, U, k, excl_ids, excl_rows,
                    excl_rowptr, excl_items, targets, top_items, top_scores, pos, sums, ws, ws_bytes,
                    (cudaStream_t)stream);
}

size_t mr_catalogue_topk_workspace_bytes(const MrModel* model, int64_t U, int32_t k) {
  return serving_model_ok(model, false) ? topk_bytes(model, U, model->num_items, k) : 0;
}

int mr_catalogue_topk(const MrModel* model, const int32_t* users, int64_t U, int32_t k, int32_t excl_rows,
                      const int64_t* excl_rowptr, const int32_t* excl_items, const int32_t* targets, int32_t* top_items,
                      float* top_scores, int32_t* pos, float* sums, float* scores, void* ws, size_t ws_bytes,
                      void* stream) {
  const int rc = check_model(model);
  if (rc != MR_OK) return rc;
  // exclusion lists are indexed by user id
  return topk_query("catalogue_topk", model, scores, model->num_items, users, model->num_users, U, k, users, excl_rows,
                    excl_rowptr, excl_items, targets, top_items, top_scores, pos, sums, ws, ws_bytes,
                    (cudaStream_t)stream);
}

size_t mr_targets_scores_workspace_bytes(int64_t U, int32_t N, int64_t nnz_t) { return targets_bytes(nullptr, U, N, nnz_t); }

int mr_targets_scores(const float* scores, int64_t U, int32_t N, const int32_t* excl_ids, int32_t excl_rows,
                      const int64_t* excl_rowptr, const int32_t* excl_items, const int64_t* tgt_rowptr,
                      const int32_t* tgt_items, int64_t nnz_t, const int32_t* ks, int32_t n_ks, int32_t* tpos,
                      float* sums, void* ws, size_t ws_bytes, void* stream) {
  return targets_query("targets_scores", nullptr, const_cast<float*>(scores), N, nullptr, 0, U, excl_ids, excl_rows,
                       excl_rowptr, excl_items, tgt_rowptr, tgt_items, nnz_t, ks, n_ks, tpos, sums, ws, ws_bytes,
                       (cudaStream_t)stream);
}

size_t mr_catalogue_targets_workspace_bytes(const MrModel* model, int64_t U, int64_t nnz_t) {
  return serving_model_ok(model, true) ? targets_bytes(model, U, model->num_items, nnz_t) : 0;
}

int mr_catalogue_targets(const MrModel* model, const int32_t* users, int64_t U, int32_t excl_rows,
                         const int64_t* excl_rowptr, const int32_t* excl_items, const int64_t* tgt_rowptr,
                         const int32_t* tgt_items, int64_t nnz_t, const int32_t* ks, int32_t n_ks, int32_t* tpos,
                         float* sums, void* ws, size_t ws_bytes, void* stream) {
  const int rc = check_model(model);
  if (rc != MR_OK) return rc;
  // exclusion lists are indexed by user id
  return targets_query("catalogue_targets", model, nullptr, model->num_items, users, model->num_users, U, users,
                       excl_rows, excl_rowptr, excl_items, tgt_rowptr, tgt_items, nnz_t, ks, n_ks, tpos, sums, ws,
                       ws_bytes, (cudaStream_t)stream);
}

size_t mr_audience_scores_workspace_bytes(int64_t U, int32_t M, int32_t k) { return audience_bytes(nullptr, U, M, k); }

int mr_audience_scores(const float* scores, int64_t U, int32_t M, int32_t k, const int32_t* users,
                       const int32_t* excl_ids, int32_t excl_rows, const int64_t* excl_rowptr, const int32_t* excl_users,
                       const int32_t* targets, int32_t* top_users, float* top_scores, int32_t* pos, float* sums,
                       void* ws, size_t ws_bytes, void* stream) {
  // no model: every id >= 0 is a user
  return audience_query("audience_scores", nullptr, const_cast<float*>(scores), nullptr, M, k, users, INT32_MAX, U,
                        excl_ids, excl_rows, excl_rowptr, excl_users, targets, top_users, top_scores, pos, sums, ws,
                        ws_bytes, (cudaStream_t)stream);
}

size_t mr_catalogue_audience_workspace_bytes(const MrModel* model, int64_t U, int32_t M, int32_t k) {
  return serving_model_ok(model, false) ? audience_bytes(model, U, M, k) : 0;
}

int mr_catalogue_audience(const MrModel* model, const int32_t* items, int32_t M, int32_t k, const int32_t* users,
                          int64_t U, int32_t excl_rows, const int64_t* excl_rowptr, const int32_t* excl_users,
                          const int32_t* targets, int32_t* top_users, float* top_scores, int32_t* pos, float* sums,
                          float* scores, void* ws, size_t ws_bytes, void* stream) {
  const int rc = check_model(model);
  if (rc != MR_OK) return rc;
  // exclusion lists are indexed by item id
  return audience_query("catalogue_audience", model, scores, items, M, k, users, model->num_users, U, items, excl_rows,
                        excl_rowptr, excl_users, targets, top_users, top_scores, pos, sums, ws, ws_bytes,
                        (cudaStream_t)stream);
}

size_t mr_topk_lists_workspace_bytes(int64_t U, int64_t nnz, int32_t k) { return lists_bytes(nullptr, U, nnz, k); }

int mr_topk_lists(const float* scores, int64_t U, const int64_t* rowptr, int64_t nnz, int32_t k, const int32_t* targets,
                  int32_t* top_pos, float* top_scores, int32_t* pos, float* sums, void* ws, size_t ws_bytes, void* stream) {
  return lists_query("topk_lists", nullptr, const_cast<float*>(scores), nullptr, U, rowptr, nullptr, nnz, k, targets,
                     top_pos, nullptr, top_scores, pos, sums, ws, ws_bytes, (cudaStream_t)stream);
}

size_t mr_rank_lists_workspace_bytes(const MrModel* model, int64_t U, int64_t nnz, int32_t k) {
  return serving_model_ok(model, true) ? lists_bytes(model, U, nnz, k) : 0;
}

int mr_rank_lists(const MrModel* model, const int32_t* users, int64_t U, const int64_t* rowptr, const int32_t* items,
                  int64_t nnz, int32_t k, const int32_t* targets, int32_t* top_pos, int32_t* top_items, float* top_scores,
                  int32_t* pos, float* sums, float* probs, void* ws, size_t ws_bytes, void* stream) {
  const int rc = check_model(model);
  if (rc != MR_OK) return rc;
  return lists_query("rank_lists", model, probs, users, U, rowptr, items, nnz, k, targets, top_pos, top_items,
                     top_scores, pos, sums, ws, ws_bytes, (cudaStream_t)stream);
}

int mr_sample_negatives(const int64_t* csr_rowptr, const int32_t* csr_items, int32_t num_items, const int32_t* pos_users,
                        const int32_t* pos_items, int64_t P, int64_t first_index, int32_t negs, uint64_t seed,
                        uint64_t epoch, int32_t* out_users, int32_t* out_items, float* out_labels, void* stream) {
  MR_REQUIRE(csr_rowptr && csr_items && pos_users && pos_items, "sample_negatives: NULL pointer");
  MR_REQUIRE(P >= 0 && num_items > 0, "sample_negatives: bad sizes");
  MR_REQUIRE(negs >= 1 && negs <= MR_MAX_NEGS, "sample_negatives: negs=%d out of [1,%d]", negs, MR_MAX_NEGS);
  prof_mark(MR_PHASE_SAMPLER, (cudaStream_t)stream);
  int rc = launch_sample_negatives(csr_rowptr, csr_items, num_items, pos_users, pos_items, P, first_index, negs, seed,
                                   epoch, out_users, out_items, out_labels, (cudaStream_t)stream);
  prof_mark(-1, (cudaStream_t)stream);
  return rc;
}

// ---- fold-in: the other side's half of the first layer once per call over its table (the tensor-core table GEMM
// where the other side's width is the one the eval's item projection takes, else a per-element kernel), the new rows
// sorted by list length, one kernel.  One path for both directions: FoldSide names the sides. --------------------------
static bool fold_in_tc_proj(const MrModel& m, const FoldSide& sd) {
  return use_tc(m) && m.n_layers >= 3 && sd.d_o % 128 == 0 && sd.d_o <= 256 && m.L[1] == sd.d_o;
}

// Po = E_other . W1[other rows] over the other side's whole table, no bias (needs a hidden layer; pack: room for the
// packed row block when fold_in_tc_proj).
static int project_other_side(const MrModel& m, const FoldSide& sd, float* pack, float* Po, cudaStream_t st) {
  if (fold_in_tc_proj(m, sd)) {
    const int rc = launch_pack_weights(sd.W1o, sd.d_o, m.L[1], 0, pack, st);
    return rc != MR_OK ? rc : tc_project_table(m, sd.other_mlp, sd.num_other, sd.d_o, pack, Po, st);
  }
  return launch_fold_in_project(sd.other_mlp, sd.num_other, sd.d_o, sd.W1o, m.L[1], Po, st);
}

struct FoldWs {
  int32_t *flags, *keys, *sorted_keys, *order;
  void* sort_ws;
  size_t sort_ws_bytes;
  float *wt, *Po, *pack_fo;
  size_t total;
};

static FoldWs carve_fold_in(const MrModel& m, const FoldSide& sd, int64_t U, void* ws) {
  FoldWs w{};
  Carver cv(ws);
  w.flags = cv.take<int32_t>(64);
  w.keys = cv.take<int32_t>(U);
  w.sorted_keys = cv.take<int32_t>(U);
  w.order = cv.take<int32_t>(U);
  w.sort_ws_bytes = sort_workspace_bytes(U);
  w.sort_ws = cv.take<char>(w.sort_ws_bytes);
  w.wt = cv.take<float>(m.dense_count);
  if (m.n_layers > 1) w.Po = cv.take<float>((size_t)sd.num_other * m.L[1]);
  if (fold_in_tc_proj(m, sd)) w.pack_fo = cv.take<float>((size_t)2 * sd.d_o * m.L[1]);
  w.total = cv.off;
  return w;
}

static size_t fold_in_workspace_bytes(const MrModel* model, bool items, int64_t U, int64_t nnz) {
  if (check_model(model) != MR_OK || U < 0 || U > INT32_MAX || nnz < 0 || nnz > INT32_MAX) return 0;
  return carve_fold_in(*model, fold_side(*model, items), U, nullptr).total;
}

size_t mr_fold_in_workspace_bytes(const MrModel* model, int64_t U, int64_t nnz) {
  return fold_in_workspace_bytes(model, false, U, nnz);
}

size_t mr_fold_in_items_workspace_bytes(const MrModel* model, int64_t M, int64_t nnz) {
  return fold_in_workspace_bytes(model, true, M, nnz);
}

// The words of one direction's error messages.
struct FoldNames {
  const char *fn, *self, *other_id, *init, *covers;
};
static const FoldNames kFoldUsers = {"fold_in", "user", "an item id", "an init user", "a history covers every item"};
static const FoldNames kFoldItems = {"fold_in_items", "item", "a user id", "an init item",
                                     "a rater list covers every user"};

static int fold_in_call(const MrModel* model, bool items, const int64_t* rowptr, const int32_t* ids, int64_t U,
                        int64_t nnz, const int32_t* init_rows, const MrFoldIn* cfg, float* out_mlp, float* out_gmf,
                        float* out_loss, void* ws, size_t ws_bytes, void* stream) {
  int rc = check_model(model);
  if (rc != MR_OK) return rc;
  const MrModel& m = *model;
  const FoldNames& nm = items ? kFoldItems : kFoldUsers;
  const char* fn = nm.fn;
  cudaStream_t st = (cudaStream_t)stream;
  MR_REQUIRE(cfg != nullptr, "%s: cfg is NULL", fn);
  MR_REQUIRE(cfg->steps >= 0, "%s: steps=%d must be >= 0", fn, cfg->steps);
  MR_REQUIRE(cfg->negs >= 1 && cfg->negs <= MR_MAX_NEGS, "%s: negs=%d out of [1,%d]", fn, cfg->negs, MR_MAX_NEGS);
  MR_REQUIRE(cfg->optimizer == MR_OPT_ADAM || cfg->optimizer == MR_OPT_SGD, "%s: unknown optimizer %d", fn,
             cfg->optimizer);
  MR_REQUIRE(isfinite(cfg->lr), "%s: lr must be finite", fn);
  if (cfg->optimizer == MR_OPT_ADAM)
    MR_REQUIRE(cfg->beta_1 >= 0.f && cfg->beta_1 < 1.f && cfg->beta_2 >= 0.f && cfg->beta_2 < 1.f && cfg->epsilon > 0.f,
               "%s: Adam needs beta_1, beta_2 in [0, 1) and epsilon > 0", fn);
  MR_REQUIRE(U >= 0 && U <= INT32_MAX && nnz >= 0 && nnz <= INT32_MAX, "%s: bad sizes U=%lld nnz=%lld", fn,
             (long long)U, (long long)nnz);
  MR_REQUIRE(rowptr != nullptr, "%s: rowptr is NULL", fn);
  MR_REQUIRE(nnz == 0 || ids != nullptr, "%s: %s is NULL", fn, items ? "users" : "items");
  MR_REQUIRE(U == 0 || out_mlp != nullptr, "%s: out_%s_mlp is NULL", fn, nm.self);
  MR_REQUIRE(U == 0 || m.mf_dim == 0 || out_gmf != nullptr, "%s: out_%s_gmf is NULL but mf_dim > 0", fn, nm.self);
  const FoldSide sd = fold_side(m, items);
  MR_REQUIRE(fold_in_supported(m, sd), "%s: layer widths too large for the kernel's shared memory", fn);
  const FoldWs w = carve_fold_in(m, sd, U, ws);
  if (ws == nullptr || ws_bytes < w.total) {
    set_error("%s: workspace %zu bytes < %zu", fn, ws_bytes, w.total);
    return MR_ERR_WORKSPACE;
  }
  if (U == 0) return MR_OK;

  // the lists are checked before any other work: one small kernel and a one-word read-back
  MR_CUDA(cudaMemsetAsync(w.flags, 0, sizeof(int32_t), st));
  rc = launch_fold_in_check(rowptr, ids, U, nnz, sd.num_other, init_rows, sd.num_self, w.keys, w.flags, st);
  if (rc != MR_OK) return rc;
  int32_t bad = 0;
  MR_CUDA(cudaMemcpyAsync(&bad, w.flags, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  MR_CUDA(cudaStreamSynchronize(st));
  MR_REQUIRE(!(bad & 1), "%s: rowptr must start at 0, never decrease and end at nnz, and every list must be "
             "strictly ascending", fn);
  MR_REQUIRE(!(bad & 2), "%s: %s lies outside [0, %d)", fn, nm.other_id, sd.num_other);
  MR_REQUIRE(!(bad & 4), "%s: %s lies outside [-1, %d)", fn, nm.init, sd.num_self);
  MR_REQUIRE(!(bad & 8), "%s: %s: no negatives to draw", fn, nm.covers);

  rc = launch_sort_pairs(w.keys, U, bits_for((int64_t)sd.num_other + 1), w.sorted_keys, w.order, w.sort_ws,
                         w.sort_ws_bytes, st);
  if (rc == MR_OK) rc = launch_transpose_kernels(m, w.wt, st);
  if (rc == MR_OK && m.n_layers > 1) rc = project_other_side(m, sd, w.pack_fo, w.Po, st);
  if (rc != MR_OK) return rc;
  FoldInArgs a{};
  a.model = model;
  a.side = sd;
  a.wt = w.wt;
  a.Po = w.Po;
  a.rowptr = rowptr;
  a.ids = ids;
  a.init_rows = init_rows;
  a.order = w.order;
  a.U = U;
  a.cfg = *cfg;
  a.out_mlp = out_mlp;
  a.out_gmf = out_gmf;
  a.out_loss = out_loss;
  return launch_fold_in(a, st);
}

int mr_fold_in_users(const MrModel* model, const int64_t* rowptr, const int32_t* items, int64_t U, int64_t nnz,
                     const int32_t* init_users, const MrFoldIn* cfg, float* out_user_mlp, float* out_user_gmf,
                     float* out_loss, void* ws, size_t ws_bytes, void* stream) {
  return fold_in_call(model, false, rowptr, items, U, nnz, init_users, cfg, out_user_mlp, out_user_gmf, out_loss, ws,
                      ws_bytes, stream);
}

int mr_fold_in_items(const MrModel* model, const int64_t* rowptr, const int32_t* users, int64_t M, int64_t nnz,
                     const int32_t* init_items, const MrFoldIn* cfg, float* out_item_mlp, float* out_item_gmf,
                     float* out_loss, void* ws, size_t ws_bytes, void* stream) {
  return fold_in_call(model, true, rowptr, users, M, nnz, init_items, cfg, out_item_mlp, out_item_gmf, out_loss, ws,
                      ws_bytes, stream);
}

// ---- similar items / users: the side's representation once per call (its first-layer part as fold-in projects the
// other side, then normalised and packed as a tensor-core operand), then per chunk of queries the representation of the
// queries, the score GEMM and the row selection without the query itself ----------------------------------------------
struct SimilarShape {
  FoldSide sd;       // its OTHER side is the side searched
  int L1, f, n_parts, Dpad;
  int64_t C, C_pad, N_pad;  // queries per chunk and the row counts of the two operand images
};

static SimilarShape similar_shape(const MrModel& m, int32_t side, int64_t M) {
  SimilarShape s{};
  s.sd = fold_side(m, side == MR_SIDE_USERS);
  s.L1 = m.n_layers >= 2 ? m.L[1] : 0;
  s.f = m.mf_dim;
  s.n_parts = (s.L1 > 0 ? 1 : 0) + (s.f > 0 ? 1 : 0);
  s.Dpad = (int)align_up((size_t)(s.L1 + s.f), 32);
  const int32_t N = s.sd.num_other;
  s.C = clamp_users(M, catalogue_chunk_users(N));
  s.C_pad = (int64_t)align_up((size_t)s.C, kSimTileQ);
  s.N_pad = (int64_t)align_up((size_t)N, kSimTileC);
  return s;
}

struct SimilarWs {
  float *P, *pack, *R, *A, *S;
  void* topk;
  size_t total;
};

static SimilarWs carve_similar(const MrModel& m, const SimilarShape& s, int32_t k, void* ws) {
  SimilarWs w{};
  Carver cv(ws);
  const int32_t N = s.sd.num_other;
  if (s.L1 > 0) w.P = cv.take<float>((size_t)N * s.L1);
  if (s.L1 > 0 && fold_in_tc_proj(m, s.sd)) w.pack = cv.take<float>((size_t)2 * s.sd.d_o * s.L1);
  w.R = cv.take<float>((size_t)2 * s.Dpad * s.N_pad);
  w.A = cv.take<float>((size_t)2 * s.Dpad * s.C_pad);
  w.S = cv.take<float>((size_t)s.C * N);
  w.topk = cv.take<char>(topk_workspace_bytes(s.C, N, k));
  w.total = cv.off;
  return w;
}

static int similar_check(const MrModel* model, int32_t side, int64_t M, int32_t k, int32_t excl_rows,
                         const int64_t* excl_rowptr, const int32_t* excl_list) {
  int rc = check_model(model);
  if (rc != MR_OK) return rc;
  MR_REQUIRE(side == MR_SIDE_ITEMS || side == MR_SIDE_USERS, "similar: side=%d is neither MR_SIDE_ITEMS nor "
             "MR_SIDE_USERS", side);
  MR_REQUIRE(k >= 1 && k <= MR_MAX_TOPK, "similar: k=%d out of [1,%d]", k, MR_MAX_TOPK);
  MR_REQUIRE(M >= 0 && M <= INT32_MAX, "similar: bad M=%lld", (long long)M);
  MR_REQUIRE(model->n_layers >= 2 || model->mf_dim > 0, "similar: a model with one layer and mf_dim == 0 has no "
             "vector to compare");
  MR_REQUIRE(excl_rows >= 0 && (excl_rowptr == nullptr || excl_list != nullptr), "similar: bad exclusion lists");
  return MR_OK;
}

size_t mr_similar_workspace_bytes(const MrModel* model, int32_t side, int64_t M, int32_t k) {
  if (similar_check(model, side, M, k, 0, nullptr, nullptr) != MR_OK) return 0;
  return carve_similar(*model, similar_shape(*model, side, M), k, nullptr).total;
}

int mr_similar(const MrModel* model, int32_t side, const int32_t* ids, int64_t M, int32_t k, const int32_t* excl_ids,
               int32_t excl_rows, const int64_t* excl_rowptr, const int32_t* excl_list, int32_t* top_ids,
               float* top_scores, float* scores, void* ws, size_t ws_bytes, void* stream) {
  int rc = similar_check(model, side, M, k, excl_rows, excl_rowptr, excl_list);
  if (rc != MR_OK) return rc;
  if (M == 0) return MR_OK;
  MR_REQUIRE(ids != nullptr && ws != nullptr, "similar: ids / ws is NULL");
  const MrModel& m = *model;
  const SimilarShape s = similar_shape(m, side, M);
  const SimilarWs w = carve_similar(m, s, k, ws);
  if (ws_bytes < w.total) {
    set_error("similar workspace too small: %zu < %zu", ws_bytes, w.total);
    return MR_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const FoldSide& sd = s.sd;
  const int32_t N = sd.num_other;
  prof_mark(MR_PHASE_MISC, st);
  if (s.L1 > 0) rc = project_other_side(m, sd, w.pack, w.P, st);
  if (rc == MR_OK)
    rc = launch_similar_pack(w.P, s.L1, sd.other_gmf, m.w_out, s.f, N, nullptr, N, s.N_pad, s.Dpad, s.n_parts, w.R, st);
  TopkArgs a{};
  a.N = N;
  a.k = k;
  a.excl_ids = excl_ids;
  a.excl_rows = excl_rows;
  a.excl_rowptr = excl_rowptr;
  a.excl_items = excl_list;
  a.users = ids;  // an out-of-range query gets -1 / NaN; the query's own id is left out of its selection
  a.num_users = N;
  a.top_items = top_ids;
  a.top_scores = top_scores;
  for (int64_t q0 = 0; q0 < M && rc == MR_OK; q0 += s.C) {
    const int64_t c = M - q0 < s.C ? M - q0 : s.C;
    float* out = scores != nullptr ? scores + q0 * N : w.S;
    prof_mark(MR_PHASE_MISC, st);
    rc = launch_similar_pack(w.P, s.L1, sd.other_gmf, m.w_out, s.f, N, ids + q0, c, s.C_pad, s.Dpad, s.n_parts, w.A,
                             st);
    if (rc != MR_OK) break;
    prof_mark(MR_PHASE_TC_DENSE_FWD, st);
    rc = launch_similar_gemm(w.A, s.C_pad, w.R, s.N_pad, s.Dpad, c, N, out, st);
    if (rc != MR_OK || (top_ids == nullptr && top_scores == nullptr)) continue;
    prof_mark(MR_PHASE_RANK, st);
    a.u0 = q0;
    a.U = c;
    a.scores = out;
    rc = launch_topk(a, w.topk, st, true);
  }
  prof_mark(-1, st);
  return rc;
}

int mr_users_grouped(const int32_t* users, int64_t n, int32_t group, int32_t* flag, void* stream) {
  MR_REQUIRE(users != nullptr && flag != nullptr, "users_grouped: NULL pointer");
  MR_REQUIRE(n >= 0 && group >= 1, "users_grouped: bad sizes");
  return launch_check_grouped(users, n, group, flag, (cudaStream_t)stream);
}

size_t mr_sparse_rows_workspace_bytes(int64_t n, int32_t d0, int32_t d1) {
  if (n < 0) return 0;
  return align_up((size_t)n * 4, 256) * 2 + sort_workspace_bytes(n) + segreduce_workspace_bytes(n, d0 + d1) + 256;
}

int mr_sparse_rows_update(float* table0, float* m0, float* v0, int32_t d0, float* table1, float* m1, float* v1,
                          int32_t d1, int32_t num_rows, const int32_t* row_ids, const float* grad_rows, int64_t n,
                          int32_t optimizer, float lr, float lr_t, float beta_1, float beta_2, float epsilon,
                          void* ws, size_t ws_bytes, void* stream) {
  if (n == 0) return MR_OK;
  MR_REQUIRE(table0 && row_ids && grad_rows && ws, "sparse_rows_update: NULL pointer");
  MR_REQUIRE(d0 > 0 && d1 >= 0 && num_rows > 0 && n > 0 && n < ((int64_t)1 << 31), "sparse_rows_update: bad sizes");
  MR_REQUIRE(optimizer == MR_OPT_SGD || (m0 && v0 && (d1 == 0 || (m1 && v1))), "sparse_rows_update: Adam state is NULL");
  MR_REQUIRE(d1 == 0 || table1 != nullptr, "sparse_rows_update: table1 is NULL");
  if (ws_bytes < mr_sparse_rows_workspace_bytes(n, d0, d1)) {
    set_error("sparse_rows_update workspace too small");
    return MR_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  Carver cv(ws);
  int32_t* skeys = cv.take<int32_t>(n);
  int32_t* sidx = cv.take<int32_t>(n);
  const size_t sort_bytes = sort_workspace_bytes(n);
  void* sort_ws = cv.take<char>(sort_bytes);
  const size_t seg_bytes = segreduce_workspace_bytes(n, d0 + d1);
  void* seg_ws = cv.take<char>(seg_bytes);
  prof_mark(MR_PHASE_SORT, st);
  int rc = sort_row_ids(row_ids, n, num_rows, skeys, sidx, sort_ws, sort_bytes, st);
  if (rc != MR_OK) return rc;
  RowUpdate u{};
  u.mode = MR_TABLES_SPARSE;
  u.optimizer = optimizer;
  u.lr = lr;
  u.lr_t = lr_t;
  u.beta_1 = beta_1;
  u.beta_2 = beta_2;
  u.epsilon = epsilon;
  u.d0 = d0;
  u.d1 = d1;
  u.num_rows = num_rows;
  u.p0 = table0; u.m0 = m0; u.v0 = v0;
  u.p1 = table1; u.m1 = m1; u.v1 = v1;
  prof_mark(MR_PHASE_SEGREDUCE, st);
  rc = launch_segreduce(skeys, sidx, n, grad_rows, u, seg_ws, seg_bytes, st);
  prof_mark(-1, st);
  return rc;
}

int mr_uses_item_projection(const MrModel* model, int64_t rows) {
  if (model == nullptr || model->n_layers < 1 || model->n_layers > MR_MAX_LAYERS) return 0;
  return item_proj_ok(*model, rows) ? 1 : 0;
}

int mr_uses_user_projection(const MrModel* model, int64_t rows, int32_t group) {
  if (model == nullptr || model->n_layers < 1 || model->n_layers > MR_MAX_LAYERS) return 0;
  return user_proj_ok(*model, rows, group) ? 1 : 0;
}

int mr_uses_small_tower(const MrModel* model, int64_t rows, int32_t group) {
  if (model == nullptr || model->n_layers < 1 || model->n_layers > MR_MAX_LAYERS) return 0;
  return small_proj_ok(*model, rows, group) ? 1 : 0;
}

int mr_uses_tensor_cores(const MrModel* model) {
  if (model == nullptr || model->n_layers < 1 || model->n_layers > MR_MAX_LAYERS) return 0;
  return use_tc(*model) ? 1 : 0;
}

int mr_profile_begin(void) {
  g_prof.on = true;
  g_prof.overflow = false;
  g_prof.used = 0;
  g_prof.launches = 0;
  return MR_OK;
}

int mr_profile_end(float* phase_ms, int64_t* phase_count, int64_t* kernel_launches) {
  Profiler& p = g_prof;
  MR_REQUIRE(p.on, "mr_profile_end without mr_profile_begin");
  p.on = false;
  for (int i = 0; i < MR_NUM_PHASES; ++i) {
    if (phase_ms) phase_ms[i] = 0.f;
    if (phase_count) phase_count[i] = 0;
  }
  if (kernel_launches) *kernel_launches = p.launches;
  if (p.used > 0) MR_CUDA(cudaEventSynchronize(p.events[p.used - 1]));
  for (size_t i = 0; i + 1 < p.used; ++i) {
    const int ph = p.phase[i];
    if (ph < 0 || ph >= MR_NUM_PHASES) continue;
    float ms = 0.f;
    MR_CUDA(cudaEventElapsedTime(&ms, p.events[i], p.events[i + 1]));
    if (phase_ms) phase_ms[ph] += ms;
    if (phase_count) phase_count[ph] += 1;
  }
  p.used = 0;
  MR_REQUIRE(!p.overflow, "profile event buffer overflowed; profile fewer steps");
  return MR_OK;
}

size_t mr_split_workspace_bytes(int64_t n) { return split_workspace_bytes(n < 0 ? 0 : n); }

int mr_split_last_two(const int32_t* users, int64_t n, int32_t num_users, int32_t* order, int32_t* part, int32_t* flag,
                      void* ws, size_t ws_bytes, void* stream) {
  MR_REQUIRE(n >= 0 && n < ((int64_t)1 << 31) && num_users > 0, "split: bad n / num_users");
  if (n == 0) return MR_OK;
  MR_REQUIRE(users && order && part && flag && ws, "split: NULL pointer");
  return launch_split_last_two(users, n, num_users, order, part, flag, ws, ws_bytes, (cudaStream_t)stream);
}

size_t mr_remap_workspace_bytes(int64_t n) { return remap_workspace_bytes(n < 0 ? 0 : n); }

int mr_remap_ids(const int32_t* ids, int64_t n, int32_t id_limit, int32_t* dense_ids, int32_t* unique_ids,
                 int64_t* num_unique, int32_t* flag, void* ws, size_t ws_bytes, void* stream) {
  MR_REQUIRE(n >= 0 && n < ((int64_t)1 << 31) && id_limit > 0, "remap: bad n / id_limit");
  MR_REQUIRE(num_unique && flag && ws && (n == 0 || (ids && dense_ids && unique_ids)), "remap: NULL pointer");
  return launch_remap_ids(ids, n, id_limit, dense_ids, unique_ids, num_unique, flag, ws, ws_bytes, (cudaStream_t)stream);
}

size_t mr_user_csr_workspace_bytes(int64_t n) { return user_csr_workspace_bytes(n < 0 ? 0 : n); }

int mr_build_user_csr(const int32_t* users, const int32_t* items, int64_t n, int32_t num_users, int32_t num_items,
                      int64_t* rowptr, int32_t* csr_items, int32_t* flag, void* ws, size_t ws_bytes, void* stream) {
  MR_REQUIRE(n >= 0 && n < ((int64_t)1 << 31) && num_users > 0 && num_items > 0, "user csr: bad sizes");
  MR_REQUIRE(rowptr && flag && ws && (n == 0 || (users && items && csr_items)), "user csr: NULL pointer");
  return launch_build_user_csr(users, items, n, num_users, num_items, rowptr, csr_items, flag, ws, ws_bytes,
                               (cudaStream_t)stream);
}

size_t mr_sort_workspace_bytes(int64_t n) { return sort_workspace_bytes(n < 0 ? 0 : n); }

int mr_sort_pairs(const int32_t* keys, int64_t n, int32_t key_bits, int32_t* sorted_keys, int32_t* sorted_index,
                  void* ws, size_t ws_bytes, void* stream) {
  MR_REQUIRE(keys && sorted_keys && sorted_index && ws, "sort_pairs: NULL pointer");
  MR_REQUIRE(n >= 0 && key_bits >= 1 && key_bits <= 32, "sort_pairs: bad n/key_bits");
  return launch_sort_pairs(keys, n, key_bits, sorted_keys, sorted_index, ws, ws_bytes, (cudaStream_t)stream);
}

int mr_optimizer_flat(float* p, const float* g, float* m, float* v, int64_t n, int32_t optimizer, float lr_t,
                      float beta_1, float beta_2, float epsilon, float l2, void* stream) {
  MR_REQUIRE(p && g && n >= 0, "optimizer_flat: NULL pointer");
  MR_REQUIRE(optimizer == MR_OPT_SGD || (m && v), "optimizer_flat: Adam needs m and v");
  return launch_optimizer_flat(p, g, m, v, n, optimizer, lr_t, beta_1, beta_2, epsilon, l2, (cudaStream_t)stream);
}

int mr_dp_reduce_apply(const float* const* grad_peers, float* const* param_peers, int32_t world, int32_t rank, float* m,
                       float* v, int64_t lo, int64_t hi, int32_t optimizer, float lr_t, float beta_1, float beta_2,
                       float epsilon, float l2, const float* grad_multicast, float* param_multicast, void* stream) {
  MR_REQUIRE(grad_peers && param_peers, "dp_reduce_apply: NULL pointer array");
  MR_REQUIRE((world >= 1 && world <= 8) || world == 16, "dp_reduce_apply: world size %d (1..8 or 16 ranks of one box)",
             world);
  MR_REQUIRE(rank >= 0 && rank < world, "dp_reduce_apply: rank %d of %d", rank, world);
  MR_REQUIRE(lo >= 0 && hi >= lo && (lo & 3) == 0 && (hi & 3) == 0, "dp_reduce_apply: [lo, hi) must be multiples of 4");
  MR_REQUIRE(optimizer == MR_OPT_SGD || (m && v), "dp_reduce_apply: Adam needs m and v");
  MR_REQUIRE(optimizer == MR_OPT_SGD || ((reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v)) & 15) == 0,
             "dp_reduce_apply: m and v must be 16-byte aligned");
  for (int r = 0; r < world; ++r)
    MR_REQUIRE(grad_peers[r] && param_peers[r] && ((reinterpret_cast<uintptr_t>(grad_peers[r]) |
                                                     reinterpret_cast<uintptr_t>(param_peers[r])) & 15) == 0,
               "dp_reduce_apply: rank %d's pointers must be non-NULL and 16-byte aligned", r);
  MR_REQUIRE((grad_multicast == nullptr) == (param_multicast == nullptr) &&
                 ((reinterpret_cast<uintptr_t>(grad_multicast) | reinterpret_cast<uintptr_t>(param_multicast)) & 15) == 0,
             "dp_reduce_apply: multicast addresses come as a 16-byte aligned pair or not at all");
  return launch_dp_reduce_apply(grad_peers, param_peers, world, rank, m, v, lo, hi, optimizer, lr_t, beta_1, beta_2,
                                epsilon, l2, grad_multicast, param_multicast, (cudaStream_t)stream);
}

}  // extern "C"
