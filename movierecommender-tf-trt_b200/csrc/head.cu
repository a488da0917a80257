// NeuMF head (tensor-core path): GMF product, output unit, sigmoid, BCE and their gradients, fused in
// one HBM-bound pass over the rows (model.py:184-188 and 213-215; GMF branch per He et al. 2017).
//   z = b_o + w_o[:f].(gu*gi) + w_o[f:].h ,  p = sigmoid(z) ,  loss += bce(z, y)
//   dz = (p - y) / B_global ;  dh = dz * w_o[f:] * (h > 0)  -> dz_last (enters the tower's backward)
//   d gu = dz * w_o[:f] * gi , d gi = dz * w_o[:f] * gu     -> GMF columns of the staged row gradients
//   d w_o = sum_r dz * [gu*gi | h] , d b_o = sum_r dz       -> per-warp partials, reduced in fixed order
// One warp per row, lanes across columns (every row is read with coalesced 128-byte requests).
// Algorithmic bytes per row: 4*L_last (h) + 8*f (GMF rows) + 12 (ids, label) read,
// 4*L_last + 8*f + 8 written.
#include "launchers.h"

namespace mr {

constexpr int kHeadThreads = 256;
constexpr int kHeadMaxQ = 16;  // (f + L_last) / 32 columns per lane at most (f + L_last <= 512)

struct HeadParams {
  MrModel m;
  const float* h_last;
  const int32_t* users;
  const int32_t* items;
  const float* labels;
  int64_t rows, row0;
  int32_t user_div;
  int32_t group;  // > 0: grouped batch -- a warp takes whole groups and stages ONE GMF user-gradient row per group
  float inv_batch;
  float* logits;
  float* probs;
  float* dz_last;
  float* stage_u;
  float* stage_i;
  float* head_partial;  // [grid][ncols + 2]: d w_out (ncols), d b_out, loss
  int32_t* flags;
};

// MAXQ = columns per lane (compile-time so the per-lane arrays stay in registers and small models get
// high occupancy: the kernel is latency/HBM bound).  KR = rows per warp and iteration.  GROUPED: the KR rows
// are one group of a grouped batch (same user): the GMF user row is read once and its gradient, summed over
// the group in row order, is staged once at row (row0 / KR + group index) of stage_u.
template <int MAXQ, int KR, bool GROUPED>
__global__ void __launch_bounds__(kHeadThreads, MAXQ <= 4 ? 2 : 1) head_kernel(const HeadParams p) {
  __shared__ float red[kHeadThreads / 32][MAXQ * 32 + 2];
  const MrModel& m = p.m;
  const int f = m.mf_dim, Ln = m.L[m.n_layers - 1], ncols = f + Ln;
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u;
  const int su = d_u + f, si = d_i + f;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool train = p.labels != nullptr;
  float accw[MAXQ];
#pragma unroll
  for (int q = 0; q < MAXQ; ++q) accw[q] = 0.f;
  float accb = 0.f, accl = 0.f;

  // kRows rows per warp and iteration, phases interleaved across the rows (ids of all rows, then all
  // row loads, then the reductions, then the stores): the kernel is latency-bound, so the loads of
  // several independent rows must be in flight together.  The order in which a warp folds rows into
  // its d w_out / d b_out / loss sums is fixed (rr = 0..kRows-1), so results stay deterministic.
  constexpr int kRows = KR;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  for (int64_t base = w0 * kRows; base < p.rows; base += warps * kRows) {
    int u[kRows], it[kRows];
    bool live[kRows], bad[kRows];
#pragma unroll
    for (int rr = 0; rr < kRows; ++rr) {
      const int64_t lr = base + rr;
      live[rr] = lr < p.rows;
      u[rr] = 0;
      it[rr] = 0;
      if (live[rr]) {
        u[rr] = __ldg(p.users + (GROUPED ? p.row0 + base : (p.row0 + lr) / p.user_div));
        it[rr] = __ldg(p.items + p.row0 + lr);
      }
    }
    float gu_acc[MAXQ];  // GROUPED: gradient of the group's GMF user row
#pragma unroll
    for (int q = 0; q < MAXQ; ++q) gu_acc[q] = 0.f;
    // column j of the head input: j < f -> gu[j]*gi[j], else h[j - f]; lane owns columns lane + 32q
    float hv[kRows][MAXQ], ga[kRows][MAXQ], gb[kRows][MAXQ];
#pragma unroll
    for (int rr = 0; rr < kRows; ++rr) {
      bad[rr] = (unsigned)u[rr] >= (unsigned)m.num_users || (unsigned)it[rr] >= (unsigned)m.num_items;
      if (bad[rr]) {
        if (lane == 0) atomicOr(p.flags, 1);
        u[rr] = 0;
        it[rr] = 0;
      }
      const int64_t lr = base + rr;
#pragma unroll
      for (int q = 0; q < MAXQ; ++q) {
        const int j = lane + 32 * q;
        hv[rr][q] = 0.f;
        ga[rr][q] = 0.f;
        gb[rr][q] = 0.f;
        if (live[rr]) {
          if (j < f) {
            ga[rr][q] = (GROUPED && rr > 0) ? ga[0][q] : __ldg(m.user_gmf + (size_t)u[rr] * f + j);
            gb[rr][q] = __ldg(m.item_gmf + (size_t)it[rr] * f + j);
          } else if (j < ncols) {
            hv[rr][q] = __ldg(p.h_last + (size_t)lr * Ln + (j - f));
          }
        }
      }
    }
    float wv[MAXQ];
#pragma unroll
    for (int q = 0; q < MAXQ; ++q) wv[q] = (lane + 32 * q < ncols) ? __ldg(m.w_out + lane + 32 * q) : 0.f;
    const float b_out = __ldg(m.b_out);
#pragma unroll
    for (int rr = 0; rr < kRows; ++rr) {
      if (!live[rr]) continue;  // warp-uniform
      const int64_t lr = base + rr, gr = p.row0 + lr;
      float s = 0.f;
#pragma unroll
      for (int q = 0; q < MAXQ; ++q) {
        if (lane + 32 * q < f) hv[rr][q] = ga[rr][q] * gb[rr][q];
        s = fmaf(wv[q], hv[rr][q], s);
      }
      s = warp_sum(s);
      const float z = s + b_out;
      const float pr = sigmoidf_stable(z);
      if (lane == 0) {
        if (p.logits != nullptr) p.logits[gr] = bad[rr] ? nanf("") : z;
        if (p.probs != nullptr) p.probs[gr] = bad[rr] ? nanf("") : pr;
      }
      if (train) {
        const float y = __ldg(p.labels + gr);
        const float dz = bad[rr] ? 0.f : (pr - y) * p.inv_batch;
        if (!bad[rr]) accl += bce_logits(z, y);
        accb += dz;
#pragma unroll
        for (int q = 0; q < MAXQ; ++q) {
          const int j = lane + 32 * q;
          if (j < ncols) {
            accw[q] = fmaf(dz, hv[rr][q], accw[q]);
            const float g = dz * wv[q];
            if (j < f) {
              if (GROUPED) gu_acc[q] = fmaf(g, gb[rr][q], gu_acc[q]);
              else p.stage_u[(size_t)gr * su + d_u + j] = g * gb[rr][q];
              p.stage_i[(size_t)gr * si + d_i + j] = g * ga[rr][q];
            } else {
              p.dz_last[(size_t)lr * Ln + (j - f)] = hv[rr][q] > 0.f ? g : 0.f;
            }
          }
        }
      }
    }
    if (GROUPED && train && live[0]) {
      const int64_t grp = (p.row0 + base) / kRows;
#pragma unroll
      for (int q = 0; q < MAXQ; ++q) {
        const int j = lane + 32 * q;
        if (j < f) p.stage_u[(size_t)grp * su + d_u + j] = gu_acc[q];
      }
    }
  }
  if (train) {
    // per-warp sums -> shared -> this CTA's partial row, warps added in index order
#pragma unroll
    for (int q = 0; q < MAXQ; ++q) red[warp][lane + 32 * q] = accw[q];
    if (lane == 0) {
      red[warp][MAXQ * 32] = accb;  // every lane holds the same accb / accl
      red[warp][MAXQ * 32 + 1] = accl;
    }
    __syncthreads();
    float* dst = p.head_partial + (size_t)blockIdx.x * (ncols + 2);
    for (int j = threadIdx.x; j < ncols + 2; j += blockDim.x) {
      const int src = j < ncols ? j : MAXQ * 32 + (j - ncols);
      float t = 0.f;
      for (int w = 0; w < kHeadThreads / 32; ++w) t += red[w][src];
      dst[j] += t;  // the partial rows are zeroed once per step and accumulate over the step's launches
    }
  }
}

// Grouped train head, specialised and software-pipelined: mf_dim = 32 * FQ and the last layer width = 32 * HQ are
// compile-time, so a row's values take FQ + HQ registers per lane instead of MAXQ for each of three arrays, and
// the freed registers hold the NEXT group: its row loads are issued before the current group is reduced and its
// ids one group earlier still (the generic kernel above has no load in flight while it waits for ids or while
// it reduces and stores: ncu showed it at ~2 TB/s of its ~1.5 GB per step).  Same arithmetic per row, same
// outputs, same per-warp accumulation order as head_kernel<.., GROUPED = true>.
template <int FQ, int HQ, int KR>
__global__ void __launch_bounds__(kHeadThreads, 2) head_group_kernel(const HeadParams p) {
  constexpr int f = 32 * FQ, Ln = 32 * HQ, ncols = f + Ln;
  __shared__ float red[kHeadThreads / 32][ncols + 2];
  const MrModel& m = p.m;
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u;
  const int su = d_u + f, si = d_i + f;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float wg[FQ], wh[HQ];
#pragma unroll
  for (int q = 0; q < FQ; ++q) wg[q] = __ldg(m.w_out + lane + 32 * q);
#pragma unroll
  for (int q = 0; q < HQ; ++q) wh[q] = __ldg(m.w_out + f + lane + 32 * q);
  const float b_out = __ldg(m.b_out);
  float accg[FQ], acch[HQ], accb = 0.f, accl = 0.f;
#pragma unroll
  for (int q = 0; q < FQ; ++q) accg[q] = 0.f;
#pragma unroll
  for (int q = 0; q < HQ; ++q) acch[q] = 0.f;

  struct Ids {
    int u, it[KR];
    float y[KR];
  };
  struct Rows {
    float gu[FQ], gi[KR][FQ], h[KR][HQ], y[KR];
    unsigned bad;  // bit rr: row rr has an out-of-range id
  };
  const int64_t ngroups = p.rows / KR;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  auto load_ids = [&](int64_t g, Ids& d) {
    const int64_t gr0 = p.row0 + g * KR;
    d.u = __ldg(p.users + gr0);
#pragma unroll
    for (int rr = 0; rr < KR; ++rr) {
      d.it[rr] = __ldg(p.items + gr0 + rr);
      d.y[rr] = __ldg(p.labels + gr0 + rr);
    }
  };
  auto load_rows = [&](int64_t g, const Ids& d, Rows& r) {
    const bool bad_u = (unsigned)d.u >= (unsigned)m.num_users;
    const int u = bad_u ? 0 : d.u;
    r.bad = 0;
#pragma unroll
    for (int q = 0; q < FQ; ++q) r.gu[q] = __ldg(m.user_gmf + (size_t)u * f + lane + 32 * q);
#pragma unroll
    for (int rr = 0; rr < KR; ++rr) {
      const bool bad_i = (unsigned)d.it[rr] >= (unsigned)m.num_items;
      const int it = bad_i ? 0 : d.it[rr];
      if (bad_u || bad_i) r.bad |= 1u << rr;
      r.y[rr] = d.y[rr];
#pragma unroll
      for (int q = 0; q < FQ; ++q) r.gi[rr][q] = __ldg(m.item_gmf + (size_t)it * f + lane + 32 * q);
#pragma unroll
      for (int q = 0; q < HQ; ++q) r.h[rr][q] = __ldg(p.h_last + (size_t)(g * KR + rr) * Ln + lane + 32 * q);
    }
  };
  auto compute = [&](int64_t g, const Rows& r) {
    if (r.bad && lane == 0) atomicOr(p.flags, 1);
    float gu_acc[FQ];
#pragma unroll
    for (int q = 0; q < FQ; ++q) gu_acc[q] = 0.f;
#pragma unroll
    for (int rr = 0; rr < KR; ++rr) {
      const int64_t lr = g * KR + rr, gr = p.row0 + lr;
      float x[FQ];
      float s = 0.f;
#pragma unroll
      for (int q = 0; q < FQ; ++q) {
        x[q] = r.gu[q] * r.gi[rr][q];
        s = fmaf(wg[q], x[q], s);
      }
#pragma unroll
      for (int q = 0; q < HQ; ++q) s = fmaf(wh[q], r.h[rr][q], s);
      s = warp_sum(s);
      const float z = s + b_out;
      const float pr = sigmoidf_stable(z);
      const bool bad = (r.bad >> rr) & 1u;
      if (lane == 0 && p.probs != nullptr) p.probs[gr] = bad ? nanf("") : pr;
      const float y = r.y[rr];
      const float dz = bad ? 0.f : (pr - y) * p.inv_batch;
      if (!bad) accl += bce_logits(z, y);
      accb += dz;
#pragma unroll
      for (int q = 0; q < FQ; ++q) {
        accg[q] = fmaf(dz, x[q], accg[q]);
        const float gv = dz * wg[q];
        gu_acc[q] = fmaf(gv, r.gi[rr][q], gu_acc[q]);
        p.stage_i[(size_t)gr * si + d_i + lane + 32 * q] = gv * r.gu[q];
      }
#pragma unroll
      for (int q = 0; q < HQ; ++q) {
        acch[q] = fmaf(dz, r.h[rr][q], acch[q]);
        p.dz_last[(size_t)lr * Ln + lane + 32 * q] = r.h[rr][q] > 0.f ? dz * wh[q] : 0.f;
      }
    }
    const int64_t grp = (p.row0 + g * KR) / KR;
#pragma unroll
    for (int q = 0; q < FQ; ++q) p.stage_u[(size_t)grp * su + d_u + lane + 32 * q] = gu_acc[q];
  };

  Ids ids;
  Rows ra, rb;
  int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (g < ngroups) {
    load_ids(g, ids);
    load_rows(g, ids, ra);
    if (g + warps < ngroups) load_ids(g + warps, ids);
  }
  while (g < ngroups) {
    // ra holds group g; ids hold group g + warps
    if (g + warps < ngroups) {
      load_rows(g + warps, ids, rb);
      if (g + 2 * warps < ngroups) load_ids(g + 2 * warps, ids);
    }
    compute(g, ra);
    g += warps;
    if (g >= ngroups) break;
    if (g + warps < ngroups) {
      load_rows(g + warps, ids, ra);
      if (g + 2 * warps < ngroups) load_ids(g + 2 * warps, ids);
    }
    compute(g, rb);
    g += warps;
  }

  // per-warp sums -> shared -> this CTA's partial row, warps added in index order
#pragma unroll
  for (int q = 0; q < FQ; ++q) red[warp][lane + 32 * q] = accg[q];
#pragma unroll
  for (int q = 0; q < HQ; ++q) red[warp][f + lane + 32 * q] = acch[q];
  if (lane == 0) {
    red[warp][ncols] = accb;
    red[warp][ncols + 1] = accl;
  }
  __syncthreads();
  float* dst = p.head_partial + (size_t)blockIdx.x * (ncols + 2);
  for (int j = threadIdx.x; j < ncols + 2; j += blockDim.x) {
    float t = 0.f;
    for (int w = 0; w < kHeadThreads / 32; ++w) t += red[w][j];
    dst[j] += t;
  }
}

// Grouped train head, third form (mf_dim = 64, last width = 64, groups of at most 5 rows): EIGHT LANES PER ROW.  A
// quad of eight lanes owns a whole group -- its user GMF row, the KR rows of H_last and of item GMF rows, the group's
// user-gradient row -- so a warp instruction moves four rows with 128-bit accesses (128 contiguous bytes per quad),
// a row's dot product folds with three shuffles instead of five, and all 4 * KR rows of a warp iteration are in
// flight together while the next iteration's ids are already on their way.  ncu on the warp-per-row kernels above:
// 60 % issue-active at 3 TB/s -- instruction-bound, not HBM-bound; this layout issues a quarter of the memory
// instructions per row.  Same arithmetic per row; the sums over rows (d w_out, d b_out, loss) fold per quad in row
// order, then quads and warps in index order (deterministic).
constexpr int kQuadThreads = 128;
template <int KR>
__global__ void __launch_bounds__(kQuadThreads) head_quad_kernel(const HeadParams p) {
  constexpr int f = 64, Ln = 64, ncols = f + Ln, NV = 2;
  constexpr int kWarps = kQuadThreads / 32;
  __shared__ __align__(16) float red[kWarps * 4][ncols + 4];  // rows of 16-byte multiples: the lanes store float4
  const MrModel& m = p.m;
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u;
  const int su = d_u + f, si = d_i + f;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane & 7, quad = lane >> 3;
  float4 wg[NV], wh[NV], accg[NV], acch[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    wg[v] = ldg4(m.w_out + 32 * v + 4 * sub);
    wh[v] = ldg4(m.w_out + f + 32 * v + 4 * sub);
    accg[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    acch[v] = accg[v];
  }
  const float b_out = __ldg(m.b_out);
  float accb = 0.f, accl = 0.f;
  const int64_t ngroups = p.rows / KR;
  const int64_t nwarps = (int64_t)gridDim.x * kWarps;

  // ids of a warp iteration (groups g0 .. g0 + 3 = rows g0 * KR .. + 4 * KR - 1), lane-distributed; the quad's user
  auto load_ids = [&](int64_t g0, int& item, float& y, int& u) {
    const int64_t r0 = g0 * KR, left = p.rows - r0;
    item = 0;
    y = 0.f;
    if (lane < 4 * KR && lane < left) {
      item = __ldg(p.items + p.row0 + r0 + lane);
      y = __ldg(p.labels + p.row0 + r0 + lane);
    }
    const int64_t g = g0 + quad;
    u = g < ngroups ? __ldg(p.users + p.row0 + g * KR) : 0;
  };
  int64_t itn = (int64_t)blockIdx.x * kWarps + warp;
  int item_c = 0, u_c = 0, item_n = 0, u_n = 0;
  float y_c = 0.f, y_n = 0.f;
  if (4 * itn < ngroups) load_ids(4 * itn, item_c, y_c, u_c);
  for (; 4 * itn < ngroups; itn += nwarps) {
    const int64_t g = 4 * itn + quad;
    const bool live = g < ngroups;
    if (4 * (itn + nwarps) < ngroups) load_ids(4 * (itn + nwarps), item_n, y_n, u_n);
    const bool bad_u = live && (unsigned)u_c >= (unsigned)m.num_users;
    const int uu = (bad_u || !live) ? 0 : u_c;
    const int64_t lr0 = (live ? g : 0) * KR;  // launch-local first row of the quad's group (dead quads re-read group 0)
    float4 gu[NV], gi[KR][NV], h[KR][NV];
    int itv[KR];
    float yv[KR];
#pragma unroll
    for (int rr = 0; rr < KR; ++rr) {
      itv[rr] = __shfl_sync(0xffffffffu, item_c, quad * KR + rr);
      yv[rr] = __shfl_sync(0xffffffffu, y_c, quad * KR + rr);
    }
#pragma unroll
    for (int v = 0; v < NV; ++v) gu[v] = ldg4(m.user_gmf + (size_t)uu * f + 32 * v + 4 * sub);
#pragma unroll
    for (int rr = 0; rr < KR; ++rr) {
      const int iv = (unsigned)itv[rr] >= (unsigned)m.num_items ? 0 : itv[rr];
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        gi[rr][v] = ldg4(m.item_gmf + (size_t)iv * f + 32 * v + 4 * sub);
        h[rr][v] = ldg4(p.h_last + (size_t)(lr0 + rr) * Ln + 32 * v + 4 * sub);
      }
    }
    float4 gu_acc[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) gu_acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    bool any_bad = false;
#pragma unroll
    for (int rr = 0; rr < KR; ++rr) {
      const int64_t lr = lr0 + rr, gr = p.row0 + lr;
      float4 x[NV];
      float s = 0.f;
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        x[v] = make_float4(gu[v].x * gi[rr][v].x, gu[v].y * gi[rr][v].y, gu[v].z * gi[rr][v].z, gu[v].w * gi[rr][v].w);
        s = fmaf(wg[v].x, x[v].x, s);
        s = fmaf(wg[v].y, x[v].y, s);
        s = fmaf(wg[v].z, x[v].z, s);
        s = fmaf(wg[v].w, x[v].w, s);
      }
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        s = fmaf(wh[v].x, h[rr][v].x, s);
        s = fmaf(wh[v].y, h[rr][v].y, s);
        s = fmaf(wh[v].z, h[rr][v].z, s);
        s = fmaf(wh[v].w, h[rr][v].w, s);
      }
      s += __shfl_xor_sync(0xffffffffu, s, 1);
      s += __shfl_xor_sync(0xffffffffu, s, 2);
      s += __shfl_xor_sync(0xffffffffu, s, 4);
      const float z = s + b_out;
      const float pr = sigmoidf_stable(z);
      const bool bad = bad_u || (unsigned)itv[rr] >= (unsigned)m.num_items;
      any_bad |= bad && live;
      if (live && sub == 0 && p.probs != nullptr) p.probs[gr] = bad ? nanf("") : pr;
      const float y = yv[rr];
      const float dz = (bad || !live) ? 0.f : (pr - y) * p.inv_batch;
      if (live && !bad) accl += bce_logits(z, y);
      accb += dz;
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        accg[v].x = fmaf(dz, x[v].x, accg[v].x);
        accg[v].y = fmaf(dz, x[v].y, accg[v].y);
        accg[v].z = fmaf(dz, x[v].z, accg[v].z);
        accg[v].w = fmaf(dz, x[v].w, accg[v].w);
        const float4 gv = make_float4(dz * wg[v].x, dz * wg[v].y, dz * wg[v].z, dz * wg[v].w);
        gu_acc[v].x = fmaf(gv.x, gi[rr][v].x, gu_acc[v].x);
        gu_acc[v].y = fmaf(gv.y, gi[rr][v].y, gu_acc[v].y);
        gu_acc[v].z = fmaf(gv.z, gi[rr][v].z, gu_acc[v].z);
        gu_acc[v].w = fmaf(gv.w, gi[rr][v].w, gu_acc[v].w);
        acch[v].x = fmaf(dz, h[rr][v].x, acch[v].x);
        acch[v].y = fmaf(dz, h[rr][v].y, acch[v].y);
        acch[v].z = fmaf(dz, h[rr][v].z, acch[v].z);
        acch[v].w = fmaf(dz, h[rr][v].w, acch[v].w);
        if (live) {
          *reinterpret_cast<float4*>(p.stage_i + (size_t)gr * si + d_i + 32 * v + 4 * sub) =
              make_float4(gv.x * gu[v].x, gv.y * gu[v].y, gv.z * gu[v].z, gv.w * gu[v].w);
          *reinterpret_cast<float4*>(p.dz_last + (size_t)lr * Ln + 32 * v + 4 * sub) =
              make_float4(h[rr][v].x > 0.f ? dz * wh[v].x : 0.f, h[rr][v].y > 0.f ? dz * wh[v].y : 0.f,
                          h[rr][v].z > 0.f ? dz * wh[v].z : 0.f, h[rr][v].w > 0.f ? dz * wh[v].w : 0.f);
        }
      }
    }
    if (live) {
      const int64_t grp = (p.row0 + g * KR) / KR;
#pragma unroll
      for (int v = 0; v < NV; ++v)
        *reinterpret_cast<float4*>(p.stage_u + (size_t)grp * su + d_u + 32 * v + 4 * sub) = gu_acc[v];
      if (any_bad && sub == 0) atomicOr(p.flags, 1);
    }
    item_c = item_n;
    y_c = y_n;
    u_c = u_n;
  }

  // per-quad sums -> shared -> this CTA's partial row, quads and warps added in index order
  float* my = red[warp * 4 + quad];
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    *reinterpret_cast<float4*>(my + 32 * v + 4 * sub) = accg[v];
    *reinterpret_cast<float4*>(my + f + 32 * v + 4 * sub) = acch[v];
  }
  if (sub == 0) {
    my[ncols] = accb;  // every lane of a quad holds the same accb / accl
    my[ncols + 1] = accl;
  }
  __syncthreads();
  float* dst = p.head_partial + (size_t)blockIdx.x * (ncols + 2);
  for (int j = threadIdx.x; j < ncols + 2; j += blockDim.x) {
    float t = 0.f;
    for (int w = 0; w < kWarps * 4; ++w) t += red[w][j];
    dst[j] += t;
  }
}

// Ranking evaluation, fused: GMF product + output unit + sigmoid of the `group` candidates of one user AND the
// position of the positive (the LAST candidate, data_pipeline.py:113,148) under the RankLayer order
// (model.py:344-352: descending probability, lower index first among ties), in one kernel -- the scores never
// leave the SM unless the caller asks for them.  One CTA per group: its 8 warps score interleaved slices of
// the candidates (8 rows per warp in flight), the probabilities meet in shared memory and the whole CTA counts
//   pos = #{j : p_j > p_pos  or  (p_j == p_pos and j < group - 1)}.
template <int MAXQ>
__global__ void __launch_bounds__(kHeadThreads, 2) head_rank_kernel(const HeadParams p, int group,
                                                                    int32_t* __restrict__ pos,
                                                                    float* __restrict__ probs) {
  __shared__ float sc[kHeadThreads];  // probabilities of the group's candidates (group <= 256)
  const MrModel& m = p.m;
  const int f = m.mf_dim, Ln = m.L[m.n_layers - 1], ncols = f + Ln;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int kWarps = kHeadThreads / 32;
  constexpr int kRows = 8;  // rows scored per warp iteration: their loads are all in flight together
  float wv[MAXQ];
#pragma unroll
  for (int q = 0; q < MAXQ; ++q) wv[q] = (lane + 32 * q < ncols) ? __ldg(m.w_out + lane + 32 * q) : 0.f;
  const float b_out = __ldg(m.b_out);
  const int64_t ngroups = p.rows / group;
  const int per_warp = (group + kWarps - 1) / kWarps;  // <= 32: candidate j = warp + kWarps * i, i < per_warp
  for (int64_t g = blockIdx.x; g < ngroups; g += gridDim.x) {
    const int64_t gg = p.row0 / group + g;  // global group index: users holds one id per group
    const int64_t lr_first = g * group;
    int u = __ldg(p.users + gg);
    // this warp's item ids, lane-distributed: lane i holds the id of candidate warp + kWarps * i
    const int jmine = warp + kWarps * lane;
    const int idreg = (lane < per_warp && jmine < group) ? __ldg(p.items + p.row0 + lr_first + jmine) : 0;
    const bool bad_u = (unsigned)u >= (unsigned)m.num_users;
    if (bad_u) u = 0;
    float gu[MAXQ];
#pragma unroll
    for (int q = 0; q < MAXQ; ++q) gu[q] = (lane + 32 * q < f) ? __ldg(m.user_gmf + (size_t)u * f + lane + 32 * q) : 0.f;
    for (int i0 = 0; i0 < per_warp; i0 += kRows) {
      int it[kRows];
      bool live[kRows];
      float hv[kRows][MAXQ];
#pragma unroll
      for (int rr = 0; rr < kRows; ++rr) {
        const int j = warp + kWarps * (i0 + rr);
        live[rr] = (i0 + rr) < per_warp && j < group;
        it[rr] = __shfl_sync(0xffffffffu, idreg, (i0 + rr) & 31);
      }
      // loads first, unconditional (dead rows re-read the positive's row) and with no arithmetic on the loaded
      // values: a branch or a multiply per row here makes the in-order issue wait for each row's data before
      // the next row's loads go out (ncu: the first version spent 8 serial memory latencies per iteration)
#pragma unroll
      for (int rr = 0; rr < kRows; ++rr) {
        const int j = live[rr] ? warp + kWarps * (i0 + rr) : group - 1;
        const int iv = ((unsigned)it[rr] >= (unsigned)m.num_items) ? 0 : it[rr];
        const float* hrow = p.h_last + (size_t)(lr_first + j) * Ln;
        const float* grow = m.item_gmf + (size_t)iv * f;
#pragma unroll
        for (int q = 0; q < MAXQ; ++q) {
          const int c = lane + 32 * q;
          const float* src = c < f ? grow + c : hrow + (c < ncols ? c - f : 0);
          hv[rr][q] = (c < ncols) ? __ldg(src) : 0.f;
        }
      }
#pragma unroll
      for (int rr = 0; rr < kRows; ++rr) {
        if (!live[rr]) continue;  // warp-uniform
        const int j = warp + kWarps * (i0 + rr);
        float sacc = 0.f;
#pragma unroll
        for (int q = 0; q < MAXQ; ++q) {
          const float x = (lane + 32 * q < f) ? gu[q] * hv[rr][q] : hv[rr][q];
          sacc = fmaf(wv[q], x, sacc);
        }
        sacc = warp_sum(sacc);
        const bool bad = bad_u || (unsigned)it[rr] >= (unsigned)m.num_items;
        const float pr = bad ? nanf("") : sigmoidf_stable(sacc + b_out);
        if (lane == 0) {
          sc[j] = pr;
          if (probs != nullptr) probs[p.row0 + lr_first + j] = pr;
          if (bad) atomicOr(p.flags, 1);
        }
      }
    }
    __syncthreads();
    const float key_pos = rank_key(sc[group - 1]);
    const int j = threadIdx.x;
    const int above = (j < group - 1) && (rank_key(sc[j]) >= key_pos);  // a negative that ties ranks first (lower index)
    const int cnt = __syncthreads_count(above);
    if (threadIdx.x == 0) pos[gg] = cnt;
  }
}

// Probability of one row of the partial-logit form, eight lanes per row: lane `sub` of the row's eight holds columns
// 32 v + 4 sub .. + 3 of wu = w_out[:f] * (user GMF row) and of the item GMF row; z = the last hidden layer already
// dotted with its output weights.  All 32 lanes must call it (the shuffles).  head_rank_warp_kernel and
// catalogue_head_kernel both score through it, so a (user, item) pair gets bit-identical probabilities from the
// sampled ranking eval and from the catalogue sweep.
template <int NV>
__device__ __forceinline__ float gmf_head_prob(const float4 (&wu)[NV], const float4 (&gi)[NV], float z, float b_out,
                                               bool bad) {
  float s = 0.f;
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    s = fmaf(wu[v].x, gi[v].x, s);
    s = fmaf(wu[v].y, gi[v].y, s);
    s = fmaf(wu[v].z, gi[v].z, s);
    s = fmaf(wu[v].w, gi[v].w, s);
  }
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  s += __shfl_xor_sync(0xffffffffu, s, 4);
  return bad ? nanf("") : sigmoidf_stable(s + z + b_out);
}

// Score + position with ONE WARP PER GROUP, for the partial-logit form (p.h_last = one float per row: the last
// hidden layer already dotted with its output-unit weights by tc_dense EPI_HEAD_DOT).  What is left per candidate
// is the GMF term, a dot product of f = 32 * NV floats: eight lanes take one row (NV 128-bit loads each, 128
// contiguous bytes per eight lanes), so a load instruction covers four rows and the reduction is three shuffles;
// the group's scores meet in the warp's slice of shared memory and the position is a ballot-free count.  No CTA
// barrier: the CTA-per-group kernels above spend ~6 us per group on two serial half-group round trips with 16 warps
// per SM (ncu: issue-active 60 %, 3 TB/s); here every warp is independent and KS steps (4 * KS rows) are in flight.
template <int NV>
__global__ void __launch_bounds__(kHeadThreads) head_rank_warp_kernel(const HeadParams p, int group,
                                                                      int32_t* __restrict__ pos,
                                                                      float* __restrict__ probs) {
  constexpr int f = 32 * NV, KS = 5;
  constexpr int kWarps = kHeadThreads / 32;
  __shared__ float sc[kWarps][256];
  const MrModel& m = p.m;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int sub = lane & 7, quad = lane >> 3;
  float4 wg[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) wg[v] = ldg4(m.w_out + 32 * v + 4 * sub);
  const float b_out = __ldg(m.b_out);
  const int64_t ngroups = p.rows / group;
  const int64_t nwarps = (int64_t)gridDim.x * kWarps;
  const int nsteps = (group + 3) >> 2;
  float* my_sc = sc[warp];
  for (int64_t g = (int64_t)blockIdx.x * kWarps + warp; g < ngroups; g += nwarps) {
    const int64_t gg = p.row0 / group + g;
    int u = __ldg(p.users + gg);
    const bool bad_u = (unsigned)u >= (unsigned)m.num_users;
    if (bad_u) u = 0;
    float4 gu[NV];  // w_out[:f] * user GMF row, this lane's columns
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const float4 x = ldg4(m.user_gmf + (size_t)u * f + 32 * v + 4 * sub);
      gu[v] = make_float4(x.x * wg[v].x, x.y * wg[v].y, x.z * wg[v].z, x.w * wg[v].w);
    }
    const int64_t lr0 = g * group;  // launch-local first row of the group
    for (int s0 = 0; s0 < nsteps; s0 += KS) {
      int it[KS];
      float4 gi[KS][NV];
      float z[KS];
#pragma unroll
      for (int k = 0; k < KS; ++k) {
        const int row = (s0 + k) * 4 + quad;
        const int rr = row < group ? row : group - 1;  // dead slots re-read the positive's row
        it[k] = __ldg(p.items + p.row0 + lr0 + rr);
        z[k] = __ldg(p.h_last + lr0 + rr);
      }
#pragma unroll
      for (int k = 0; k < KS; ++k) {
        const int iv = (unsigned)it[k] >= (unsigned)m.num_items ? 0 : it[k];
#pragma unroll
        for (int v = 0; v < NV; ++v) gi[k][v] = ldg4(m.item_gmf + (size_t)iv * f + 32 * v + 4 * sub);
      }
#pragma unroll
      for (int k = 0; k < KS; ++k) {
        const int row = (s0 + k) * 4 + quad;
        const bool bad = bad_u || (unsigned)it[k] >= (unsigned)m.num_items;
        const float pr = gmf_head_prob<NV>(gu, gi[k], z[k], b_out, bad);
        if (sub == 0 && row < group) {
          my_sc[row] = pr;
          if (probs != nullptr) probs[p.row0 + lr0 + row] = pr;
          if (bad) atomicOr(p.flags, 1);
        }
      }
    }
    __syncwarp();
    const float key_pos = rank_key(my_sc[group - 1]);
    int cnt = 0;
    for (int j = lane; j < group - 1; j += 32) cnt += rank_key(my_sc[j]) >= key_pos ? 1 : 0;  // ties rank first
    cnt = warp_sum_int(cnt);
    if (lane == 0) pos[gg] = cnt;
    __syncwarp();
  }
}

// Catalogue sweep: the partial-logit form for `rows` rows where row r pairs users[r / group] with item r % group (one
// user against the whole catalogue per `group` rows).  Row-parallel -- a group here is tens of thousands of rows, far
// beyond the warp-per-group kernel's shared-memory slice -- with the per-row arithmetic of head_rank_warp_kernel
// (gmf_head_prob).  Four rows per warp step, KS steps in flight.
// HEAD_RAGGED (candidate lists): row r is global row row0 + r, pairing users[seg[row0 + r]] with items[row0 + r]; h_dot
// is launch-local; an out-of-range user, item or list index gives NaN.
// HEAD_TILED (an item list tiled over the users: audiences): row r pairs users[r / group] with items[r]; an
// out-of-range user or item gives NaN.
enum { HEAD_CATALOGUE = 0, HEAD_RAGGED = 1, HEAD_TILED = 2 };
template <int NV, int MODE>
__global__ void __launch_bounds__(kHeadThreads) catalogue_head_kernel(const MrModel m, const float* __restrict__ h_dot,
                                                                      const int32_t* __restrict__ users, int64_t rows,
                                                                      int group, float* __restrict__ probs,
                                                                      const int32_t* __restrict__ seg,
                                                                      const int32_t* __restrict__ items, int64_t row0,
                                                                      int64_t num_lists) {
  constexpr int f = 32 * NV, KS = NV >= 4 ? 1 : 2;  // (KS = 4 spills at NV = 1 and needs 170 registers at NV = 4)
  const int lane = threadIdx.x & 31;
  const int sub = lane & 7, quad = lane >> 3;
  float4 wg[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) wg[v] = ldg4(m.w_out + 32 * v + 4 * sub);
  const float b_out = __ldg(m.b_out);
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r0 = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * (4 * KS); r0 < rows;
       r0 += nwarps * (4 * KS)) {
    float4 wu[KS][NV], gi[KS][NV];
    float z[KS];
    bool bad[KS];
#pragma unroll
    for (int k = 0; k < KS; ++k) {
      int64_t row = r0 + 4 * k + quad;
      if (row >= rows) row = rows - 1;  // dead slots re-read the last row
      int u, it;
      if (MODE == HEAD_RAGGED) {
        const int sg = __ldg(seg + row0 + row);
        u = (unsigned)sg < (uint64_t)num_lists ? __ldg(users + sg) : -1;
        it = __ldg(items + row0 + row);
        bad[k] = (unsigned)u >= (unsigned)m.num_users || (unsigned)it >= (unsigned)m.num_items;
        if (bad[k]) u = it = 0;
      } else if (MODE == HEAD_TILED) {
        u = __ldg(users + row / group);
        it = __ldg(items + row);
        bad[k] = (unsigned)u >= (unsigned)m.num_users || (unsigned)it >= (unsigned)m.num_items;
        if (bad[k]) u = it = 0;
      } else {
        const int64_t slot = row / group;
        it = (int)(row - slot * group);
        u = __ldg(users + slot);
        bad[k] = (unsigned)u >= (unsigned)m.num_users;
        if (bad[k]) u = 0;
      }
      z[k] = __ldg(h_dot + row);
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const float4 x = ldg4(m.user_gmf + (size_t)u * f + 32 * v + 4 * sub);
        wu[k][v] = make_float4(x.x * wg[v].x, x.y * wg[v].y, x.z * wg[v].z, x.w * wg[v].w);
        gi[k][v] = ldg4(m.item_gmf + (size_t)it * f + 32 * v + 4 * sub);
      }
    }
#pragma unroll
    for (int k = 0; k < KS; ++k) {
      const int64_t row = r0 + 4 * k + quad;
      const float pr = gmf_head_prob<NV>(wu[k], gi[k], z[k], b_out, bad[k]);
      if (sub == 0 && row < rows) probs[(MODE == HEAD_RAGGED ? row0 : 0) + row] = pr;
    }
  }
}

// d w_out / d b_out / loss: sum of the CTA partial rows, one warp per column, lanes stride over the rows
// and fold with the fixed shuffle tree (deterministic).  Runs once per step.
__global__ void __launch_bounds__(256) head_reduce_kernel(const float* __restrict__ head_partial, int grid_ctas,
                                                          int ncols, float* __restrict__ d_wout,
                                                          float* __restrict__ d_bout, float* __restrict__ loss_sum) {
  const int lane = threadIdx.x & 31;
  const int j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (j >= ncols + 2) return;
  float s = 0.f;
  for (int c = lane; c < grid_ctas; c += 32) s += head_partial[(size_t)c * (ncols + 2) + j];
  s = warp_sum(s);
  if (lane == 0) {
    if (j < ncols) d_wout[j] += s;
    else if (j == ncols) *d_bout += s;
    else *loss_sum += s;
  }
}

int head_grid() { return sm_count() * 8; }

// widths the pipelined specialisation is instantiated for: (mf_dim, last layer)
static bool head_special_widths(const MrModel& m) {
  const int f = m.mf_dim, Ln = m.L[m.n_layers - 1];
  return (f == 64 && Ln == 64) || (f == 128 && Ln == 64);
}

bool head_supports_group(const MrModel& m, int group) {
  return group >= 2 && group <= 8 && (m.mf_dim + m.L[m.n_layers - 1] <= 128 || head_special_widths(m));
}

size_t head_partial_floats(const MrModel& m) { return (size_t)head_grid() * (m.mf_dim + m.L[m.n_layers - 1] + 2); }

int launch_head(const HeadArgs& a, cudaStream_t st) {
  const MrModel& m = *a.model;
  const int ncols = m.mf_dim + m.L[m.n_layers - 1];
  if (ncols > kHeadMaxQ * 32) {
    set_error("head kernel: mf_dim + last layer width = %d exceeds %d", ncols, kHeadMaxQ * 32);
    return MR_ERR_INVALID;
  }
  if (a.rows == 0) return MR_OK;
  HeadParams p{};
  p.m = m;
  p.h_last = a.h_last;
  p.users = a.users;
  p.items = a.items;
  p.labels = a.labels;
  p.rows = a.rows;
  p.row0 = a.row0;
  p.user_div = a.user_div < 1 ? 1 : a.user_div;
  p.inv_batch = a.inv_batch;
  p.logits = a.logits;
  p.probs = a.probs;
  p.dz_last = a.dz_last;
  p.stage_u = a.stage_u;
  p.stage_i = a.stage_i;
  p.head_partial = a.head_partial;
  p.flags = a.flags;
  p.group = a.group;
  const int grid = head_grid();
  if (a.group > 0) {
    if (!head_supports_group(m, a.group) || a.rows % a.group || a.row0 % a.group || p.user_div != 1) {
      set_error("head kernel: grouped mode needs group <= 8, supported head widths and whole groups");
      return MR_ERR_INVALID;
    }
    const bool wide = ncols > 128;  // only the specialisation covers these
    const bool special = a.labels != nullptr && head_special_widths(m);
    const uintptr_t al = reinterpret_cast<uintptr_t>(m.user_gmf) | reinterpret_cast<uintptr_t>(m.item_gmf) |
                         reinterpret_cast<uintptr_t>(m.w_out) | reinterpret_cast<uintptr_t>(a.h_last) |
                         reinterpret_cast<uintptr_t>(a.dz_last) | reinterpret_cast<uintptr_t>(a.stage_u) |
                         reinterpret_cast<uintptr_t>(a.stage_i);
    if (special && m.mf_dim == 64 && a.group <= 5 && (al & 15) == 0 && (m.L[0] / 2) % 4 == 0) {  // eight lanes per row
      const int64_t want = (a.rows / a.group + 15) / 16;  // 16 groups per CTA iteration
      const unsigned qgrid = (unsigned)(want < grid ? want : grid);
      switch (a.group) {
        case 2: head_quad_kernel<2><<<qgrid, kQuadThreads, 0, st>>>(p); break;
        case 3: head_quad_kernel<3><<<qgrid, kQuadThreads, 0, st>>>(p); break;
        case 4: head_quad_kernel<4><<<qgrid, kQuadThreads, 0, st>>>(p); break;
        default: head_quad_kernel<5><<<qgrid, kQuadThreads, 0, st>>>(p); break;
      }
      MR_LAUNCH_CHECK("head_quad_kernel");
      return MR_OK;
    }
    if (special) {  // the pipelined specialisation: BASELINE configs[2] (f = 64) and configs[4] (f = 128), last layer 64
#define MR_HEAD_GROUP(FQ_)                                                                                   \
  switch (a.group) {                                                                                       \
    case 2: head_group_kernel<FQ_, 2, 2><<<grid, kHeadThreads, 0, st>>>(p); break;                          \
    case 3: head_group_kernel<FQ_, 2, 3><<<grid, kHeadThreads, 0, st>>>(p); break;                          \
    case 4: head_group_kernel<FQ_, 2, 4><<<grid, kHeadThreads, 0, st>>>(p); break;                          \
    case 5: head_group_kernel<FQ_, 2, 5><<<grid, kHeadThreads, 0, st>>>(p); break;                          \
    case 6: head_group_kernel<FQ_, 2, 6><<<grid, kHeadThreads, 0, st>>>(p); break;                          \
    case 7: head_group_kernel<FQ_, 2, 7><<<grid, kHeadThreads, 0, st>>>(p); break;                          \
    default: head_group_kernel<FQ_, 2, 8><<<grid, kHeadThreads, 0, st>>>(p); break;                         \
  }
      if (m.mf_dim == 64) { MR_HEAD_GROUP(2) } else { MR_HEAD_GROUP(4) }
#undef MR_HEAD_GROUP
      MR_LAUNCH_CHECK("head_group_kernel");
      return MR_OK;
    }
    if (wide) {
      set_error("head kernel: grouped training with mf_dim + last width = %d needs labels", ncols);
      return MR_ERR_INVALID;
    }
    switch (a.group) {
      case 2: head_kernel<4, 2, true><<<grid, kHeadThreads, 0, st>>>(p); break;
      case 3: head_kernel<4, 3, true><<<grid, kHeadThreads, 0, st>>>(p); break;
      case 4: head_kernel<4, 4, true><<<grid, kHeadThreads, 0, st>>>(p); break;
      case 5: head_kernel<4, 5, true><<<grid, kHeadThreads, 0, st>>>(p); break;
      case 6: head_kernel<4, 6, true><<<grid, kHeadThreads, 0, st>>>(p); break;
      case 7: head_kernel<4, 7, true><<<grid, kHeadThreads, 0, st>>>(p); break;
      default: head_kernel<4, 8, true><<<grid, kHeadThreads, 0, st>>>(p); break;
    }
  } else if (ncols <= 128) head_kernel<4, 4, false><<<grid, kHeadThreads, 0, st>>>(p);
  else if (ncols <= 256) head_kernel<8, 2, false><<<grid, kHeadThreads, 0, st>>>(p);
  else head_kernel<16, 2, false><<<grid, kHeadThreads, 0, st>>>(p);
  MR_LAUNCH_CHECK("head_kernel");
  return MR_OK;
}

bool head_rank_supported(const MrModel& m) { return m.mf_dim + m.L[m.n_layers - 1] <= 128; }

bool catalogue_head_supported(const MrModel& m) {
  const bool widths = m.mf_dim == 32 || m.mf_dim == 64 || m.mf_dim == 128;  // gmf_head_prob<1 | 2 | 4>
  return widths && (reinterpret_cast<uintptr_t>(m.user_gmf) | reinterpret_cast<uintptr_t>(m.item_gmf) |
                    reinterpret_cast<uintptr_t>(m.w_out)) % 16 == 0;
}

bool head_rank_takes_dot(const MrModel& m, int group) {
  return catalogue_head_supported(m) && group >= 2 && group <= 256;
}

int launch_catalogue_head(const MrModel& m, const float* h_dot, const int32_t* users, int64_t rows, int group,
                          float* probs, cudaStream_t st, const int32_t* seg, const int32_t* items, int64_t row0,
                          int64_t num_lists) {
  if (!catalogue_head_supported(m) || group < 1) {
    set_error("catalogue head: needs mf_dim 32, 64 or 128 and 16-byte aligned GMF tables / output weights");
    return MR_ERR_INVALID;
  }
  if (rows == 0) return MR_OK;
  const int64_t want = (rows + 4 * (kHeadThreads / 32) - 1) / (4 * (kHeadThreads / 32));
  const int64_t cap = (int64_t)sm_count() * 8;
  const unsigned grid = (unsigned)(want < cap ? want : cap);
#define MR_CATALOGUE_HEAD(MODE_)                                                                                  \
  if (m.mf_dim == 32)                                                                                            \
    catalogue_head_kernel<1, MODE_><<<grid, kHeadThreads, 0, st>>>(m, h_dot, users, rows, group, probs, seg, items, \
                                                                   row0, num_lists);                             \
  else if (m.mf_dim == 64)                                                                                       \
    catalogue_head_kernel<2, MODE_><<<grid, kHeadThreads, 0, st>>>(m, h_dot, users, rows, group, probs, seg, items, \
                                                                   row0, num_lists);                             \
  else                                                                                                           \
    catalogue_head_kernel<4, MODE_><<<grid, kHeadThreads, 0, st>>>(m, h_dot, users, rows, group, probs, seg, items, \
                                                                   row0, num_lists);
  if (seg != nullptr) { MR_CATALOGUE_HEAD(HEAD_RAGGED) }
  else if (items != nullptr) { MR_CATALOGUE_HEAD(HEAD_TILED) }
  else { MR_CATALOGUE_HEAD(HEAD_CATALOGUE) }
#undef MR_CATALOGUE_HEAD
  MR_LAUNCH_CHECK("catalogue_head_kernel");
  return MR_OK;
}

// Fused score + rank of whole groups (forward only): a.users holds ONE id per group (global group index),
// a.rows / a.row0 are rows (multiples of `group`); pos is indexed by the global group, probs by the global row.
int launch_head_rank(const HeadArgs& a, int group, int32_t* pos, float* probs, cudaStream_t st) {
  const MrModel& m = *a.model;
  if (!(a.h_is_dot ? head_rank_takes_dot(m, group) : head_rank_supported(m)) || group < 2 || group > 256 ||
      a.rows % group || a.row0 % group) {
    set_error("head_rank kernel: needs mf_dim + last width <= 128 (or the partial-logit form with mf_dim 32, 64 or "
              "128) and whole groups of at most 256 rows");
    return MR_ERR_INVALID;
  }
  if (a.rows == 0) return MR_OK;
  HeadParams p{};
  p.m = m;
  p.h_last = a.h_last;
  p.users = a.users;
  p.items = a.items;
  p.rows = a.rows;
  p.row0 = a.row0;
  p.user_div = 1;
  p.flags = a.flags;
  const int64_t ngroups = a.rows / group;
  const int64_t cap = (int64_t)sm_count() * 2;  // persistent: two resident CTAs per SM, groups taken round-robin
  const unsigned grid = (unsigned)(ngroups < cap ? ngroups : cap);
  if (a.h_is_dot) {
    // one warp per group: enough CTAs for full occupancy, groups taken round-robin by the warps
    const int64_t wcap = (int64_t)sm_count() * 8;
    const int64_t want = (ngroups + kHeadThreads / 32 - 1) / (kHeadThreads / 32);
    const unsigned wgrid = (unsigned)(want < wcap ? want : wcap);
    if (m.mf_dim == 32)
      head_rank_warp_kernel<1><<<wgrid, kHeadThreads, 0, st>>>(p, group, pos, probs);
    else if (m.mf_dim == 64)
      head_rank_warp_kernel<2><<<wgrid, kHeadThreads, 0, st>>>(p, group, pos, probs);
    else
      head_rank_warp_kernel<4><<<wgrid, kHeadThreads, 0, st>>>(p, group, pos, probs);
  } else {
    head_rank_kernel<4><<<grid, kHeadThreads, 0, st>>>(p, group, pos, probs);
  }
  MR_LAUNCH_CHECK("head_rank_kernel");
  return MR_OK;
}

int launch_head_reduce(const MrModel& m, const float* head_partial, float* d_wout_row0, float* d_bout_row0,
                       float* loss_sum, cudaStream_t st) {
  const int ncols = m.mf_dim + m.L[m.n_layers - 1];
  const int warps = ncols + 2;
  head_reduce_kernel<<<(warps + 7) / 8, 256, 0, st>>>(head_partial, head_grid(), ncols, d_wout_row0, d_bout_row0, loss_sum);
  MR_LAUNCH_CHECK("head_reduce_kernel");
  return MR_OK;
}

}  // namespace mr
