// Fold-in of new users (include/movierec_b200.h: mr_fold_in_users): the item tables and the dense block are frozen and
// only each user's MLP and GMF rows are optimised against the user's history and sampled negatives.
//
// One persistent CTA per user at a time, all steps inside the kernel; users are taken longest history first.  The
// user's rows, their Adam moments, the user half of the first layer (Pu = e_u . W1u + b1) and the running gradient
// sums live in shared memory.  A step walks the user's rows (n positives x (negs + 1)) in chunks of at most kChunkRows:
// one thread per positive draws the chunk's negatives (negative_draw.cuh, the batch sampler's rule), then tiles of TM
// rows go through relu(Pi[item] + Pu), the later layers (tile_gemm, weights read through L1), the head with the GMF
// product, dz and the backward to the masked dZ1.  Per tile, each column of sum dZ1 and of the GMF row gradient is
// summed over the tile's rows in row order and added to the running sum in tile order: a fixed order, no atomics.  At
// the end of the step dE_u = (sum dZ1) . W1u^T + 2 l2[0] e_u, and the rows are updated in shared memory.
#include "launchers.h"
#include "negative_draw.cuh"
#include "neumf_tile.cuh"

namespace mr {

constexpr int kFoldThreads = 256;
constexpr int kChunkRows = 1024;  // rows whose negatives are drawn at once (>= negs + 1 = MR_MAX_NEGS + 1)

struct FoldParams {
  MrModel m;
  const float* Wt[MR_MAX_LAYERS];  // Wt[l] = W[l]^T, (L[l], L[l-1])
  const float* Pi;                 // (num_items, L1): E_item . W1[item rows]; NULL without a hidden layer
  const int64_t* rowptr;
  const int32_t* items;
  const int32_t* init_users;
  const int32_t* order;            // users, longest history first
  int64_t U;
  int32_t steps, negs, optimizer;
  float lr, beta_1, beta_2, epsilon;
  uint64_t seed;
  float* out_mlp;
  float* out_gmf;
  float* out_loss;
  int32_t ld[MR_MAX_LAYERS];
  int32_t act_off[MR_MAX_LAYERS];
  int32_t gi_off, ldf, ga_off, gb_off, ldg;
  int32_t e_off, g_off, me_off, ve_off, mg_off, vg_off, pu_off, s_off, gacc_off;
  int32_t dz_off, loss_off, ids_off, picked_off;
};

template <int TM>
__global__ void __launch_bounds__(kFoldThreads) fold_in_kernel(const FoldParams p) {
  extern __shared__ __align__(16) float smem[];
  const MrModel& m = p.m;
  const int n = m.n_layers, f = m.mf_dim;
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u;
  const int L1 = n > 1 ? m.L[1] : 0;
  const int Ln = m.L[n - 1];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const int group = p.negs + 1;
  const int gpc = kChunkRows / group;  // positives per chunk
  const float c2 = 2.f * m.l2[0];
  const bool adam = p.optimizer == MR_OPT_ADAM;

  float* s_e = smem + p.e_off;
  float* s_g = smem + p.g_off;
  float* s_me = smem + p.me_off;
  float* s_ve = smem + p.ve_off;
  float* s_mg = smem + p.mg_off;
  float* s_vg = smem + p.vg_off;
  float* s_pu = smem + p.pu_off;
  float* s_sum = smem + p.s_off;     // sum of dZ1 over the step's rows (L1), or of dz (one float) without hidden layer
  float* s_gacc = smem + p.gacc_off; // GMF row gradient (f)
  float* gi = smem + p.gi_off;
  float* s_dz = smem + p.dz_off;
  float* s_loss = smem + p.loss_off;  // TM row losses, then [TM] = the step's running loss sum
  int* s_ids = reinterpret_cast<int*>(smem + p.ids_off);
  int* s_picked = reinterpret_cast<int*>(smem + p.picked_off);
  float* actL = smem + p.act_off[n - 1];

  for (int64_t slot = blockIdx.x; slot < p.U; slot += gridDim.x) {
    const int u = __ldg(p.order + slot);
    const int64_t lo = __ldg(p.rowptr + u);
    const int len = (int)(__ldg(p.rowptr + u + 1) - lo);
    const int32_t* hist = p.items + lo;
    const int init = p.init_users != nullptr ? __ldg(p.init_users + u) : -1;
    for (int k = tid; k < d_u; k += blockDim.x) {
      s_e[k] = init >= 0 ? m.user_mlp[(size_t)init * d_u + k] : 0.f;
      s_me[k] = 0.f;
      s_ve[k] = 0.f;
    }
    for (int j = tid; j < f; j += blockDim.x) {
      s_g[j] = init >= 0 ? m.user_gmf[(size_t)init * f + j] : 0.f;
      s_mg[j] = 0.f;
      s_vg[j] = 0.f;
    }
    const int64_t R = (int64_t)len * group;
    const float inv_r = R > 0 ? 1.f / (float)R : 0.f;
    float last_loss = nanf("");
    __syncthreads();

    for (int t = 0; t < p.steps; ++t) {
      // ---- once per step: Pu = e_u . W1u + b1, the sums cleared --------------------------------------------------
      for (int c = tid; c < L1; c += blockDim.x) {
        float s = 0.f;
        for (int k = 0; k < d_u; ++k) s = fmaf(s_e[k], __ldg(m.W[1] + (size_t)k * L1 + c), s);
        s_pu[c] = s + __ldg(m.b[1] + c);
        s_sum[c] = 0.f;
      }
      if (n == 1 && tid == 0) s_sum[0] = 0.f;
      for (int j = tid; j < f; j += blockDim.x) s_gacc[j] = 0.f;
      if (tid == 0) s_loss[TM] = 0.f;
      __syncthreads();

      for (int g0 = 0; g0 < len; g0 += gpc) {
        const int ng = min(gpc, len - g0);
        const int rows = ng * group;
        // ---- the chunk's rows: group j = the negatives of positive g0 + j, then the positive ----------------------
        for (int j = tid; j < ng; j += blockDim.x) {
          int* out = s_ids + j * group;
          draw_negatives(hist, len, m.num_items, p.negs, (uint64_t)(g0 + j), p.seed, (uint64_t)t,
                         s_picked + j * p.negs, [&](int q, int item) { out[q] = item; });
          out[p.negs] = __ldg(hist + g0 + j);
        }
        __syncthreads();

        for (int row0 = 0; row0 < rows; row0 += TM) {
          const int valid = min(TM, rows - row0);
          // ---- first layer (or nothing without a hidden layer) and the GMF item rows ----------------------------
          if (n > 1) {
            float* h1 = smem + p.act_off[1];
            for (int e = tid; e < TM * L1; e += blockDim.x) {
              const int r = e / L1, c = e - r * L1;
              float v = 0.f;
              if (r < valid) v = fmaxf(__ldg(p.Pi + (size_t)s_ids[row0 + r] * L1 + c) + s_pu[c], 0.f);
              h1[r * p.ld[1] + c] = v;
            }
          }
          for (int e = tid; e < TM * f; e += blockDim.x) {
            const int r = e / f, c = e - r * f;
            gi[r * p.ldf + c] = r < valid ? __ldg(m.item_gmf + (size_t)s_ids[row0 + r] * f + c) : 0.f;
          }
          __syncthreads();
          for (int l = 2; l < n; ++l) {
            TileOut o{};
            o.smem = smem + p.act_off[l];
            o.ld = p.ld[l];
            tile_gemm<TM, true>(smem + p.act_off[l - 1], p.ld[l - 1], m.L[l - 1], m.W[l], m.L[l], m.b[l], o);
            __syncthreads();
          }

          // ---- head: z = b + w[:f].(g_u*g_i) + w[f:].x ; sigmoid ; BCE ; dz --------------------------------------
          const int ldL = p.ld[n - 1];
          for (int r = warp; r < TM; r += nwarps) {
            float s = 0.f;
            if (r < valid) {
              for (int j = lane; j < f; j += 32) s = fmaf(__ldg(m.w_out + j), s_g[j] * gi[r * p.ldf + j], s);
              if (n > 1) {
                for (int c = lane; c < Ln; c += 32) s = fmaf(__ldg(m.w_out + f + c), actL[r * ldL + c], s);
              } else {
                const float* ei = m.item_mlp + (size_t)s_ids[row0 + r] * d_i;
                for (int c = lane; c < d_u; c += 32) s = fmaf(__ldg(m.w_out + f + c), s_e[c], s);
                for (int c = lane; c < d_i; c += 32) s = fmaf(__ldg(m.w_out + f + d_u + c), __ldg(ei + c), s);
              }
            }
            s = warp_sum(s);
            if (lane == 0) {
              float dz = 0.f, lo_r = 0.f;
              if (r < valid) {
                const float z = s + __ldg(m.b_out);
                const float y = ((row0 + r) % group == p.negs) ? 1.f : 0.f;
                lo_r = bce_logits(z, y);
                dz = (sigmoidf_stable(z) - y) * inv_r;
              }
              s_dz[r] = dz;
              s_loss[r] = lo_r;
            }
          }
          __syncthreads();
          if (warp == 0) {
            float s = 0.f;
            for (int r = lane; r < TM; r += 32) s += s_loss[r];
            s = warp_sum(s);
            if (lane == 0) s_loss[TM] += s;
          }

          // ---- backward: GMF row gradient, dZ of the last hidden layer, then down to dZ1 --------------------------
          for (int j = tid; j < f; j += blockDim.x) {
            const float w = __ldg(m.w_out + j);
            float s = 0.f;
            for (int r = 0; r < valid; ++r) s = fmaf(s_dz[r] * w, gi[r * p.ldf + j], s);
            s_gacc[j] += s;
          }
          if (n == 1) {
            if (tid == 0) {
              float s = 0.f;
              for (int r = 0; r < valid; ++r) s += s_dz[r];
              s_sum[0] += s;
            }
          } else {
            float* gcur = smem + p.ga_off;
            float* gnext = smem + p.gb_off;
            for (int e = tid; e < TM * Ln; e += blockDim.x) {
              const int r = e / Ln, c = e - r * Ln;
              const float v = s_dz[r] * __ldg(m.w_out + f + c);
              gcur[r * p.ldg + c] = actL[r * ldL + c] > 0.f ? v : 0.f;
            }
            __syncthreads();
            for (int l = n - 1; l >= 2; --l) {
              TileOut o{};
              o.smem = gnext;
              o.ld = p.ldg;
              o.mask = smem + p.act_off[l - 1];
              o.mask_ld = p.ld[l - 1];
              tile_gemm<TM, false>(gcur, p.ldg, m.L[l], p.Wt[l], m.L[l - 1], nullptr, o);
              __syncthreads();
              float* tmp = gcur;
              gcur = gnext;
              gnext = tmp;
            }
            for (int c = tid; c < L1; c += blockDim.x) {
              float s = 0.f;
              for (int r = 0; r < valid; ++r) s += gcur[r * p.ldg + c];
              s_sum[c] += s;
            }
          }
          __syncthreads();
        }
      }

      // ---- end of step: the row gradients and the update --------------------------------------------------------
      const float lr_t = adam ? (float)((double)p.lr * sqrt(1.0 - pow((double)p.beta_2, (double)(t + 1))) /
                                        (1.0 - pow((double)p.beta_1, (double)(t + 1))))
                              : p.lr;
      for (int k = tid; k < d_u; k += blockDim.x) {
        float d = 0.f;
        if (n > 1) {
          for (int c = 0; c < L1; ++c) d = fmaf(__ldg(m.W[1] + (size_t)k * L1 + c), s_sum[c], d);
        } else {
          d = s_sum[0] * __ldg(m.w_out + f + k);
        }
        const float g = plus_l2(d, s_e[k], c2);
        if (adam) adam_step(s_e[k], g, s_me[k], s_ve[k], lr_t, p.beta_1, p.beta_2, p.epsilon);
        else s_e[k] = sgd_step(s_e[k], g, lr_t);
      }
      for (int j = tid; j < f; j += blockDim.x) {
        const float g = plus_l2(s_gacc[j], s_g[j], c2);
        if (adam) adam_step(s_g[j], g, s_mg[j], s_vg[j], lr_t, p.beta_1, p.beta_2, p.epsilon);
        else s_g[j] = sgd_step(s_g[j], g, lr_t);
      }
      last_loss = R > 0 ? s_loss[TM] * inv_r : nanf("");
      __syncthreads();
    }

    for (int k = tid; k < d_u; k += blockDim.x) p.out_mlp[(size_t)u * d_u + k] = s_e[k];
    for (int j = tid; j < f; j += blockDim.x) p.out_gmf[(size_t)u * f + j] = s_g[j];
    if (tid == 0 && p.out_loss != nullptr) p.out_loss[u] = last_loss;
    __syncthreads();
  }
}

// Pi[i][c] = sum_k E_item[i][k] W1[d_u + k][c] for the towers the tensor-core table GEMM does not take (odd widths,
// small towers): one thread per output, consecutive threads on consecutive columns.
__global__ void fold_in_project_kernel(MrModel m, float* __restrict__ Pi) {
  const int d_u = m.L[0] / 2, d_i = m.L[0] - d_u, L1 = m.L[1];
  const float* W1i = m.W[1] + (size_t)d_u * L1;
  const int64_t total = (int64_t)m.num_items * L1;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / L1;
    const int c = (int)(e - i * L1);
    const float* ei = m.item_mlp + i * d_i;
    float s = 0.f;
    for (int k = 0; k < d_i; ++k) s = fmaf(__ldg(ei + k), __ldg(W1i + (size_t)k * L1 + c), s);
    Pi[e] = s;
  }
}

// Validation of the histories and init rows (flags: bit 0 malformed rowptr or a list not strictly ascending, bit 1
// an item out of range, bit 2 an init user out of range, bit 3 a list covering every item), and the sort key of each
// user: num_items - length, so that the stable ascending sort takes the longest history first.
__global__ void fold_in_check_kernel(const int64_t* __restrict__ rowptr, const int32_t* __restrict__ items, int64_t U,
                                     int64_t nnz, int32_t num_items, const int32_t* __restrict__ init_users,
                                     int32_t num_users, int32_t* __restrict__ keys, int32_t* __restrict__ flags) {
  for (int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; u < U; u += (int64_t)gridDim.x * blockDim.x) {
    int bad = 0;
    const int64_t lo = rowptr[u], hi = rowptr[u + 1];
    if ((u == 0 && lo != 0) || (u == U - 1 && hi != nnz) || lo < 0 || hi < lo || hi > nnz) bad |= 1;
    int64_t len = 0;
    if (!(bad & 1)) {
      len = hi - lo;
      int prev = -1;
      for (int64_t e = lo; e < hi; ++e) {
        const int it = items[e];
        if (it < 0 || it >= num_items) bad |= 2;
        else if (it <= prev) bad |= 1;
        prev = it;
      }
      if (len >= num_items) bad |= 8;
    }
    if (init_users != nullptr) {
      const int iu = init_users[u];
      if (iu < -1 || iu >= num_users) bad |= 4;
    }
    keys[u] = (bad != 0 || len > num_items) ? 0 : (int32_t)(num_items - len);
    if (bad) atomicOr(flags, bad);
  }
}

// ---- host side -----------------------------------------------------------------------------------------------------

static size_t fold_layout(const MrModel& m, int tm, FoldParams* p) {
  const int n = m.n_layers, f = m.mf_dim, d_u = m.L[0] / 2;
  int off = 0;
  auto take = [&](int count) {
    const int o = off;
    off += (count + 3) & ~3;
    return o;
  };
  for (int l = 0; l < n; ++l) {
    p->ld[l] = pad_ld(m.L[l]);
    p->act_off[l] = l >= 1 ? take(tm * p->ld[l]) : 0;
  }
  p->ldf = pad_ld(f > 0 ? f : 1);
  p->gi_off = take(f > 0 ? tm * p->ldf : 0);
  int gmax = 1;
  for (int l = 1; l < n; ++l) gmax = m.L[l] > gmax ? m.L[l] : gmax;
  p->ldg = pad_ld(gmax);
  p->ga_off = take(n > 1 ? tm * p->ldg : 0);
  p->gb_off = take(n > 1 ? tm * p->ldg : 0);
  p->e_off = take(d_u);
  p->me_off = take(d_u);
  p->ve_off = take(d_u);
  p->g_off = take(f);
  p->mg_off = take(f);
  p->vg_off = take(f);
  const int L1 = n > 1 ? m.L[1] : 1;
  p->pu_off = take(L1);
  p->s_off = take(L1);
  p->gacc_off = take(f);
  p->dz_off = take(tm);
  p->loss_off = take(tm + 1);
  p->ids_off = take(kChunkRows);
  p->picked_off = take(kChunkRows);
  return (size_t)off * sizeof(float);
}

// Largest tile whose shared memory lets two CTAs share an SM, else whatever fits (0: none).
static int fold_tile_rows(const MrModel& m) {
  FoldParams tmp;
  const int cands[4] = {32, 16, 8, 4};
  for (int i = 0; i < 4; ++i)
    if (fold_layout(m, cands[i], &tmp) <= 112 * 1024) return cands[i];
  for (int i = 0; i < 4; ++i)
    if (fold_layout(m, cands[i], &tmp) <= 226 * 1024) return cands[i];
  return 0;
}

bool fold_in_supported(const MrModel& m) { return fold_tile_rows(m) > 0; }

template <int TM>
static int launch_fold(const FoldParams& p, size_t smem, cudaStream_t st) {
  auto kern = fold_in_kernel<TM>;
  MR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 0;
  MR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kFoldThreads, smem));
  if (occ < 1) {
    set_error("fold-in kernel does not fit on an SM (TM=%d, smem=%zu)", TM, smem);
    return MR_ERR_INVALID;
  }
  int64_t grid = (int64_t)sm_count() * occ;
  if (grid > p.U) grid = p.U;
  kern<<<(unsigned)grid, kFoldThreads, smem, st>>>(p);
  MR_LAUNCH_CHECK("fold_in_kernel");
  return MR_OK;
}

int launch_fold_in(const FoldInArgs& a, cudaStream_t st) {
  const MrModel& m = *a.model;
  const int tm = fold_tile_rows(m);
  if (tm == 0) {
    set_error("fold-in: layer widths too large for the kernel's shared memory");
    return MR_ERR_INVALID;
  }
  if (a.U == 0) return MR_OK;
  FoldParams p{};
  const size_t smem = fold_layout(m, tm, &p);
  p.m = m;
  for (int l = 1; l < m.n_layers; ++l) p.Wt[l] = a.wt + (m.W[l] - m.dense);
  p.Pi = a.Pi;
  p.rowptr = a.rowptr;
  p.items = a.items;
  p.init_users = a.init_users;
  p.order = a.order;
  p.U = a.U;
  p.steps = a.cfg.steps;
  p.negs = a.cfg.negs;
  p.optimizer = a.cfg.optimizer;
  p.lr = a.cfg.lr;
  p.beta_1 = a.cfg.beta_1;
  p.beta_2 = a.cfg.beta_2;
  p.epsilon = a.cfg.epsilon;
  p.seed = a.cfg.seed;
  p.out_mlp = a.out_mlp;
  p.out_gmf = a.out_gmf;
  p.out_loss = a.out_loss;
  switch (tm) {
    case 32: return launch_fold<32>(p, smem, st);
    case 16: return launch_fold<16>(p, smem, st);
    case 8: return launch_fold<8>(p, smem, st);
    case 4: return launch_fold<4>(p, smem, st);
  }
  return MR_ERR_INVALID;
}

int launch_fold_in_project(const MrModel& m, float* Pi, cudaStream_t st) {
  const int64_t total = (int64_t)m.num_items * m.L[1];
  int64_t blocks = (total + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  fold_in_project_kernel<<<(unsigned)blocks, 256, 0, st>>>(m, Pi);
  MR_LAUNCH_CHECK("fold_in_project_kernel");
  return MR_OK;
}

int launch_fold_in_check(const int64_t* rowptr, const int32_t* items, int64_t U, int64_t nnz, int32_t num_items,
                         const int32_t* init_users, int32_t num_users, int32_t* keys, int32_t* flags, cudaStream_t st) {
  if (U == 0) return MR_OK;
  int64_t blocks = (U + 127) / 128;
  const int64_t cap = (int64_t)sm_count() * 8;
  if (blocks > cap) blocks = cap;
  fold_in_check_kernel<<<(unsigned)blocks, 128, 0, st>>>(rowptr, items, U, nnz, num_items, init_users, num_users, keys,
                                                         flags);
  MR_LAUNCH_CHECK("fold_in_check_kernel");
  return MR_OK;
}

}  // namespace mr
