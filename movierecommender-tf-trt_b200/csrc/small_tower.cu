// The reference's DEFAULT tower (trainer.py DEFAULT_PARAMS: layers 64-32-16-8, here with GMF 8) as a projected,
// grouped train step on CUDA cores.  The layer widths are below every tensor-core tile, and the whole per-row network
// after the first layer is 32 -> 16 -> 8 -> 1: small enough for ONE THREAD per group of rows with everything in
// registers.  model.py:154-188 (Embedding + concat + Dense/ReLU + sigmoid head), :213-215 (BCE), backward of the same.
//
//   z1[r] = E_item[i_r] . W1i + (E_user[u_r] . W1u + b1) = Pi[i_r] + Pu[u_r]          (first layer, linear before ReLU)
//
//   small_rows_gemm_kernel        Pi = E_item . W1i, Pu = E_user . W1u + b1 over the TABLES (and, backward,
//                                 dE = S . W1^T on the per-item / per-user sums S of dZ1)
//   small_tower_train_kernel      thread = group (user row loaded once), loop over its rows: gather Pi row, ReLU,
//                                 32->16->8 forward from shared-memory weights, head + GMF, BCE, full backward to dZ1,
//                                 staged rows [dZ1 | GMF row gradient] per row (items) and per group (users).
//                                 Weight gradients: the warp stages its 32 rows' activations / pre-activation
//                                 gradients in shared memory and every lane owns a slice of the accumulators
//                                 (lane k: dW2[k][0..15], ...), so each outer product is computed once, in registers,
//                                 in a fixed order; CTAs write their sums to their row of the partial buffer.
//   small_table_wgrad_kernel      dW1 = E^T . S (and db1 = colsum(Su)) over the tables, per-CTA partial rows.
// No atomics on floats; results are bit-identical run to run.
#include <mutex>

#include "launchers.h"

namespace mr {
namespace st {

constexpr int L1 = 32, L2 = 16, L3 = 8, F = 8;
constexpr int SW = L1 + F;          // staged row: [dZ1 | GMF row gradient]
#ifndef MR_ST_CTAS
#define MR_ST_CTAS 4  // resident CTAs per SM the register budget is set for (A/B: tools/build_variant.sh)
#endif
constexpr int kWarps = 4, kThreads = kWarps * 32;
constexpr int H1S = 33, DS = 28, H2S = 17, HDS = 17;  // row strides of the per-warp staging tiles (floats)
constexpr int kWarpFloats = 32 * (H1S + DS + H2S + HDS);
constexpr int kSlots = 22;                            // per-lane accumulators: dW2 row 16, dW3 part 4, d w_out, bias sums

// The 681 weights behind the first layer -- W2 (32x16), b2, W3 (16x8), b3, w_out (16), b_out: contiguous in the model's
// dense block from W[2] on -- are copied into constant memory before every launch (one 2.7 KB device-to-device copy on
// the caller's stream) and enter the FMAs as constant-bank operands.  From shared memory the broadcast reads of the
// weights alone were 1,280 of the kernel's 2,100 shared-memory wavefronts per 32 rows, and the LSU bound it (0.135 ms
// for 327,680 rows; DESIGN 4.1).
constexpr int kConstFloats = L1 * L2 + L2 + L2 * L3 + L3 + F + L3 + 1;
__constant__ float c_w[kConstFloats];
constexpr int cW2 = 0, cB2 = cW2 + L1 * L2, cW3 = cB2 + L2, cB3 = cW3 + L2 * L3, cWO = cB3 + L3, cBO = cWO + F + L3;

struct Params {
  const float *Pi, *Pu, *gmf_u, *gmf_i;
  const int32_t *users, *items;
  const float* labels;
  int64_t G;
  int num_users, num_items;
  float inv_batch;
  float *probs, *stage_i, *stage_u;
  float* partial;  // this launch's rows of the dense partial buffer (row = CTA), offsets of the blocks below
  int64_t stride;
  int off_W2, off_b2, off_W3, off_b3, off_wout, off_bout;
  float* loss_partial;
  int32_t* flags;
};

template <int GROUP>
__global__ void __launch_bounds__(kThreads, MR_ST_CTAS) small_tower_train_kernel(const Params p) {
  extern __shared__ __align__(16) float smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float* h1_s = smem + warp * kWarpFloats;
  float* d_s = h1_s + 32 * H1S;   // per row: dZ2 [0,16), dZ3 [16,24), dz [24]
  float* h2_s = d_s + 32 * DS;
  float* hd_s = h2_s + 32 * H2S;  // per row: GMF products [0,8), h3 [8,16)

  float acc2[L2], acc3[4], dwo = 0.f, misc = 0.f, loss = 0.f;
#pragma unroll
  for (int j = 0; j < L2; ++j) acc2[j] = 0.f;
#pragma unroll
  for (int j = 0; j < 4; ++j) acc3[j] = 0.f;
  const int k3 = lane & 15, q3 = 4 + (lane >> 4), mi = lane < 24 ? lane : 24;
  bool any_bad = false;

  for (int64_t g0 = ((int64_t)blockIdx.x * kWarps + warp) * 32; g0 < p.G; g0 += (int64_t)gridDim.x * kThreads) {
    const int64_t g = g0 + lane;
    const bool live = g < p.G;
    float gu[F], gug[F], gsum[L1];
    bool bad_u = false;
    int u = 0, it_next = 0;
    if (live) {
      u = __ldg(p.users + g * GROUP);
      it_next = __ldg(p.items + g * GROUP);
      bad_u = (unsigned)u >= (unsigned)p.num_users;
      if (bad_u) u = 0;
      const float4* gu4 = reinterpret_cast<const float4*>(p.gmf_u + (size_t)u * F);
#pragma unroll
      for (int c = 0; c < F / 4; ++c) {
        const float4 a = __ldg(gu4 + c);
        gu[4 * c] = a.x; gu[4 * c + 1] = a.y; gu[4 * c + 2] = a.z; gu[4 * c + 3] = a.w;
      }
    } else {  // idle lane of the last iteration: zero pre-activation gradients, so its rows add nothing below
#pragma unroll
      for (int k = 0; k < DS; ++k) d_s[lane * DS + k] = 0.f;
#pragma unroll
      for (int k = 0; k < L2; ++k) h2_s[lane * H2S + k] = 0.f;
#pragma unroll
      for (int k = 0; k < F + L3; ++k) hd_s[lane * HDS + k] = 0.f;
    }
#pragma unroll
    for (int k = 0; k < L1; ++k) gsum[k] = 0.f;
#pragma unroll
    for (int k = 0; k < F; ++k) gug[k] = 0.f;

#pragma unroll 1
    for (int j = 0; j < GROUP; ++j) {
      const int64_t row = g * GROUP + j;
      int it = it_next;
      if (live && j + 1 < GROUP) it_next = __ldg(p.items + row + 1);  // one row ahead of its use
      const bool bad = live && (bad_u || (unsigned)it >= (unsigned)p.num_items);
      if (bad || !live) it = 0;
      // h1 = relu(Pi[item] + Pu[user]) of the warp's 32 rows: lane = unit, a row is one coalesced 128-byte load of each
      // table; eight rows in flight
#pragma unroll
      for (int r0 = 0; r0 < 32; r0 += 8) {
        float a[8], b[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const int ir = __shfl_sync(0xffffffffu, it, r0 + q), ur = __shfl_sync(0xffffffffu, u, r0 + q);
          a[q] = __ldg(p.Pi + (size_t)ir * L1 + lane);
          b[q] = __ldg(p.Pu + (size_t)ur * L1 + lane);
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) h1_s[(r0 + q) * H1S + lane] = fmaxf(a[q] + b[q], 0.f);
      }
      __syncwarp();
      if (live) {
        any_bad |= bad;
        const float y = __ldg(p.labels + row);
        const float4* gi4 = reinterpret_cast<const float4*>(p.gmf_i + (size_t)it * F);
        float gi[F];
#pragma unroll
        for (int c = 0; c < F / 4; ++c) {
          const float4 a = __ldg(gi4 + c);
          gi[4 * c] = a.x; gi[4 * c + 1] = a.y; gi[4 * c + 2] = a.z; gi[4 * c + 3] = a.w;
        }
        // ---- forward ----
        float z2[L2];
#pragma unroll
        for (int o = 0; o < L2; ++o) z2[o] = c_w[cB2 + o];
        uint32_t m1 = 0;
#pragma unroll
        for (int k = 0; k < L1; ++k) {
          const float hv = h1_s[lane * H1S + k];
          if (hv > 0.f) m1 |= 1u << k;
#pragma unroll
          for (int o = 0; o < L2; ++o) z2[o] = fmaf(hv, c_w[cW2 + k * L2 + o], z2[o]);
        }
        uint32_t m2 = 0;
        float z3[L3];
#pragma unroll
        for (int o = 0; o < L3; ++o) z3[o] = c_w[cB3 + o];
#pragma unroll
        for (int k = 0; k < L2; ++k) {
          const float h = fmaxf(z2[k], 0.f);
          h2_s[lane * H2S + k] = h;
          if (h > 0.f) m2 |= 1u << k;
#pragma unroll
          for (int o = 0; o < L3; ++o) z3[o] = fmaf(h, c_w[cW3 + k * L3 + o], z3[o]);
        }
        uint32_t m3 = 0;
        float s = c_w[cBO];
#pragma unroll
        for (int f = 0; f < F; ++f) {
          const float gp = gu[f] * gi[f];
          hd_s[lane * HDS + f] = gp;
          s = fmaf(c_w[cWO + f], gp, s);
        }
#pragma unroll
        for (int o = 0; o < L3; ++o) {
          const float h = fmaxf(z3[o], 0.f);
          hd_s[lane * HDS + F + o] = h;
          if (h > 0.f) m3 |= 1u << o;
          s = fmaf(c_w[cWO + F + o], h, s);
        }
        const float pr = sigmoidf_stable(s);
        const float dz = bad ? 0.f : (pr - y) * p.inv_batch;
        if (!bad) loss += bce_logits(s, y);
        if (p.probs != nullptr) p.probs[row] = bad ? nanf("") : pr;
        // ---- backward ----
        float dz3[L3];
#pragma unroll
        for (int o = 0; o < L3; ++o) dz3[o] = ((m3 >> o) & 1u) ? dz * c_w[cWO + F + o] : 0.f;
        float* si = p.stage_i + (size_t)row * SW;
        {
          float gq[F];
#pragma unroll
          for (int f = 0; f < F; ++f) {
            const float gv = dz * c_w[cWO + f];
            gug[f] = fmaf(gv, gi[f], gug[f]);
            gq[f] = gv * gu[f];
          }
          reinterpret_cast<float4*>(si + L1)[0] = make_float4(gq[0], gq[1], gq[2], gq[3]);
          reinterpret_cast<float4*>(si + L1)[1] = make_float4(gq[4], gq[5], gq[6], gq[7]);
        }
        float dz2[L2];
#pragma unroll
        for (int k = 0; k < L2; ++k) {
          float v = 0.f;
#pragma unroll
          for (int o = 0; o < L3; ++o) v = fmaf(dz3[o], c_w[cW3 + k * L3 + o], v);
          dz2[k] = ((m2 >> k) & 1u) ? v : 0.f;
        }
        float4* dq = reinterpret_cast<float4*>(d_s + lane * DS);
        dq[0] = make_float4(dz2[0], dz2[1], dz2[2], dz2[3]);
        dq[1] = make_float4(dz2[4], dz2[5], dz2[6], dz2[7]);
        dq[2] = make_float4(dz2[8], dz2[9], dz2[10], dz2[11]);
        dq[3] = make_float4(dz2[12], dz2[13], dz2[14], dz2[15]);
        dq[4] = make_float4(dz3[0], dz3[1], dz3[2], dz3[3]);
        dq[5] = make_float4(dz3[4], dz3[5], dz3[6], dz3[7]);
        d_s[lane * DS + 24] = dz;
#pragma unroll
        for (int c = 0; c < L1 / 4; ++c) {
          float o4[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int k = 4 * c + q;
            float v = 0.f;
#pragma unroll
            for (int o = 0; o < L2; ++o) v = fmaf(dz2[o], c_w[cW2 + k * L2 + o], v);
            v = ((m1 >> k) & 1u) ? v : 0.f;
            gsum[k] += v;
            o4[q] = v;
          }
          reinterpret_cast<float4*>(si)[c] = make_float4(o4[0], o4[1], o4[2], o4[3]);
        }
      }
      __syncwarp();
      // ---- weight gradients of the warp's 32 rows: lane = one slice of the accumulators ----
#pragma unroll 4
      for (int r = 0; r < 32; ++r) {
        const float a = h1_s[r * H1S + lane];
        const float4* dr = reinterpret_cast<const float4*>(d_s + r * DS);
#pragma unroll
        for (int o4 = 0; o4 < L2 / 4; ++o4) {
          const float4 dv = dr[o4];
          acc2[4 * o4] = fmaf(a, dv.x, acc2[4 * o4]);
          acc2[4 * o4 + 1] = fmaf(a, dv.y, acc2[4 * o4 + 1]);
          acc2[4 * o4 + 2] = fmaf(a, dv.z, acc2[4 * o4 + 2]);
          acc2[4 * o4 + 3] = fmaf(a, dv.w, acc2[4 * o4 + 3]);
        }
        const float b = h2_s[r * H2S + k3];
        const float4 t3 = dr[q3];
        acc3[0] = fmaf(b, t3.x, acc3[0]); acc3[1] = fmaf(b, t3.y, acc3[1]);
        acc3[2] = fmaf(b, t3.z, acc3[2]); acc3[3] = fmaf(b, t3.w, acc3[3]);
        dwo = fmaf(d_s[r * DS + 24], hd_s[r * HDS + k3], dwo);
        misc += d_s[r * DS + mi];
      }
      __syncwarp();
    }
    if (live) {
      float4* su = reinterpret_cast<float4*>(p.stage_u + (size_t)g * SW);
#pragma unroll
      for (int c = 0; c < L1 / 4; ++c) su[c] = make_float4(gsum[4 * c], gsum[4 * c + 1], gsum[4 * c + 2], gsum[4 * c + 3]);
      su[L1 / 4] = make_float4(gug[0], gug[1], gug[2], gug[3]);
      su[L1 / 4 + 1] = make_float4(gug[4], gug[5], gug[6], gug[7]);
    }
  }
  if (any_bad) atomicOr(p.flags, 1);

  // ---- per-CTA sums, fixed order over the warps, into this CTA's row of the partial buffer ----
  __syncthreads();
  float* red = smem;  // [warp][slot][lane]
  {
    float* rw = red + warp * kSlots * 32;
#pragma unroll
    for (int j = 0; j < L2; ++j) rw[j * 32 + lane] = acc2[j];
#pragma unroll
    for (int j = 0; j < 4; ++j) rw[(16 + j) * 32 + lane] = acc3[j];
    rw[20 * 32 + lane] = dwo;
    rw[21 * 32 + lane] = misc;
  }
  loss = warp_sum(loss);
  __shared__ float loss_s[kWarps];
  if (lane == 0) loss_s[warp] = loss;
  __syncthreads();
  auto total = [&](int slot, int ln) {
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) v += red[(w * kSlots + slot) * 32 + ln];
    return v;
  };
  float* out = p.partial + (size_t)blockIdx.x * p.stride;
  for (int i = tid; i < L1 * L2; i += kThreads) out[p.off_W2 + i] = total(i % L2, i / L2);
  for (int i = tid; i < L2 * L3; i += kThreads) {
    const int k = i / L3, j = i % L3;
    out[p.off_W3 + i] = total(16 + (j & 3), k + 16 * (j >> 2));
  }
  if (tid < F + L3) out[p.off_wout + tid] = total(20, tid);
  if (tid < L2) out[p.off_b2 + tid] = total(21, tid);
  if (tid < L3) out[p.off_b3 + tid] = total(21, 16 + tid);
  if (tid == 0) {
    out[p.off_bout] = total(21, 24);
    float l = 0.f;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) l += loss_s[w];
    p.loss_partial[blockIdx.x] = l;
  }
}

// Ranking eval / forward: thread = candidate row, `group` consecutive rows share users[row / group].  The row's Pi and
// Pu are read as eight 16-byte pieces (the user's row hits L1 for the group's other candidates), layers 2-3 and the
// output unit run in registers on constant-bank weights, one probability is stored per row (NaN for a bad id).
// RAGGED (candidate lists): row r belongs to list seg[r] of num_lists; its user is users[seg[r]] and its Pu row is
// seg[r] (Pu holds one row per list).
template <bool RAGGED>
__global__ void __launch_bounds__(256) small_tower_forward_kernel(const float* __restrict__ Pi, const float* __restrict__ Pu,
                                                                  const float* __restrict__ gmf_u,
                                                                  const float* __restrict__ gmf_i,
                                                                  const int32_t* __restrict__ users,
                                                                  const int32_t* __restrict__ items, int64_t rows, int group,
                                                                  int num_users, int num_items, float* __restrict__ probs,
                                                                  const int32_t* __restrict__ seg, int64_t num_lists) {
  for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < rows; row += (int64_t)gridDim.x * blockDim.x) {
    int u, pr, it = __ldg(items + row);
    if (RAGGED) {
      pr = __ldg(seg + row);
      u = (unsigned)pr < (uint64_t)num_lists ? __ldg(users + pr) : -1;
    } else {
      pr = u = __ldg(users + row / group);
    }
    const bool bad = (unsigned)u >= (unsigned)num_users || (unsigned)it >= (unsigned)num_items;
    if (bad) pr = u = it = 0;
    const float4* pi4 = reinterpret_cast<const float4*>(Pi + (size_t)it * L1);
    const float4* pu4 = reinterpret_cast<const float4*>(Pu + (size_t)pr * L1);
    float z2[L2];
#pragma unroll
    for (int o = 0; o < L2; ++o) z2[o] = c_w[cB2 + o];
#pragma unroll
    for (int c = 0; c < L1 / 4; ++c) {
      const float4 a = __ldg(pi4 + c), b = __ldg(pu4 + c);
      const float hv[4] = {fmaxf(a.x + b.x, 0.f), fmaxf(a.y + b.y, 0.f), fmaxf(a.z + b.z, 0.f), fmaxf(a.w + b.w, 0.f)};
#pragma unroll
      for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int o = 0; o < L2; ++o) z2[o] = fmaf(hv[q], c_w[cW2 + (4 * c + q) * L2 + o], z2[o]);
    }
    float z3[L3];
#pragma unroll
    for (int o = 0; o < L3; ++o) z3[o] = c_w[cB3 + o];
#pragma unroll
    for (int k = 0; k < L2; ++k) {
      const float h = fmaxf(z2[k], 0.f);
#pragma unroll
      for (int o = 0; o < L3; ++o) z3[o] = fmaf(h, c_w[cW3 + k * L3 + o], z3[o]);
    }
    float s = c_w[cBO];
    const float4* gu4 = reinterpret_cast<const float4*>(gmf_u + (size_t)u * F);
    const float4* gi4 = reinterpret_cast<const float4*>(gmf_i + (size_t)it * F);
#pragma unroll
    for (int c = 0; c < F / 4; ++c) {
      const float4 a = __ldg(gu4 + c), b = __ldg(gi4 + c);
      s = fmaf(c_w[cWO + 4 * c], a.x * b.x, s);
      s = fmaf(c_w[cWO + 4 * c + 1], a.y * b.y, s);
      s = fmaf(c_w[cWO + 4 * c + 2], a.z * b.z, s);
      s = fmaf(c_w[cWO + 4 * c + 3], a.w * b.w, s);
    }
#pragma unroll
    for (int o = 0; o < L3; ++o) s = fmaf(c_w[cWO + F + o], fmaxf(z3[o], 0.f), s);
    probs[row] = bad ? nanf("") : sigmoidf_stable(s);
  }
}

// out[r][j] = (bias ? bias[j] : 0) + sum_k A[r][k] * Wv(k, j), Wv(k, j) = transpose ? W[j * ldw + k] : W[k * ldw + j];
// K, N multiples of 4, K * N <= 4096.  256 threads = 256 / (N / 4) rows per CTA, four outputs per thread.
__global__ void __launch_bounds__(256) small_rows_gemm_kernel(const float* __restrict__ A, int64_t rows, int K,
                                                              const float* __restrict__ W, int ldw, int N, int transpose,
                                                              const float* __restrict__ bias, float* __restrict__ out) {
  __shared__ __align__(16) float W_s[4096];
  for (int i = threadIdx.x; i < K * N; i += 256) {
    const int k = i / N, j = i % N;
    W_s[i] = transpose ? W[(size_t)j * ldw + k] : W[(size_t)k * ldw + j];
  }
  __syncthreads();
  const int nq = N >> 2, rpc = 256 / nq;
  const int rl = threadIdx.x / nq, jq = threadIdx.x % nq;
  if (rl >= rpc) return;
  for (int64_t r = (int64_t)blockIdx.x * rpc + rl; r < rows; r += (int64_t)gridDim.x * rpc) {
    float4 acc = bias != nullptr ? *reinterpret_cast<const float4*>(bias + 4 * jq) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float4* a4 = reinterpret_cast<const float4*>(A + (size_t)r * K);
    for (int k4 = 0; k4 < (K >> 2); ++k4) {
      const float4 a = __ldg(a4 + k4);
      const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 w = *reinterpret_cast<const float4*>(W_s + (4 * k4 + q) * N + 4 * jq);
        acc.x = fmaf(av[q], w.x, acc.x); acc.y = fmaf(av[q], w.y, acc.y);
        acc.z = fmaf(av[q], w.z, acc.z); acc.w = fmaf(av[q], w.w, acc.w);
      }
    }
    *reinterpret_cast<float4*>(out + (size_t)r * N + 4 * jq) = acc;
  }
}

// dW[i][j] = sum_r E[r][i] * S[r][j] (i < 32, j < 32), db[j] = sum_r S[r][j]: CTA = chunks of 32 rows staged in
// shared memory, thread = (i, four j); the CTA's sum goes to its row of the partial buffer.
constexpr int kWgRows = 32;
__global__ void __launch_bounds__(256) small_table_wgrad_kernel(const float* __restrict__ E, const float* __restrict__ S,
                                                                int64_t rows, float* __restrict__ dw_partial,
                                                                float* __restrict__ db_partial, int64_t stride) {
  __shared__ __align__(16) float E_s[kWgRows * 33];
  __shared__ __align__(16) float S_s[kWgRows * 32];
  const int i = threadIdx.x >> 3, jq = threadIdx.x & 7;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  float db = 0.f;
  for (int64_t r0 = (int64_t)blockIdx.x * kWgRows; r0 < rows; r0 += (int64_t)gridDim.x * kWgRows) {
    const int n = (int)(rows - r0 < kWgRows ? rows - r0 : kWgRows);
    __syncthreads();
    for (int t = threadIdx.x; t < kWgRows * 32; t += 256) {
      const int r = t >> 5, c = t & 31;
      E_s[r * 33 + c] = r < n ? __ldg(E + (size_t)(r0 + r) * 32 + c) : 0.f;
      S_s[t] = r < n ? __ldg(S + (size_t)(r0 + r) * 32 + c) : 0.f;
    }
    __syncthreads();
#pragma unroll 4
    for (int r = 0; r < kWgRows; ++r) {
      const float e = E_s[r * 33 + i];
      const float4 s = *reinterpret_cast<const float4*>(S_s + r * 32 + 4 * jq);
      acc.x = fmaf(e, s.x, acc.x); acc.y = fmaf(e, s.y, acc.y); acc.z = fmaf(e, s.z, acc.z); acc.w = fmaf(e, s.w, acc.w);
    }
    if (db_partial != nullptr && threadIdx.x < 32)
      for (int r = 0; r < kWgRows; ++r) db += S_s[r * 32 + threadIdx.x];
  }
  float* dw = dw_partial + (size_t)blockIdx.x * stride;
  *reinterpret_cast<float4*>(dw + i * 32 + 4 * jq) = acc;
  if (db_partial != nullptr && threadIdx.x < 32) db_partial[(size_t)blockIdx.x * stride + threadIdx.x] = db;
}

}  // namespace st

// __constant__ memory is per device; so is the event recorded after the kernel that reads the image
constexpr int kMaxDevices = 64;
static std::mutex g_const_mutex;
static cudaEvent_t g_const_free_of[kMaxDevices] = {};

// (call with g_const_mutex held) waits for the last reader of the constant image, then copies this model's weights
static int upload_weights(const MrModel& m, cudaStream_t stream, cudaEvent_t* free_event) {
  int dev = 0;
  MR_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= kMaxDevices) {
    set_error("small tower: device ordinal %d out of range", dev);
    return MR_ERR_INVALID;
  }
  cudaEvent_t& g_const_free = g_const_free_of[dev];
  if (g_const_free == nullptr) MR_CUDA(cudaEventCreateWithFlags(&g_const_free, cudaEventDisableTiming));
  *free_event = g_const_free;
  MR_CUDA(cudaStreamWaitEvent(stream, g_const_free, 0));
  MR_CUDA(cudaMemcpyToSymbolAsync(st::c_w, m.W[2], st::kConstFloats * sizeof(float), 0, cudaMemcpyDeviceToDevice, stream));
  return MR_OK;
}

bool small_tower_supported(const MrModel& m, int group) {
  return m.n_layers == 4 && m.L[0] == 2 * st::L1 && m.L[1] == st::L1 && m.L[2] == st::L2 && m.L[3] == st::L3 &&
         m.mf_dim == st::F && group == 5;
}

int launch_small_tower_train(const SmallTowerArgs& a, cudaStream_t stream, int* grid_out) {
  const MrModel& m = *a.model;
  st::Params p{};
  p.Pi = a.Pi; p.Pu = a.Pu; p.gmf_u = m.user_gmf; p.gmf_i = m.item_gmf;
  p.users = a.users; p.items = a.items; p.labels = a.labels;
  p.G = a.B / 5;
  p.num_users = m.num_users; p.num_items = m.num_items;
  p.inv_batch = a.inv_batch;
  p.probs = a.probs; p.stage_i = a.stage_i; p.stage_u = a.stage_u;
  p.partial = a.dense_partial; p.stride = a.dense_stride;
  p.off_W2 = (int)(m.W[2] - m.dense); p.off_b2 = (int)(m.b[2] - m.dense);
  p.off_W3 = (int)(m.W[3] - m.dense); p.off_b3 = (int)(m.b[3] - m.dense);
  p.off_wout = (int)(m.w_out - m.dense); p.off_bout = (int)(m.b_out - m.dense);
  p.loss_partial = a.loss_partial; p.flags = a.flags;
  const size_t smem = (size_t)(st::kWarps * st::kWarpFloats) * sizeof(float);
  auto kern = st::small_tower_train_kernel<5>;
  static_assert((size_t)(st::kWarps * st::kWarpFloats) * sizeof(float) <= 48 * 1024, "fits the default dynamic shared memory");
  int occ = 0;
  MR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, st::kThreads, smem));
  if (occ < 1) occ = 1;
  int64_t grid = (p.G + st::kThreads - 1) / st::kThreads;
  const int64_t cap = (int64_t)sm_count() * occ < a.max_ctas ? (int64_t)sm_count() * occ : a.max_ctas;
  if (grid > cap) grid = cap;
  if (grid < 1) grid = 1;
  // the constant image belongs to one launch at a time: a launch on another stream waits for the previous kernel
  {
    std::lock_guard<std::mutex> lock(g_const_mutex);
    cudaEvent_t g_const_free = nullptr;
    int rc = upload_weights(m, stream, &g_const_free);
    if (rc != MR_OK) return rc;
    kern<<<(unsigned)grid, st::kThreads, smem, stream>>>(p);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "small_tower_train_kernel");
    count_launch();
    MR_CUDA(cudaEventRecord(g_const_free, stream));
  }
  *grid_out = (int)grid;
  return MR_OK;
}

int launch_small_tower_forward(const MrModel& m, const float* Pi, const float* Pu, const int32_t* users,
                               const int32_t* items, int64_t rows, int group, float* probs, cudaStream_t stream,
                               const int32_t* seg, int64_t num_lists) {
  if (rows == 0) return MR_OK;
  int64_t grid = (rows + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 8;
  if (grid > cap) grid = cap;
  std::lock_guard<std::mutex> lock(g_const_mutex);
  cudaEvent_t g_const_free = nullptr;
  int rc = upload_weights(m, stream, &g_const_free);
  if (rc != MR_OK) return rc;
  if (seg != nullptr)
    st::small_tower_forward_kernel<true><<<(unsigned)grid, 256, 0, stream>>>(Pi, Pu, m.user_gmf, m.item_gmf, users, items,
                                                                           rows, 1, m.num_users, m.num_items, probs, seg,
                                                                           num_lists);
  else
    st::small_tower_forward_kernel<false><<<(unsigned)grid, 256, 0, stream>>>(Pi, Pu, m.user_gmf, m.item_gmf, users, items,
                                                                            rows, group, m.num_users, m.num_items, probs,
                                                                            nullptr, 0);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "small_tower_forward_kernel");
  count_launch();
  MR_CUDA(cudaEventRecord(g_const_free, stream));
  return MR_OK;
}

int launch_small_rows_gemm(const float* A, int64_t rows, int K, const float* W, int ldw, int N, bool transpose,
                           const float* bias, float* out, cudaStream_t stream) {
  if (rows == 0) return MR_OK;
  if ((K & 3) || (N & 3) || K * N > 4096 || N > 256) {
    set_error("small_rows_gemm: K=%d N=%d not supported", K, N);
    return MR_ERR_INVALID;
  }
  const int rpc = 256 / (N >> 2);
  int64_t grid = (rows + rpc - 1) / rpc;
  const int64_t cap = (int64_t)sm_count() * 8;
  if (grid > cap) grid = cap;
  st::small_rows_gemm_kernel<<<(unsigned)grid, 256, 0, stream>>>(A, rows, K, W, ldw, N, transpose ? 1 : 0, bias, out);
  MR_LAUNCH_CHECK("small_rows_gemm_kernel");
  return MR_OK;
}

int launch_small_table_wgrad(const float* E, const float* S, int64_t rows, float* dw_partial, float* db_partial,
                             int64_t stride, int max_ctas, cudaStream_t stream, int* grid_out) {
  int64_t grid = (rows + st::kWgRows - 1) / st::kWgRows;
  if (grid > max_ctas) grid = max_ctas;
  if (grid < 1) grid = 1;
  st::small_table_wgrad_kernel<<<(unsigned)grid, 256, 0, stream>>>(E, S, rows, dw_partial, db_partial, stride);
  MR_LAUNCH_CHECK("small_table_wgrad_kernel");
  *grid_out = (int)grid;
  return MR_OK;
}

}  // namespace mr
