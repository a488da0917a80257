// Data-parallel replicas on one box: all-reduce(sum) of the gradients + optimizer step + all-gather of the new
// weights as ONE kernel over NVLink peer memory (SURVEY 8e; the reference is single-process, so there is no reference
// collective to mirror -- this is the exchange step of the data-parallel train step).
//
// Every rank owns a contiguous slice [lo, hi) of a region of the flat parameter buffer.  For its slice a rank
//   1. loads the `world` ranks' gradient values straight from their HBM (peer pointers) and adds them in rank order
//      0, 1, ..., world-1 -- the same order on every rank for every element, so the sum is deterministic;
//   2. adds the tables' l2 term, runs legacy-Keras Adam / SGD with ITS OWN m and v (optimizer state is sharded:
//      1/world of the sweep's HBM bytes per rank);
//   3. stores the new weights into every rank's parameter buffer (peer stores): replicas stay bit-identical by
//      construction.
// NVLink traffic per rank: (world-1)/world of the region inbound for the gradients, the same again inbound for the
// weights written by the other owners; local HBM: the slice's p, m, v.  What an NCCL all-reduce followed by a full
// optimizer sweep moves in two passes (and 28 B/element of local HBM on every rank) goes through once.
// With multicast addresses of the two buffers (NVSwitch / NVLS) steps 1 and 3 are one `multimem.ld_reduce` and one
// `multimem.st` per 16 bytes: the switch adds the replicas' values and replicates the store, so a rank receives its
// slice's sum once instead of `world` values and sends its new weights once instead of `world - 1` times -- per rank
// (1/world + (world-1)/world) of the region in each direction instead of 2 (world-1)/world.  The order in which the
// switch adds is its own (fixed for a given group of GPUs); replicas still end bit-identical.
// The caller orders the kernel against the producers of the gradients and the readers of the weights on the OTHER
// ranks with cross-rank barriers (movierec/_distributed.py).
#include "launchers.h"

namespace mr {

constexpr int kDpThreads = 128;   // small CTAs with few registers: they fit next to a persistent tcgen05 CTA
constexpr int kDpMaxWorld = 16;

struct DpPeers {
  const float* g[kDpMaxWorld];
  float* p[kDpMaxWorld];
};

// the element arithmetic of mr_optimizer_flat (common.cuh): the exchange's step is bit-identical to the flat sweep's
__device__ __forceinline__ void adam4(float4& p, const float4& g, float4& m, float4& v, float lr_t, float b1, float b2,
                                      float eps) {
  adam_step(p.x, g.x, m.x, v.x, lr_t, b1, b2, eps);
  adam_step(p.y, g.y, m.y, v.y, lr_t, b1, b2, eps);
  adam_step(p.z, g.z, m.z, v.z, lr_t, b1, b2, eps);
  adam_step(p.w, g.w, m.w, v.w, lr_t, b1, b2, eps);
}

// NVSwitch multicast (NVLS): one load that the switch answers with the SUM of the word in every replica of a
// multicast object, one store that the switch replicates into all of them.
__device__ __forceinline__ float4 multimem_ld_sum(const float4* mc) {
  float4 r;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(mc)
               : "memory");
  return r;
}
__device__ __forceinline__ void multimem_st(float4* mc, const float4& v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}

// lo4 / hi4: the slice in units of four floats (every region starts 256-byte aligned and is padded to 64 floats).
// WORLD = 0: the multicast form (mc_g / mc_p: multicast addresses of the gradient / parameter buffers).
// A thread keeps U elements in flight (the peer form has WORLD loads per element already).
template <bool ADAM, int WORLD>
__global__ void __launch_bounds__(kDpThreads) dp_reduce_apply_kernel(const DpPeers peers, int rank, float* __restrict__ m,
                                                                     float* __restrict__ v, int64_t lo4, int64_t hi4,
                                                                     float lr_t, float b1, float b2, float eps, float l2,
                                                                     const float4* mc_g, float4* mc_p) {
  constexpr int U = WORLD == 0 ? 4 : (WORLD <= 2 ? 2 : 1);
  const int64_t nth = (int64_t)gridDim.x * blockDim.x;
  const float c2 = 2.f * l2;
  const float4* p_own = reinterpret_cast<const float4*>(peers.p[rank]);
  for (int64_t i0 = lo4 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < hi4; i0 += nth * U) {
    float4 g[U], pv[U], mv[U], vv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = i0 + u * nth;
      if (i < hi4) {
        if (WORLD == 0) {
          g[u] = multimem_ld_sum(mc_g + i);
        } else {
          float4 gr[WORLD > 0 ? WORLD : 1];
#pragma unroll
          for (int r = 0; r < WORLD; ++r) gr[r] = __ldcg(reinterpret_cast<const float4*>(peers.g[r]) + i);
          g[u] = gr[0];
#pragma unroll
          for (int r = 1; r < WORLD; ++r) {  // rank order: the same sum on every rank
            g[u].x += gr[r].x; g[u].y += gr[r].y; g[u].z += gr[r].z; g[u].w += gr[r].w;
          }
        }
        pv[u] = p_own[i];
        if (ADAM) {
          mv[u] = reinterpret_cast<const float4*>(m)[i];
          vv[u] = reinterpret_cast<const float4*>(v)[i];
        }
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = i0 + u * nth;
      if (i < hi4) {
        if (l2 != 0.f) {
          g[u].x = plus_l2(g[u].x, pv[u].x, c2); g[u].y = plus_l2(g[u].y, pv[u].y, c2);
          g[u].z = plus_l2(g[u].z, pv[u].z, c2); g[u].w = plus_l2(g[u].w, pv[u].w, c2);
        }
        if (ADAM) {
          adam4(pv[u], g[u], mv[u], vv[u], lr_t, b1, b2, eps);
          reinterpret_cast<float4*>(m)[i] = mv[u];
          reinterpret_cast<float4*>(v)[i] = vv[u];
        } else {
          pv[u].x = sgd_step(pv[u].x, g[u].x, lr_t); pv[u].y = sgd_step(pv[u].y, g[u].y, lr_t);
          pv[u].z = sgd_step(pv[u].z, g[u].z, lr_t); pv[u].w = sgd_step(pv[u].w, g[u].w, lr_t);
        }
        if (WORLD == 0) {
          multimem_st(mc_p + i, pv[u]);
        } else {
#pragma unroll
          for (int r = 0; r < WORLD; ++r) reinterpret_cast<float4*>(peers.p[r])[i] = pv[u];
        }
      }
    }
  }
}

template <bool ADAM>
static int launch_world(const DpPeers& peers, int world, int rank, float* m, float* v, int64_t lo4, int64_t hi4,
                        float lr_t, float b1, float b2, float eps, float l2, const float* mc_g, float* mc_p,
                        cudaStream_t st) {
  int64_t blocks = (hi4 - lo4 + kDpThreads - 1) / kDpThreads;
  const int64_t cap = (int64_t)sm_count() * 4;
  if (blocks > cap) blocks = cap;
  if (mc_g != nullptr && mc_p != nullptr) world = 0;
#define MR_DP_CASE(W)                                                                                               \
  case W:                                                                                                           \
    dp_reduce_apply_kernel<ADAM, W><<<(unsigned)blocks, kDpThreads, 0, st>>>(                                       \
        peers, rank, m, v, lo4, hi4, lr_t, b1, b2, eps, l2, reinterpret_cast<const float4*>(mc_g),                  \
        reinterpret_cast<float4*>(mc_p));                                                                           \
    break;
  switch (world) {
    MR_DP_CASE(0) MR_DP_CASE(1) MR_DP_CASE(2) MR_DP_CASE(3) MR_DP_CASE(4) MR_DP_CASE(5) MR_DP_CASE(6) MR_DP_CASE(7)
    MR_DP_CASE(8) MR_DP_CASE(16)
    default:
      set_error("dp_reduce_apply: world size %d (1..8 or 16 ranks of one box)", world);
      return MR_ERR_INVALID;
  }
#undef MR_DP_CASE
  MR_LAUNCH_CHECK("dp_reduce_apply_kernel");
  return MR_OK;
}

int launch_dp_reduce_apply(const float* const* grad_peers, float* const* param_peers, int world, int rank, float* m,
                           float* v, int64_t lo, int64_t hi, int optimizer, float lr_t, float beta_1, float beta_2,
                           float epsilon, float l2, const float* grad_multicast, float* param_multicast,
                           cudaStream_t st) {
  if (hi <= lo) return MR_OK;
  DpPeers peers{};
  for (int r = 0; r < world; ++r) {
    peers.g[r] = grad_peers[r];
    peers.p[r] = param_peers[r];
  }
  if (optimizer == MR_OPT_ADAM)
    return launch_world<true>(peers, world, rank, m, v, lo >> 2, hi >> 2, lr_t, beta_1, beta_2, epsilon, l2,
                              grad_multicast, param_multicast, st);
  return launch_world<false>(peers, world, rank, m, v, lo >> 2, hi >> 2, lr_t, beta_1, beta_2, epsilon, l2,
                             grad_multicast, param_multicast, st);
}

}  // namespace mr
