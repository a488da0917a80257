// Elementwise legacy-Keras optimizers over a flat fp32 buffer (movierec/model.py:197-204; SURVEY
// App. A-4):  Adam  m = b1*m + (1-b1)*g ; v = b2*v + (1-b2)*g^2 ; p -= lr_t * m / (sqrt(v) + eps)
// with lr_t = lr*sqrt(1-b2^t)/(1-b1^t) computed on the host;  SGD  p -= lr*g.
// `l2` adds the regulariser gradient 2*l2*p (embedding tables with layers_l2reg[0] != 0).
// Every path computes an element with common.cuh's adam_step / sgd_step / plus_l2: the same bits whatever the path.
// HBM-bound: 28 bytes per element (read p,g,m,v; write p,m,v); 128-bit accesses, grid-stride.
#include "launchers.h"

namespace mr {

template <bool ADAM>
__global__ void __launch_bounds__(256) optimizer_flat_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                             float* __restrict__ m, float* __restrict__ v,
                                                             int64_t n, float lr_t, float b1, float b2, float eps,
                                                             float l2, bool vec) {
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nth = (int64_t)gridDim.x * blockDim.x;
  const float c2 = 2.f * l2;
  if (vec) {
    const int64_t n4 = n >> 2;
    for (int64_t i = tid; i < n4; i += nth) {
      float4 pv = reinterpret_cast<float4*>(p)[i];
      float4 gv = reinterpret_cast<const float4*>(g)[i];
      if (l2 != 0.f) {
        gv.x = plus_l2(gv.x, pv.x, c2); gv.y = plus_l2(gv.y, pv.y, c2);
        gv.z = plus_l2(gv.z, pv.z, c2); gv.w = plus_l2(gv.w, pv.w, c2);
      }
      if (ADAM) {
        float4 mv = reinterpret_cast<float4*>(m)[i];
        float4 vv = reinterpret_cast<float4*>(v)[i];
        adam_step(pv.x, gv.x, mv.x, vv.x, lr_t, b1, b2, eps);
        adam_step(pv.y, gv.y, mv.y, vv.y, lr_t, b1, b2, eps);
        adam_step(pv.z, gv.z, mv.z, vv.z, lr_t, b1, b2, eps);
        adam_step(pv.w, gv.w, mv.w, vv.w, lr_t, b1, b2, eps);
        reinterpret_cast<float4*>(m)[i] = mv;
        reinterpret_cast<float4*>(v)[i] = vv;
      } else {
        pv.x = sgd_step(pv.x, gv.x, lr_t); pv.y = sgd_step(pv.y, gv.y, lr_t);
        pv.z = sgd_step(pv.z, gv.z, lr_t); pv.w = sgd_step(pv.w, gv.w, lr_t);
      }
      reinterpret_cast<float4*>(p)[i] = pv;
    }
    for (int64_t i = (n4 << 2) + tid; i < n; i += nth) {
      const float gi = l2 != 0.f ? plus_l2(g[i], p[i], c2) : g[i];
      if (ADAM) adam_step(p[i], gi, m[i], v[i], lr_t, b1, b2, eps);
      else p[i] = sgd_step(p[i], gi, lr_t);
    }
  } else {
    for (int64_t i = tid; i < n; i += nth) {
      const float gi = l2 != 0.f ? plus_l2(g[i], p[i], c2) : g[i];
      if (ADAM) adam_step(p[i], gi, m[i], v[i], lr_t, b1, b2, eps);
      else p[i] = sgd_step(p[i], gi, lr_t);
    }
  }
}

// The same sweep over up to kMaxOptRegions buffers in ONE launch (the five launches of a small model's update -- dense
// block + four tables -- cost more in launch latency than in bytes): a block belongs to one region and strides over it
// with that region's other blocks.  128-bit path only (launch_optimizer_regions falls back to per-region launches).
template <bool ADAM>
__global__ void __launch_bounds__(256) optimizer_regions_kernel(const OptRegions r, float lr_t, float b1, float b2,
                                                                float eps) {
  int k = 0;
#pragma unroll
  for (int i = 1; i < kMaxOptRegions; ++i)
    if (i < r.count && (int)blockIdx.x >= r.block_start[i]) k = i;
  const int64_t nth = (int64_t)(r.block_start[k + 1] - r.block_start[k]) * blockDim.x;
  const int64_t tid = (int64_t)((int)blockIdx.x - r.block_start[k]) * blockDim.x + threadIdx.x;
  float* __restrict__ p = r.p[k];
  const float* __restrict__ g = r.g[k];
  float* __restrict__ m = r.m[k];
  float* __restrict__ v = r.v[k];
  const int64_t n = r.n[k], n4 = n >> 2;
  const float l2 = r.l2[k], c2 = 2.f * l2;
  for (int64_t i = tid; i < n4; i += nth) {
    float4 pv = reinterpret_cast<float4*>(p)[i];
    float4 gv = reinterpret_cast<const float4*>(g)[i];
    if (l2 != 0.f) {
      gv.x = plus_l2(gv.x, pv.x, c2); gv.y = plus_l2(gv.y, pv.y, c2);
      gv.z = plus_l2(gv.z, pv.z, c2); gv.w = plus_l2(gv.w, pv.w, c2);
    }
    if (ADAM) {
      float4 mv = reinterpret_cast<float4*>(m)[i];
      float4 vv = reinterpret_cast<float4*>(v)[i];
      adam_step(pv.x, gv.x, mv.x, vv.x, lr_t, b1, b2, eps);
      adam_step(pv.y, gv.y, mv.y, vv.y, lr_t, b1, b2, eps);
      adam_step(pv.z, gv.z, mv.z, vv.z, lr_t, b1, b2, eps);
      adam_step(pv.w, gv.w, mv.w, vv.w, lr_t, b1, b2, eps);
      reinterpret_cast<float4*>(m)[i] = mv;
      reinterpret_cast<float4*>(v)[i] = vv;
    } else {
      pv.x = sgd_step(pv.x, gv.x, lr_t); pv.y = sgd_step(pv.y, gv.y, lr_t);
        pv.z = sgd_step(pv.z, gv.z, lr_t); pv.w = sgd_step(pv.w, gv.w, lr_t);
    }
    reinterpret_cast<float4*>(p)[i] = pv;
  }
  for (int64_t i = (n4 << 2) + tid; i < n; i += nth) {
    const float gi = l2 != 0.f ? plus_l2(g[i], p[i], c2) : g[i];
    if (ADAM) adam_step(p[i], gi, m[i], v[i], lr_t, b1, b2, eps);
    else p[i] = sgd_step(p[i], gi, lr_t);
  }
}

int launch_optimizer_regions(OptRegions r, int optimizer, float lr_t, float beta_1, float beta_2, float epsilon,
                             cudaStream_t st) {
  uintptr_t a = 0;
  int count = 0;
  OptRegions q{};
  for (int i = 0; i < r.count; ++i) {  // drop empty regions
    if (r.n[i] <= 0) continue;
    q.p[count] = r.p[i]; q.g[count] = r.g[i]; q.m[count] = r.m[i]; q.v[count] = r.v[i];
    q.n[count] = r.n[i]; q.l2[count] = r.l2[i];
    a |= reinterpret_cast<uintptr_t>(r.p[i]) | reinterpret_cast<uintptr_t>(r.g[i]);
    if (optimizer == MR_OPT_ADAM) a |= reinterpret_cast<uintptr_t>(r.m[i]) | reinterpret_cast<uintptr_t>(r.v[i]);
    ++count;
  }
  q.count = count;
  if (count == 0) return MR_OK;
  if ((a & 15) != 0) {  // unaligned buffers: the scalar path of the per-region kernel
    for (int i = 0; i < count; ++i) {
      const int rc = launch_optimizer_flat(q.p[i], q.g[i], q.m[i], q.v[i], q.n[i], optimizer, lr_t, beta_1, beta_2,
                                           epsilon, q.l2[i], st);
      if (rc != MR_OK) return rc;
    }
    return MR_OK;
  }
  const int64_t cap = (int64_t)sm_count() * 16;
  q.block_start[0] = 0;
  for (int i = 0; i < count; ++i) {
    int64_t blocks = (q.n[i] / 4 + 255) / 256;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    q.block_start[i + 1] = q.block_start[i] + (int)blocks;
  }
  if (optimizer == MR_OPT_ADAM)
    optimizer_regions_kernel<true><<<(unsigned)q.block_start[count], 256, 0, st>>>(q, lr_t, beta_1, beta_2, epsilon);
  else
    optimizer_regions_kernel<false><<<(unsigned)q.block_start[count], 256, 0, st>>>(q, lr_t, beta_1, beta_2, epsilon);
  MR_LAUNCH_CHECK("optimizer_regions_kernel");
  return MR_OK;
}

int launch_optimizer_flat(float* p, const float* g, float* m, float* v, int64_t n, int optimizer, float lr_t,
                          float beta_1, float beta_2, float epsilon, float l2, cudaStream_t st) {
  if (n == 0) return MR_OK;
  uintptr_t a = reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g);
  if (optimizer == MR_OPT_ADAM) a |= reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v);
  const bool vec = (a & 15) == 0;
  int64_t blocks = ((vec ? n / 4 : n) + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  if (optimizer == MR_OPT_ADAM)
    optimizer_flat_kernel<true><<<(unsigned)blocks, 256, 0, st>>>(p, g, m, v, n, lr_t, beta_1, beta_2, epsilon, l2, vec);
  else
    optimizer_flat_kernel<false><<<(unsigned)blocks, 256, 0, st>>>(p, g, m, v, n, lr_t, beta_1, beta_2, epsilon, l2, vec);
  MR_LAUNCH_CHECK("optimizer_flat_kernel");
  return MR_OK;
}

}  // namespace mr
