// The negative sampler's draws, shared by the batch sampler (sampler.cu) and the fold-in kernel (fold_in.cu) so that
// both draw exactly the same items for the same (list, index, epoch, seed).
//
// Draw j of a group uses word (j % 4) of
//   Philox4x32-10(counter = (j / 4, index.lo, index.hi, epoch.lo), key = (seed.lo, seed.hi ^ epoch.hi))
// so the output is a pure function of the arguments (no RNG state, any launch geometry).  A 32-bit word x picks
// r = (x * n) >> 32 among the n candidates still available; r is then mapped to the r-th item that is neither in the
// user's sorted interaction list nor already picked -- exact uniform sampling without replacement
// (data_pipeline.py:108-112).  With fewer candidates than `negs` the reference samples WITH replacement (:111); so does
// this.  oracle/movierec_oracle.py:device_sample_group restates this bit for bit.
#pragma once

#include "common.cuh"

namespace mr {

struct Philox {
  uint32_t c[4];
};

__device__ __forceinline__ Philox philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0;
    c1 = lo1;
    c2 = n2;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  Philox o;
  o.c[0] = c0; o.c[1] = c1; o.c[2] = c2; o.c[3] = c3;
  return o;
}

// The r-th item outside the ascending list seen[0, deg): item = r + #{t : seen[t] - t <= r}
__device__ __forceinline__ int unseen_item(const int32_t* __restrict__ seen, int deg, int r) {
  int a = 0, b = deg;
  while (a < b) {
    const int mid = (a + b) >> 1;
    if (__ldg(seen + mid) - mid <= r) a = mid + 1;
    else b = mid;
  }
  return r + a;
}

// The `negs` negatives of one positive: emit(j, item) for j = 0 .. negs-1, in draw order.  seen = the user's ascending
// list of deg items; `picked` has room for negs ints (the sorted candidate ranks already taken).  Item 0 for every draw
// when no item is left.
template <typename Emit>
__device__ __forceinline__ void draw_negatives(const int32_t* __restrict__ seen, int deg, int32_t num_items, int negs,
                                               uint64_t index, uint64_t seed, uint64_t epoch, int* picked, Emit emit) {
  // the candidates are arange(num_items) minus the seen items (np.setdiff1d, data_pipeline.py:104-108): seen ids at
  // or beyond num_items (raw id spaces, a patched num_items) take no candidate away
  if (deg > 0 && __ldg(seen + deg - 1) >= num_items) {
    int a = 0, b = deg;
    while (a < b) {
      const int mid = (a + b) >> 1;
      if (__ldg(seen + mid) < num_items) a = mid + 1;
      else b = mid;
    }
    deg = a;
  }
  const int C = num_items - deg;
  const bool replace = C < negs;
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32) ^ (uint32_t)(epoch >> 32);
  Philox w;
  int npicked = 0;
  for (int j = 0; j < negs; ++j) {
    if ((j & 3) == 0) w = philox4x32_10((uint32_t)(j >> 2), (uint32_t)index, (uint32_t)(index >> 32), (uint32_t)epoch, k0, k1);
    const uint32_t x = w.c[j & 3];
    int item = 0;
    if (C > 0) {
      const uint32_t nc = (uint32_t)(replace ? C : C - j);
      int r = (int)__umulhi(x, nc);
      if (!replace) {
        int ins = 0;
        while (ins < npicked && r >= picked[ins]) {  // skip past every earlier pick at or below r
          ++r;
          ++ins;
        }
        for (int q = npicked; q > ins; --q) picked[q] = picked[q - 1];
        picked[ins] = r;
        ++npicked;
      }
      item = unseen_item(seen, deg, r);
    }
    emit(j, item);
  }
}

}  // namespace mr
