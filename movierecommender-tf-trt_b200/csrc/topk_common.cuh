// Shared by the per-warp selection (topk.cu) and the large-k selection (topk_large.cu): the RankLayer keys, the
// exclusion-list cursors and the clamped list segments.  See topk.cu for the order the keys encode.
#pragma once
#include <limits.h>

#include "launchers.h"

namespace mr {

constexpr unsigned long long kNoKey = ~0ull;

__device__ __forceinline__ unsigned long long topk_key(float p, int item) {
  uint32_t b = __float_as_uint(rank_key(p) + 0.0f);
  b = (b & 0x80000000u) ? ~b : (b | 0x80000000u);  // ascending with the float value
  return ((unsigned long long)(~b) << 32) | (uint32_t)item;
}

// The first index of the ascending list items[b, e) whose entry is >= v (e when none).
__device__ __forceinline__ int64_t list_lower_bound(const int32_t* __restrict__ items, int64_t b, int64_t e, int v) {
  while (b < e) {
    const int64_t mid = (b + e) >> 1;
    if (__ldg(items + mid) < v) b = mid + 1;
    else e = mid;
  }
  return b;
}

// A warp's cursor [ep, ee) into the exclusion list of global row gu, from the first entry >= lo (empty when the row
// has no list).
__device__ __forceinline__ void excl_cursor(const int32_t* __restrict__ excl_ids, int32_t excl_rows,
                                            const int64_t* __restrict__ excl_rowptr, const int32_t* __restrict__ excl_items,
                                            int64_t gu, int lo, int64_t& ep, int64_t& ee) {
  ep = ee = 0;
  if (excl_rowptr == nullptr) return;
  const int64_t r = excl_ids != nullptr ? (int64_t)__ldg(excl_ids + gu) : gu;
  if (r >= 0 && r < excl_rows) {
    ee = excl_rowptr[r + 1];
    ep = list_lower_bound(excl_items, excl_rowptr[r], ee, lo);
  }
}

// Bit i = items[ep, ee) holds c + i, for a warp walking its items 32 at a time in ascending c; advances ep past the
// entries below c + 32.  Warp-uniform: lists are sorted, so the entries below c + 32 are a prefix of the lanes.
__device__ __forceinline__ uint32_t list_mask(const int32_t* __restrict__ items, int64_t& ep, int64_t ee, int c,
                                              int lane) {
  uint32_t mask = 0;
  for (;;) {
    const int64_t i = ep + lane;
    const int e = i < ee ? __ldg(items + i) : INT_MAX;
    const bool in = e < c + 32;
    const int nin = __popc(__ballot_sync(0xffffffffu, in));
    mask |= __reduce_or_sync(0xffffffffu, (in && e >= c) ? 1u << (e - c) : 0u);
    ep += nin;
    if (nin < 32) break;
  }
  return mask;
}

// Bit i = the ascending list items[ep, ee) holds ids[i], for ids ascending over i (INT_MAX past the chunk's end);
// advances ep past the entries <= ids[31].  The pool's counterpart of list_mask: each list entry finds its place among
// the 32 ids by a binary search in shared memory.
__device__ __forceinline__ uint32_t ids_mask(const int32_t* __restrict__ items, int64_t& ep, int64_t ee,
                                             const int* ids, int lane) {
  const int last = ids[31];
  uint32_t mask = 0;
  for (;;) {
    const int64_t i = ep + lane;
    const int e = i < ee ? __ldg(items + i) : 0;
    const bool in = i < ee && e <= last;
    const int nin = __popc(__ballot_sync(0xffffffffu, in));
    uint32_t bit = 0;
    if (in) {
      int p = 0;  // ids below e (< 32: e <= last)
#pragma unroll
      for (int step = 16; step > 0; step >>= 1)
        if (ids[p + step - 1] < e) p += step;
      bit = ids[p] == e ? 1u << p : 0u;
    }
    mask |= __reduce_or_sync(0xffffffffu, bit);
    ep += nin;
    if (nin < 32) break;
  }
  return mask;
}

__device__ __forceinline__ void list_bounds(const int64_t* __restrict__ rowptr, int64_t u, int64_t nnz, int64_t& b,
                                            int64_t& e) {
  b = __ldg(rowptr + u);
  e = __ldg(rowptr + u + 1);
  b = b < 0 ? 0 : (b > nnz ? nnz : b);
  e = e < b ? b : (e > nnz ? nnz : e);
}

// Final outputs of slot i of list u (list start b, length len) from key m.
__device__ __forceinline__ void lists_emit(const TopkListsArgs& a, int64_t u, int64_t b, int i, unsigned long long m,
                                           bool bad_u) {
  const int p = (m == kNoKey || bad_u) ? -1 : (int)(uint32_t)m;
  const size_t o = (size_t)u * a.k + i;
  if (a.top_pos != nullptr) a.top_pos[o] = p;
  if (a.top_items != nullptr) a.top_items[o] = p < 0 ? -1 : __ldg(a.items + b + p);
  if (a.top_scores != nullptr) a.top_scores[o] = p < 0 ? nanf("") : __ldg(a.scores + b + p);
}

}  // namespace mr
