// Top-k selection over whole rows of scores (one user against the whole catalogue), with a sorted exclusion list per
// row and the 0-based place of a target item among the row's candidates.
//   order: the RankLayer order of rank_positions_kernel (rank.cu) -- descending rank_key(p) (NaN ranks as -inf),
//          the lower item id first among equal keys.
//   key(p, item) = (order-reversed bits of rank_key(p) + 0.0f) << 32 | item: ascending keys are exactly that order
//          (+ 0.0f folds -0 into +0, which the float comparison treats as equal) and every key is distinct, so the
//          top k is the unique set of the k smallest keys whatever order partial results meet in: deterministic
//          without any ordering effort.
// Pass 1: one warp per (row, slice of the items).  The warp walks its slice 32 items at a time next to the row's
//         exclusion list (binary search to the slice start, then a pointer), appends the keys below its running k-th
//         best to a shared-memory buffer and, when the buffer is full, sorts it (bitonic) and keeps k.  The same pass
//         counts the candidates whose key is below the target's (an integer: order of the sum is irrelevant).
// Pass 2: one warp per row merges the <= 32 sorted slice lists (lane = slice, k rounds of a warp minimum), writes the
//         k items / scores with -1 / NaN padding and adds the slice counts into pos.
// Algorithmic bytes per row: 4 N (scores) + 4 x (exclusion list) read; 8 k x slices written and read back.
#include "topk_common.cuh"

namespace mr {

constexpr int kTopkThreads = 128;  // four warps per CTA, each with its own buffer
constexpr int kTopkMinSlice = 1024;
constexpr int kTopkMaxSlices = 32;  // one merge lane per slice

__host__ __device__ static int topk_slice_len(int32_t N) {
  int64_t s = ((int64_t)N + kTopkMaxSlices - 1) / kTopkMaxSlices;
  s = (s + 31) / 32 * 32;
  return (int)(s < kTopkMinSlice ? kTopkMinSlice : s);
}
__host__ __device__ static int topk_slices(int32_t N) {
  return (int)(((int64_t)N + topk_slice_len(N) - 1) / topk_slice_len(N));
}
static int topk_cap(int k) {  // buffer entries: a power of two >= k + 32 (room for one more warp-wide append)
  int c = 64;
  while (c < k + 32) c <<= 1;
  return c;
}

size_t topk_workspace_bytes(int64_t U, int32_t N, int32_t k) {
  if (k > kTopkSmallK) return topk_large_workspace_bytes(U, N);
  const size_t rows = (size_t)(U < 1 ? 1 : U) * topk_slices(N);
  return align_up(rows * k * sizeof(unsigned long long), 256) + align_up(rows * sizeof(int32_t), 256);
}

// Sorts buf[0, cap) ascending after padding [n, cap) with kNoKey; returns the number of entries kept (<= k).
__device__ int topk_flush(unsigned long long* buf, int n, int cap, int k, int lane) {
  for (int i = n + lane; i < cap; i += 32) buf[i] = kNoKey;
  __syncwarp();
  for (int size = 2; size <= cap; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = lane; i < cap / 2; i += 32) {
        const int a = 2 * i - (i & (stride - 1)), b = a + stride;
        const unsigned long long x = buf[a], y = buf[b];
        if ((x > y) == ((a & size) == 0)) {
          buf[a] = y;
          buf[b] = x;
        }
      }
      __syncwarp();
    }
  }
  return n < k ? n : k;
}

// Appends the lanes' keys below the running threshold thr to the warp's buffer (n entries), sorting and cutting the
// buffer to k first when a full warp might not fit; thr becomes the k-th best key once k keys are known.
__device__ __forceinline__ void topk_push(unsigned long long* buf, int& n, unsigned long long& thr,
                                          unsigned long long key, int cap, int k, int lane) {
  if (n + 32 > cap) {
    n = topk_flush(buf, n, cap, k, lane);
    if (n == k) thr = buf[k - 1];
  }
  const bool pass = key < thr;
  const uint32_t pm = __ballot_sync(0xffffffffu, pass);
  if (pass) buf[n + __popc(pm & ((1u << lane) - 1u))] = key;
  n += __popc(pm);
  __syncwarp();
}

// Merges S <= 32 ascending lists of k keys (list j at lists + j * k, kNoKey-padded) into the k smallest: k rounds of a
// warp minimum over the lists' heads (lane = list).  Keys are distinct, so each round has one winner.  emit(i, key)
// runs on lane i % 32 for i = 0 .. k-1 (key = kNoKey past the last entry).
template <class Emit>
__device__ __forceinline__ void topk_merge_warp(const unsigned long long* lists, int S, int k, int lane, Emit emit) {
  const unsigned long long* mine = lists + (size_t)lane * k;
  int cur = 0;
  unsigned long long head = lane < S ? mine[0] : kNoKey;
  for (int i = 0; i < k; ++i) {
    unsigned long long m = head;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long x = __shfl_xor_sync(0xffffffffu, m, o);
      m = x < m ? x : m;
    }
    if (m != kNoKey && head == m) {
      ++cur;
      head = cur < k ? mine[cur] : kNoKey;
    }
    if (lane == (i & 31)) emit(i, m);
  }
}

// SKIP_SELF: the row's own id a.users[gu] is never a candidate (similar items / users).
template <bool SKIP_SELF>
__global__ void __launch_bounds__(kTopkThreads) topk_slice_kernel(const TopkArgs a, int S, int slice, int cap,
                                                                  unsigned long long* __restrict__ lists,
                                                                  int32_t* __restrict__ counts) {
  extern __shared__ unsigned long long topk_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long* buf = topk_smem + (size_t)warp * cap;
  const int64_t w = (int64_t)blockIdx.x * (kTopkThreads / 32) + warp;
  if (w >= a.U * S) return;  // warp-uniform
  const int64_t u = w / S;
  const int s = (int)(w - u * S);
  const int64_t gu = a.u0 + u;
  const int N = a.N, k = a.k;
  const float* row = a.scores + u * N;
  const int lo = s * slice, hi = min(N, lo + slice);
  int64_t ep, ee;  // exclusion list: [ep, ee) from the first entry >= lo
  excl_cursor(a.excl_ids, a.excl_rows, a.excl_rowptr, a.excl_items, gu, lo, ep, ee);
  const int t = a.targets != nullptr ? __ldg(a.targets + gu) : -1;
  const bool has_t = (unsigned)t < (unsigned)N;
  const unsigned long long key_t = has_t ? topk_key(__ldg(row + t), t) : 0ull;
  const int self = SKIP_SELF ? __ldg(a.users + gu) : -1;
  int below = 0, n = 0;
  unsigned long long thr = kNoKey;
  for (int c = lo; c < hi; c += 32) {
    const uint32_t xmask = list_mask(a.excl_items, ep, ee, c, lane);  // excluded items of [c, c + 32)
    const int item = c + lane;
    const bool cand = item < hi && (!((xmask >> lane) & 1u) || item == t) &&  // the target is never excluded
                      (!SKIP_SELF || item != self);
    const unsigned long long key = cand ? topk_key(__ldg(row + item), item) : kNoKey;
    below += (has_t && key < key_t) ? 1 : 0;
    topk_push(buf, n, thr, key, cap, k, lane);
  }
  n = topk_flush(buf, n, cap, k, lane);
  unsigned long long* out = lists + (size_t)w * k;
  for (int i = lane; i < k; i += 32) out[i] = i < n ? buf[i] : kNoKey;
  below = warp_sum_int(below);
  if (lane == 0) counts[w] = below;
}

__global__ void __launch_bounds__(kTopkThreads) topk_merge_kernel(const TopkArgs a, int S,
                                                                  const unsigned long long* __restrict__ lists,
                                                                  const int32_t* __restrict__ counts) {
  const int lane = threadIdx.x & 31;
  const int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (u >= a.U) return;  // warp-uniform
  const int64_t gu = a.u0 + u;
  const int k = a.k, N = a.N;
  const bool bad_u = a.users != nullptr && (unsigned)__ldg(a.users + gu) >= (unsigned)a.num_users;
  topk_merge_warp(lists + (size_t)u * S * k, S, k, lane, [&](int i, unsigned long long m) {
    const int item = (m == kNoKey || bad_u) ? -1 : (int)(uint32_t)m;
    if (a.top_items != nullptr) a.top_items[gu * k + i] = item;
    if (a.top_scores != nullptr) a.top_scores[gu * k + i] = item < 0 ? nanf("") : __ldg(a.scores + u * N + item);
  });
  if (a.pos != nullptr) {
    int c = lane < S ? counts[u * S + lane] : 0;
    c = warp_sum_int(c);
    const int t = __ldg(a.targets + gu);
    if (lane == 0) a.pos[gu] = (bad_u || (unsigned)t >= (unsigned)N) ? N : c;
  }
}

int launch_topk(const TopkArgs& a, void* ws, cudaStream_t st, bool skip_self) {
  if (a.U == 0) return MR_OK;
  if (skip_self && a.users == nullptr) return MR_ERR_INVALID;
  if (a.k > kTopkSmallK) return launch_topk_large(a, ws, st, skip_self);
  const int S = topk_slices(a.N), slice = topk_slice_len(a.N), cap = topk_cap(a.k);
  Carver cv(ws);
  unsigned long long* lists = cv.take<unsigned long long>((size_t)a.U * S * a.k);
  int32_t* counts = cv.take<int32_t>((size_t)a.U * S);
  const int wpc = kTopkThreads / 32;
  const size_t smem = (size_t)wpc * cap * sizeof(unsigned long long);  // <= 16 KB (cap <= 512)
  const unsigned grid = (unsigned)((a.U * S + wpc - 1) / wpc);
  if (skip_self) topk_slice_kernel<true><<<grid, kTopkThreads, smem, st>>>(a, S, slice, cap, lists, counts);
  else topk_slice_kernel<false><<<grid, kTopkThreads, smem, st>>>(a, S, slice, cap, lists, counts);
  MR_LAUNCH_CHECK("topk_slice_kernel");
  topk_merge_kernel<<<(unsigned)((a.U + wpc - 1) / wpc), kTopkThreads, 0, st>>>(a, S, lists, counts);
  MR_LAUNCH_CHECK("topk_merge_kernel");
  return MR_OK;
}

// ---- ragged lists: list u is scores[rowptr[u] .. rowptr[u+1]) ---------------------------------------------------
// The same keys with the POSITION in the list as the low half: ascending keys = descending score, the earlier position
// first among ties.  A short list (<= one slice of kTopkMinSlice) is one warp from scores to final outputs.  A long list
// is cut into topk_slices(len) <= 32 slices whose warps stage k keys each, and one merge warp per long list finishes it.
// Work items: warp w < U takes slice 0 of list w; the slices 1.. of the long lists follow at U + (their rank among all
// such slices), found by a binary search over a device scan of the per-list counts -- no read-back, and the host
// bound U + ceil(nnz / 1024) covers them (a long list has fewer than len / 1024 slices beyond its first).
// Only long lists stage: fewer than 2 nnz / 1024 slices of 8 k bytes, i.e. < nnz k / 64 bytes.
// Segments are clamped to [0, nnz), so a malformed rowptr cannot make any kernel leave its arrays.

// off[u] (u = 0 .. U): low 32 bits = staged slices of the long lists before u, high 32 bits = long lists before u; the
// slices 1.. of long list u are then work items U + (low - high) ..  One CTA, 4096 lists per round.
__global__ void __launch_bounds__(1024) topk_lists_scan_kernel(const int64_t* __restrict__ rowptr, int64_t U, int64_t nnz,
                                                               unsigned long long* __restrict__ off) {
  __shared__ unsigned long long warp_tot[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long carry = 0;
  for (int64_t base = 0; base <= U; base += 4 * 1024) {
    unsigned long long v[4], t = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int64_t u = base + 4 * threadIdx.x + q;
      v[q] = 0;
      if (u < U) {
        int64_t b, e;
        list_bounds(rowptr, u, nnz, b, e);
        if (e - b > kTopkMinSlice) v[q] = (1ull << 32) | (unsigned)topk_slices((int32_t)(e - b));
      }
      t += v[q];
    }
    unsigned long long x = t;  // inclusive warp scan of the thread totals
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_tot[warp] = x;
    __syncthreads();
    if (warp == 0) {
      unsigned long long w = warp_tot[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long y = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += y;
      }
      warp_tot[lane] = w;  // inclusive over warps
    }
    __syncthreads();
    unsigned long long run = carry + (warp > 0 ? warp_tot[warp - 1] : 0ull) + x - t;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int64_t u = base + 4 * threadIdx.x + q;
      if (u <= U) off[u] = run;
      run += v[q];
    }
    carry += warp_tot[31];
    __syncthreads();
  }
}

__device__ __forceinline__ int64_t lists_extra(unsigned long long o) { return (int64_t)(uint32_t)o - (int64_t)(o >> 32); }

__global__ void __launch_bounds__(kTopkThreads) topk_lists_slice_kernel(const TopkListsArgs a, int cap,
                                                                        const unsigned long long* __restrict__ off,
                                                                        unsigned long long* __restrict__ stage,
                                                                        int32_t* __restrict__ counts, int32_t* __restrict__ pos) {
  extern __shared__ unsigned long long topk_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long* buf = topk_smem + (size_t)warp * cap;
  const int64_t w = (int64_t)blockIdx.x * (kTopkThreads / 32) + warp;
  const int64_t U = a.U;
  int64_t u;
  int s;
  if (w < U) {
    u = w;
    s = 0;
  } else {  // slice >= 1 of a long list: the last u whose extra slices start at or before e (warp-uniform search)
    const int64_t e = w - U;
    if (e >= lists_extra(off[U])) return;
    int64_t lo = 0, hi = U - 1;
    while (lo < hi) {
      const int64_t mid = (lo + hi + 1) >> 1;
      if (lists_extra(off[mid]) <= e) lo = mid;
      else hi = mid - 1;
    }
    u = lo;
    s = 1 + (int)(e - lists_extra(off[u]));
  }
  int64_t b, e;
  list_bounds(a.rowptr, u, a.nnz, b, e);
  const int len = (int)(e - b), k = a.k;
  const bool is_long = len > kTopkMinSlice;
  const int slice = is_long ? topk_slice_len(len) : kTopkMinSlice;
  const int lo = s * slice, hi = min(len, lo + slice);
  const float* sc = a.scores + b;
  const int t = a.targets != nullptr ? __ldg(a.targets + u) : -1;
  const bool has_t = (unsigned)t < (unsigned)len;
  const unsigned long long key_t = has_t ? topk_key(__ldg(sc + t), t) : 0ull;
  int below = 0, n = 0;
  unsigned long long thr = kNoKey;
  for (int c = lo; c < hi; c += 32) {
    const int j = c + lane;
    const unsigned long long key = j < hi ? topk_key(__ldg(sc + j), j) : kNoKey;
    below += (has_t && key < key_t) ? 1 : 0;
    topk_push(buf, n, thr, key, cap, k, lane);
  }
  n = topk_flush(buf, n, cap, k, lane);
  below = warp_sum_int(below);
  if (is_long) {
    const size_t slot = (uint32_t)off[u] + s;
    unsigned long long* out = stage + slot * k;
    for (int i = lane; i < k; i += 32) out[i] = i < n ? buf[i] : kNoKey;
    if (lane == 0) counts[slot] = below;
    return;
  }
  const bool bad_u = a.users != nullptr && (unsigned)__ldg(a.users + u) >= (unsigned)a.num_users;
  for (int i = lane; i < k; i += 32) lists_emit(a, u, b, i, i < n ? buf[i] : kNoKey, bad_u);
  if (pos != nullptr && lane == 0) pos[u] = (bad_u || !has_t) ? len : below;
}

__global__ void __launch_bounds__(kTopkThreads) topk_lists_merge_kernel(const TopkListsArgs a,
                                                                        const unsigned long long* __restrict__ off,
                                                                        const unsigned long long* __restrict__ stage,
                                                                        const int32_t* __restrict__ counts,
                                                                        int32_t* __restrict__ pos) {
  const int lane = threadIdx.x & 31;
  const int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (u >= a.U) return;  // warp-uniform
  int64_t b, e;
  list_bounds(a.rowptr, u, a.nnz, b, e);
  const int len = (int)(e - b);
  if (len <= kTopkMinSlice) return;  // finished by its slice warp
  const int S = topk_slices(len), k = a.k;
  const size_t slot0 = (uint32_t)off[u];
  const bool bad_u = a.users != nullptr && (unsigned)__ldg(a.users + u) >= (unsigned)a.num_users;
  topk_merge_warp(stage + slot0 * k, S, k, lane, [&](int i, unsigned long long m) { lists_emit(a, u, b, i, m, bad_u); });
  if (pos != nullptr) {
    const int c = warp_sum_int(lane < S ? counts[slot0 + lane] : 0);
    const int t = a.targets != nullptr ? __ldg(a.targets + u) : -1;
    if (lane == 0) pos[u] = (bad_u || (unsigned)t >= (unsigned)len) ? len : c;
  }
}

static int64_t lists_stage_slots(int64_t nnz) { return (nnz + 511) / 512; }  // > the staged slices of any rowptr

size_t topk_lists_workspace_bytes(int64_t U, int64_t nnz, int32_t k) {
  if (k > kTopkSmallK) return align_up((size_t)U * sizeof(int32_t), 256);  // positions when the caller wants sums only
  const size_t slots = (size_t)lists_stage_slots(nnz);
  return align_up((size_t)(U + 1) * sizeof(unsigned long long), 256) + align_up((size_t)U * sizeof(int32_t), 256) +
         align_up(slots * k * sizeof(unsigned long long), 256) + align_up(slots * sizeof(int32_t), 256);
}

int launch_topk_lists(const TopkListsArgs& a, float* sums, void* ws, cudaStream_t st) {
  if (a.k > kTopkSmallK) {
    int32_t* pos = a.pos != nullptr ? a.pos : (sums != nullptr ? static_cast<int32_t*>(ws) : nullptr);
    const int rc = launch_topk_lists_large(a, pos, st);
    return rc != MR_OK ? rc : launch_topk_metrics(pos, a.U, a.k, sums, st);
  }
  Carver cv(ws);
  unsigned long long* off = cv.take<unsigned long long>((size_t)a.U + 1);
  int32_t* pos_buf = cv.take<int32_t>((size_t)a.U);
  const size_t slots = (size_t)lists_stage_slots(a.nnz);
  unsigned long long* stage = cv.take<unsigned long long>(slots * a.k);
  int32_t* counts = cv.take<int32_t>(slots);
  int32_t* pos = a.pos != nullptr ? a.pos : (sums != nullptr ? pos_buf : nullptr);
  if (a.U > 0) {
    const int cap = topk_cap(a.k), wpc = kTopkThreads / 32;
    const size_t smem = (size_t)wpc * cap * sizeof(unsigned long long);
    const int64_t warps = a.U + (a.nnz + kTopkMinSlice - 1) / kTopkMinSlice;
    topk_lists_scan_kernel<<<1, 1024, 0, st>>>(a.rowptr, a.U, a.nnz, off);
    MR_LAUNCH_CHECK("topk_lists_scan_kernel");
    topk_lists_slice_kernel<<<(unsigned)((warps + wpc - 1) / wpc), kTopkThreads, smem, st>>>(a, cap, off, stage, counts,
                                                                                             pos);
    MR_LAUNCH_CHECK("topk_lists_slice_kernel");
    topk_lists_merge_kernel<<<(unsigned)((a.U + wpc - 1) / wpc), kTopkThreads, 0, st>>>(a, off, stage, counts, pos);
    MR_LAUNCH_CHECK("topk_lists_merge_kernel");
  }
  return launch_topk_metrics(pos, a.U, a.k, sums, st);
}

// seg[r] = the list holding row r (the last u with rowptr[u] <= r, clamped to [0, U)), or users[that list] when
// `users` is given.  One CTA per 1024 rows: two searches bound the lists of the CTA's rows, then each thread searches
// only between them.
__device__ __forceinline__ int64_t list_of_row(const int64_t* __restrict__ rowptr, int64_t lo, int64_t hi, int64_t r) {
  while (lo < hi) {  // the last u in [lo, hi] with rowptr[u] <= r (lo when none)
    const int64_t mid = (lo + hi + 1) >> 1;
    if (__ldg(rowptr + mid) <= r) lo = mid;
    else hi = mid - 1;
  }
  return lo;
}

__global__ void __launch_bounds__(1024) list_rows_kernel(const int64_t* __restrict__ rowptr, int64_t U, int64_t nnz,
                                                         const int32_t* __restrict__ users, int32_t* __restrict__ seg) {
  __shared__ int64_t bounds[2];
  const int64_t r0 = (int64_t)blockIdx.x * 1024, r1 = min(nnz, r0 + 1024) - 1;
  if (threadIdx.x < 2) bounds[threadIdx.x] = list_of_row(rowptr, 0, U - 1, threadIdx.x == 0 ? r0 : r1);
  __syncthreads();
  const int64_t r = r0 + threadIdx.x;
  if (r > r1) return;
  int64_t lo = bounds[0], hi = bounds[1];
  if (hi < lo) {  // (only a malformed rowptr)
    lo = 0;
    hi = U - 1;
  }
  const int64_t u = list_of_row(rowptr, lo, hi, r);
  seg[r] = users != nullptr ? __ldg(users + u) : (int32_t)u;
}

int launch_list_rows(const int64_t* rowptr, int64_t U, int64_t nnz, const int32_t* users, int32_t* seg, cudaStream_t st) {
  if (nnz == 0 || U == 0) return MR_OK;
  list_rows_kernel<<<(unsigned)((nnz + 1023) / 1024), 1024, 0, st>>>(rowptr, U, nnz, users, seg);
  MR_LAUNCH_CHECK("list_rows_kernel");
  return MR_OK;
}

// One CTA: thread-strided partial sums in double, then a fixed shuffle / shared-memory tree.  The positions of a call
// cover all its rows while its workspace is bounded by one chunk, so launch_rank_metrics' per-1024-row partials
// (which grow with the row count) have no place to live; this pass needs none.
__global__ void __launch_bounds__(1024) topk_metric_kernel(const int32_t* __restrict__ pos, int64_t U, int k,
                                                           float* __restrict__ sums) {
  __shared__ double red_h[32], red_d[32];
  const float ln2 = logf(2.f);
  double h = 0.0, d = 0.0;
  for (int64_t i = threadIdx.x; i < U; i += blockDim.x) {
    const int p = pos[i];
    if (p < k) {
      h += 1.0;
      d += (double)(ln2 / logf((float)p + 2.f));
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    h += __shfl_xor_sync(0xffffffffu, h, o);
    d += __shfl_xor_sync(0xffffffffu, d, o);
  }
  if ((threadIdx.x & 31) == 0) {
    red_h[threadIdx.x >> 5] = h;
    red_d[threadIdx.x >> 5] = d;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double hh = 0.0, dd = 0.0;
    for (int w = 0; w < 32; ++w) {
      hh += red_h[w];
      dd += red_d[w];
    }
    sums[0] = (float)hh;
    sums[1] = (float)dd;
  }
}

int launch_topk_metrics(const int32_t* pos, int64_t U, int k, float* sums, cudaStream_t st) {
  if (sums == nullptr) return MR_OK;
  topk_metric_kernel<<<1, 1024, 0, st>>>(pos, U, k, sums);
  MR_LAUNCH_CHECK("topk_metric_kernel");
  return MR_OK;
}

__global__ void tile_iota_kernel(int32_t* __restrict__ out, int64_t rows, int32_t N) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x)
    out[r] = (int32_t)(r % N);
}

int launch_tile_iota(int32_t* out, int64_t rows, int32_t N, cudaStream_t st) {
  if (rows == 0) return MR_OK;
  int64_t grid = (rows + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 8;
  if (grid > cap) grid = cap;
  tile_iota_kernel<<<(unsigned)grid, 256, 0, st>>>(out, rows, N);
  MR_LAUNCH_CHECK("tile_iota_kernel");
  return MR_OK;
}

// ---- positions of many targets per row: row u's targets are tgt_items[tgt_rowptr[u] .. tgt_rowptr[u+1]) ----------
// Candidates of a row: the items not excluded plus every target (a target is never excluded); order: topk_key.  The
// position of a target = the candidates with a smaller key.  Per chunk of rows:
//  sort:     one CTA per row sorts the keys of the row's targets ascending (targets outside [0, N) as kNoKey, last):
//            a block bitonic sort in shared memory up to kTgtTile keys; longer lists sort tiles of kTgtTile, then merge
//            them in global memory (each key's output place = its place in its run + its rank in the other run).
//            It also zeroes the row's histogram, n + 1 integer bins.
//  count:    one warp per (row, slice), the slices of topk_slice_kernel: the warp walks its slice next to the
//            exclusion list and the target list, and every candidate that is not a target adds 1 to bin b = the
//            number of target keys below its own (a binary search over the sorted keys, in shared memory for lists of
//            at most kTgtSmemKeys targets, else in global memory).  Integer counts: the order of the additions is
//            irrelevant.
//  finalize: one warp per row: the sorted target j has j targets and sum_{b <= j} hist[b] other candidates below it.
//            The positions land in sorted order in spos (ascending per row) and in list order in tpos.
// After the last chunk one fixed-order pass turns spos into metric sums (below), so chunking never shows in them.
// Bytes per row: 4 N (scores) + 4 x (exclusion list) + 4 t (target list) read; about 24 t of workspace traffic.
constexpr int kTgtSortThreads = 256;
constexpr int kTgtTile = 2048;     // keys a sort CTA sorts in shared memory (16 KB)
constexpr int kTgtSmemKeys = 512;  // lists up to this length are searched and counted in shared memory
constexpr int kMetricBlocks = 128, kMetricThreads = 256;

TargetsWs carve_targets(void* ws, int64_t C, int64_t nnz_t) {
  TargetsWs w{};
  Carver cv(ws);
  const size_t t = (size_t)(nnz_t < 1 ? 1 : nnz_t);
  w.keys = cv.take<unsigned long long>(t);
  w.tmp = cv.take<unsigned long long>(t);
  w.hist = cv.take<int32_t>(t + (size_t)(C < 1 ? 1 : C));
  w.spos = cv.take<int32_t>(t);
  w.partials = cv.take<double>((size_t)kMetricBlocks * kTgtSumsMax);
  w.total = cv.off;
  return w;
}

size_t targets_workspace_bytes(int64_t C, int64_t nnz_t) { return carve_targets(nullptr, C, nnz_t).total; }

__device__ __forceinline__ bool targets_bad_user(const TargetsArgs& a, int64_t gu) {
  return a.users != nullptr && (unsigned)__ldg(a.users + gu) >= (unsigned)a.num_users;
}

// Ascending bitonic sort of buf[0, cap) (cap a power of two) by the whole block.
__device__ void block_bitonic(unsigned long long* buf, int cap) {
  for (int size = 2; size <= cap; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = threadIdx.x; i < cap / 2; i += blockDim.x) {
        const int x0 = 2 * i - (i & (stride - 1)), x1 = x0 + stride;
        const unsigned long long x = buf[x0], y = buf[x1];
        if ((x > y) == ((x0 & size) == 0)) {
          buf[x0] = y;
          buf[x1] = x;
        }
      }
      __syncthreads();
    }
  }
}

// Entries of the ascending v[b, e) below x (upper = false) or not above x (upper = true).
__device__ __forceinline__ int64_t keys_rank(const unsigned long long* v, int64_t b, int64_t e, unsigned long long x,
                                             bool upper) {
  while (b < e) {
    const int64_t mid = (b + e) >> 1;
    if (v[mid] < x || (upper && v[mid] == x)) b = mid + 1;
    else e = mid;
  }
  return b;
}

__global__ void __launch_bounds__(kTgtSortThreads) targets_sort_kernel(const TargetsArgs a, const TargetsWs w) {
  __shared__ unsigned long long tile[kTgtTile];
  const int64_t u = blockIdx.x, gu = a.u0 + u;
  int64_t tb, te;
  list_bounds(a.tgt_rowptr, gu, a.nnz_t, tb, te);
  const int64_t n = te - tb;
  int32_t* hist = w.hist + tb + u;
  for (int64_t i = threadIdx.x; i <= n; i += blockDim.x) hist[i] = 0;
  if (n == 0 || targets_bad_user(a, gu)) return;  // block-uniform; finalize gives a bad row's targets N
  const int N = a.N;
  const float* row = a.scores + u * N;
  const int32_t* items = a.tgt_items + tb;
  auto key_of = [&](int64_t i) {
    const int t = __ldg(items + i);
    return (unsigned)t < (unsigned)N ? topk_key(__ldg(row + t), t) : kNoKey;
  };
  unsigned long long* keys = w.keys + tb;
  if (n <= kTgtTile) {
    int cap = 64;
    while (cap < n) cap <<= 1;
    for (int i = threadIdx.x; i < cap; i += blockDim.x) tile[i] = i < n ? key_of(i) : kNoKey;
    __syncthreads();
    block_bitonic(tile, cap);
    for (int i = threadIdx.x; i < n; i += blockDim.x) keys[i] = tile[i];
    return;
  }
  unsigned long long *src = keys, *dst = w.tmp + tb;
  for (int64_t t0 = 0; t0 < n; t0 += kTgtTile) {
    const int m = (int)(n - t0 < kTgtTile ? n - t0 : kTgtTile);
    for (int i = threadIdx.x; i < kTgtTile; i += blockDim.x) tile[i] = i < m ? key_of(t0 + i) : kNoKey;
    __syncthreads();
    block_bitonic(tile, kTgtTile);
    for (int i = threadIdx.x; i < m; i += blockDim.x) src[t0 + i] = tile[i];
    __syncthreads();
  }
  for (int64_t width = kTgtTile; width < n; width <<= 1) {  // merge runs of `width` pairwise: src -> dst
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
      const int64_t s = i / (2 * width) * (2 * width);
      const int64_t mid = s + width < n ? s + width : n, end = s + 2 * width < n ? s + 2 * width : n;
      const unsigned long long x = src[i];
      // equal keys (only kNoKey) keep the left run first, so every output place is taken once
      const int64_t p = i < mid ? (i - s) + keys_rank(src, mid, end, x, false) - mid
                                : (i - mid) + keys_rank(src, s, mid, x, true) - s;
      dst[s + p] = x;
    }
    __syncthreads();
    unsigned long long* t = src;
    src = dst;
    dst = t;
  }
  if (src != keys) {
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) keys[i] = src[i];
  }
}

__global__ void __launch_bounds__(kTopkThreads) targets_count_kernel(const TargetsArgs a, int S, int slice,
                                                                     const TargetsWs w) {
  __shared__ unsigned long long skeys[kTopkThreads / 32][kTgtSmemKeys];
  __shared__ int32_t shist[kTopkThreads / 32][kTgtSmemKeys + 1];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t wi = (int64_t)blockIdx.x * (kTopkThreads / 32) + warp;
  if (wi >= a.U * S) return;  // warp-uniform
  const int64_t u = wi / S;
  const int s = (int)(wi - u * S);
  const int64_t gu = a.u0 + u;
  int64_t tb, te;
  list_bounds(a.tgt_rowptr, gu, a.nnz_t, tb, te);
  const int64_t n = te - tb;
  if (n == 0 || targets_bad_user(a, gu)) return;
  const int N = a.N;
  const float* row = a.scores + u * N;
  const int lo = s * slice, hi = min(N, lo + slice);
  int64_t ep, ee;
  excl_cursor(a.excl_ids, a.excl_rows, a.excl_rowptr, a.excl_items, gu, lo, ep, ee);
  int64_t tp = list_lower_bound(a.tgt_items, tb, te, lo);
  const bool local = n <= kTgtSmemKeys;
  const unsigned long long* keys = w.keys + tb;
  int32_t* hist = w.hist + tb + u;
  if (local) {
    for (int i = lane; i < n; i += 32) skeys[warp][i] = keys[i];
    for (int i = lane; i <= n; i += 32) shist[warp][i] = 0;
    keys = skeys[warp];
    hist = shist[warp];
    __syncwarp();
  }
  int64_t top = 1;
  while (2 * top <= n) top <<= 1;
  for (int c = lo; c < hi; c += 32) {
    const uint32_t skip = list_mask(a.excl_items, ep, ee, c, lane) | list_mask(a.tgt_items, tp, te, c, lane);
    const int item = c + lane;
    if (item < hi && !((skip >> lane) & 1u)) {  // a candidate that is not a target
      const unsigned long long key = topk_key(__ldg(row + item), item);
      int64_t b = 0;  // target keys below key
      for (int64_t step = top; step > 0; step >>= 1)
        if (b + step <= n && keys[b + step - 1] < key) b += step;
      atomicAdd(hist + b, 1);
    }
  }
  if (local) {
    __syncwarp();
    for (int i = lane; i <= n; i += 32) {
      const int v = shist[warp][i];
      if (v != 0) atomicAdd(w.hist + tb + u + i, v);
    }
  }
}

__global__ void __launch_bounds__(kTopkThreads) targets_finalize_kernel(const TargetsArgs a, const TargetsWs w) {
  const int lane = threadIdx.x & 31;
  const int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (u >= a.U) return;  // warp-uniform
  const int64_t gu = a.u0 + u;
  int64_t tb, te;
  list_bounds(a.tgt_rowptr, gu, a.nnz_t, tb, te);
  const int64_t n = te - tb;
  const int N = a.N;
  const bool bad_u = targets_bad_user(a, gu);
  const int32_t* hist = w.hist + tb + u;
  int64_t run = 0;  // sum of hist[0, base)
  for (int64_t base = 0; base < n; base += 32) {
    const int64_t j = base + lane;
    int64_t x = (j < n && !bad_u) ? hist[j] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (j < n) {
      const unsigned long long key = bad_u ? kNoKey : w.keys[tb + j];
      const int p = key == kNoKey ? N : (int)(j + run + x);
      w.spos[tb + j] = p;
      if (a.tpos != nullptr && key != kNoKey) {
        const int64_t i = list_lower_bound(a.tgt_items, tb, te, (int)(uint32_t)key);
        if (i < te) a.tpos[i] = p;
      }
    }
    run += __shfl_sync(0xffffffffu, x, 31);
  }
  if (a.tpos != nullptr) {  // targets outside [0, N), every target of a bad row
    for (int64_t i = tb + lane; i < te; i += 32)
      if (bad_u || (unsigned)__ldg(a.tgt_items + i) >= (unsigned)N) a.tpos[i] = N;
  }
}

int launch_targets_chunk(const TargetsArgs& a, const TargetsWs& w, cudaStream_t st) {
  if (a.U == 0 || a.tgt_rowptr == nullptr) return MR_OK;
  const int S = topk_slices(a.N), slice = topk_slice_len(a.N), wpc = kTopkThreads / 32;
  targets_sort_kernel<<<(unsigned)a.U, kTgtSortThreads, 0, st>>>(a, w);
  MR_LAUNCH_CHECK("targets_sort_kernel");
  targets_count_kernel<<<(unsigned)((a.U * S + wpc - 1) / wpc), kTopkThreads, 0, st>>>(a, S, slice, w);
  MR_LAUNCH_CHECK("targets_count_kernel");
  targets_finalize_kernel<<<(unsigned)((a.U + wpc - 1) / wpc), kTopkThreads, 0, st>>>(a, w);
  MR_LAUNCH_CHECK("targets_finalize_kernel");
  return MR_OK;
}

// Sum of v over the block in a fixed order; the result is valid in thread 0.
__device__ double block_sum_double(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();  // red may still be read from the previous call
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x == 0)
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i];
  return t;
}

__device__ __forceinline__ double dcg_gain(int p) {  // topk_metric_kernel's gain, ln2 / ln(p + 2) in float
  return (double)(logf(2.f) / logf((float)p + 2.f));
}

// Per-block partial sums: users are assigned to threads by their index alone (thread-strided over a fixed grid), each
// thread adds its users in index order and the block its threads in a fixed tree, so the sums depend on U only.
__global__ void __launch_bounds__(kMetricThreads) targets_metric_kernel(const int64_t* __restrict__ rowptr, int64_t U,
                                                                        int64_t nnz_t, const int32_t* __restrict__ spos,
                                                                        const TargetCutoffs ks,
                                                                        double* __restrict__ partials) {
  __shared__ double red[kMetricThreads / 32];
  double* out = partials + (size_t)blockIdx.x * kTgtSumsMax;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x, first = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  double users = 0.0, mrr = 0.0;
  for (int64_t u = first; u < U; u += stride) {
    int64_t b, e;
    list_bounds(rowptr, u, nnz_t, b, e);
    if (e == b) continue;
    users += 1.0;
    mrr += 1.0 / ((double)spos[b] + 1.0);
  }
  double t = block_sum_double(users, red);
  if (threadIdx.x == 0) out[MR_TGT_USERS] = t;
  t = block_sum_double(mrr, red);
  if (threadIdx.x == 0) out[MR_TGT_MRR] = t;
  for (int c = 0; c < ks.n; ++c) {
    int k = ks.k[0];  // (a constant index per step keeps the parameter array out of local memory)
#pragma unroll
    for (int i = 1; i < MR_MAX_CUTOFFS; ++i)
      if (c == i) k = ks.k[i];
    double hit = 0.0, prec = 0.0, rec = 0.0, ndcg = 0.0, map = 0.0;
    for (int64_t u = first; u < U; u += stride) {
      int64_t b, e;
      list_bounds(rowptr, u, nnz_t, b, e);
      const int64_t n = e - b;
      if (n == 0) continue;
      double h = 0.0, dcg = 0.0, ap = 0.0;
      for (int64_t j = 0; j < n; ++j) {  // positions ascend: stop at the first one outside the cutoff
        const int p = spos[b + j];
        if (p >= k) break;
        h += 1.0;
        dcg += dcg_gain(p);
        ap += (double)(j + 1) / ((double)p + 1.0);
      }
      const int64_t m = n < k ? n : k;
      double idcg = 0.0;
      for (int64_t i = 0; i < m; ++i) idcg += dcg_gain((int)i);
      hit += h > 0.0 ? 1.0 : 0.0;
      prec += h / (double)k;
      rec += h / (double)n;
      ndcg += dcg / idcg;
      map += ap / (double)m;
    }
    const double v[MR_TGT_PER_CUTOFF] = {hit, prec, rec, ndcg, map};
#pragma unroll
    for (int m = 0; m < MR_TGT_PER_CUTOFF; ++m) {
      t = block_sum_double(v[m], red);
      if (threadIdx.x == 0) out[MR_TGT_CUTOFF0 + MR_TGT_PER_CUTOFF * c + m] = t;
    }
  }
}

__global__ void targets_metric_reduce_kernel(const double* __restrict__ partials, int nm, float* __restrict__ sums) {
  const int m = threadIdx.x;
  if (m >= nm) return;
  double t = 0.0;
  for (int b = 0; b < kMetricBlocks; ++b) t += partials[(size_t)b * kTgtSumsMax + m];
  sums[m] = (float)t;
}

int launch_targets_metrics(const int64_t* tgt_rowptr, int64_t U, int64_t nnz_t, const int32_t* spos,
                           const TargetCutoffs& ks, float* sums, double* partials, cudaStream_t st) {
  if (sums == nullptr) return MR_OK;
  const int nm = MR_TGT_CUTOFF0 + MR_TGT_PER_CUTOFF * ks.n;
  if (U == 0 || tgt_rowptr == nullptr) {
    MR_CUDA(cudaMemsetAsync(sums, 0, nm * sizeof(float), st));
    return MR_OK;
  }
  targets_metric_kernel<<<kMetricBlocks, kMetricThreads, 0, st>>>(tgt_rowptr, U, nnz_t, spos, ks, partials);
  MR_LAUNCH_CHECK("targets_metric_kernel");
  targets_metric_reduce_kernel<<<1, 64, 0, st>>>(partials, nm, sums);
  MR_LAUNCH_CHECK("targets_metric_reduce_kernel");
  return MR_OK;
}

// ---- audiences: the k best pool users of every item column of (pool users x items) chunks -------------------------
// Order: topk_key(p, user id), the row selection's order with the user id as the tie-break; keys are distinct, so the
// top k is unique whatever order the chunks, splits and merges meet in.  Per item the running top-k lives in the
// workspace as S lists of k keys and k raw scores (kNoKey-padded, keys ascending); split s owns the 32-row tiles
// s, s + S, s + 2S, .. of every chunk.  Per chunk, one CTA per (32 columns, split): it reads 32 x 32 tiles as 128-byte
// row segments, transposes them through shared memory, and each warp walks 4 columns, the lanes being 32 users,
// next to each column's exclusion cursor, appending the keys below the list's k-th key (topk_push).  Only a column
// with survivors touches its list: survivors and list in one buffer, one flush, and each kept key's raw score from
// the list (a binary search) or from the chunk.  After the last chunk one warp per item merges its S lists, writes
// users and scores and looks for the target in the result: pos = its slot, k when absent.
// S > 1 only when the columns alone give fewer than ~1024 CTAs, so that a narrow call (a few new items) still fills
// the GPU.  Bytes per pair: the 4-byte score, read once; per (column, chunk, split): one 8-byte threshold read and the
// cursor's binary search, plus 12 k bytes read and written when the column has survivors.
constexpr int kAudThreads = 256;
constexpr int kAudCols = 32;                                 // columns per CTA: one tile wide
constexpr int kAudColsPerWarp = kAudCols / (kAudThreads / 32);  // 4
constexpr int kAudTargetCtas = 1024;

static int audience_cap(int k) {  // survivors (<= k after a flush) + the list must fit, and one warp-wide append
  int c = 64;
  while (c < k + 32 || c < 2 * k) c <<= 1;
  return c;
}

static int audience_splits(int64_t C, int32_t M) {
  const int64_t blocks = ((int64_t)M + kAudCols - 1) / kAudCols, tiles = (C + 31) / 32;
  int64_t s = kAudTargetCtas / (blocks < 1 ? 1 : blocks);
  if (s > 32) s = 32;
  if (s > tiles) s = tiles;
  return (int)(s < 1 ? 1 : s);
}

AudienceState carve_audience(void* ws, int64_t C, int32_t M, int32_t k) {
  AudienceState st{};
  if (k > kTopkSmallK) {
    st.lg = carve_audience_large(ws, C, M, k, st.total);
    return st;
  }
  AudienceWs& w = st.w;
  Carver cv(ws);
  w.S = audience_splits(C, M);
  const size_t entries = (size_t)(M < 1 ? 1 : M) * w.S * k;
  w.keys = cv.take<unsigned long long>(entries);
  w.scores = cv.take<float>(entries);
  w.pos = cv.take<int32_t>((size_t)(M < 1 ? 1 : M));
  w.total = st.total = cv.off;
  return st;
}

// Merges the n survivors in buf into list s of column j (k keys + k scores in the workspace).
template <bool POOL>
__device__ void audience_merge(const AudienceArgs& a, const AudienceWs& w, int j, int s, unsigned long long* buf, int n,
                               int cap, int lane) {
  const int k = a.k;
  const size_t base = ((size_t)j * w.S + s) * k;
  unsigned long long* lk = w.keys + base;
  float* ls = w.scores + base;
  n = topk_flush(buf, n, cap, k, lane);
  for (int i = lane; i < k; i += 32) buf[n + i] = lk[i];
  __syncwarp();
  topk_flush(buf, n + k, cap, k, lane);
  float sc[kTopkSmallK / 32];
#pragma unroll
  for (int q = 0; q < kTopkSmallK / 32; ++q) {
    const int i = lane + 32 * q;
    sc[q] = 0.f;
    if (i >= k) continue;
    const unsigned long long key = buf[i];
    if (key == kNoKey) continue;
    int lo = 0, hi = k;  // the key's place in the old list
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (lk[mid] < key) lo = mid + 1;
      else hi = mid;
    }
    if (lo < k && lk[lo] == key) {
      sc[q] = ls[lo];
    } else {  // a survivor of this chunk: its row holds the user
      const int uid = (int)(uint32_t)key;
      const int64_t r = POOL ? list_lower_bound(a.users, a.u0, a.u0 + a.U, uid) - a.u0 : uid - a.u0;
      sc[q] = __ldg(a.scores + r * a.M + j);
    }
  }
  __syncwarp();  // every lane has read the old list
#pragma unroll
  for (int q = 0; q < kTopkSmallK / 32; ++q) {
    const int i = lane + 32 * q;
    if (i < k) {
      lk[i] = buf[i];
      ls[i] = sc[q];
    }
  }
}

template <bool POOL>
__global__ void __launch_bounds__(kAudThreads) audience_chunk_kernel(const AudienceArgs a, const AudienceWs w, int cap) {
  extern __shared__ unsigned long long aud_smem[];
  __shared__ float tile[32][33];
  __shared__ int ids[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int S = w.S, s = blockIdx.y, k = a.k, M = a.M;
  const int64_t C = a.U, first = (int64_t)s * 32;
  if (first >= C) return;  // block-uniform: the last chunk may be short
  const int j0 = blockIdx.x * kAudCols;
  const int lo_user = POOL ? __ldg(a.users + a.u0 + first) : (int)(a.u0 + first);
  int n[kAudColsPerWarp], t[kAudColsPerWarp];
  unsigned long long thr[kAudColsPerWarp];
  int64_t ep[kAudColsPerWarp], ee[kAudColsPerWarp];
#pragma unroll
  for (int q = 0; q < kAudColsPerWarp; ++q) {
    const int j = j0 + warp * kAudColsPerWarp + q;
    n[q] = 0;
    t[q] = -1;
    thr[q] = kNoKey;
    ep[q] = ee[q] = 0;
    if (j < M) {
      thr[q] = w.keys[((size_t)j * S + s) * k + k - 1];
      excl_cursor(a.excl_ids, a.excl_rows, a.excl_rowptr, a.excl_users, j, lo_user, ep[q], ee[q]);
      if (a.targets != nullptr) t[q] = __ldg(a.targets + j);
    }
  }
  for (int64_t r0 = first; r0 < C; r0 += (int64_t)32 * S) {
    const int col = j0 + lane;
    for (int rr = warp; rr < 32; rr += kAudThreads / 32) {
      const int64_t r = r0 + rr;
      tile[rr][lane] = (r < C && col < M) ? __ldg(a.scores + r * M + col) : 0.f;
    }
    if (warp == 0) {
      const int64_t r = r0 + lane;
      ids[lane] = r < C ? (POOL ? __ldg(a.users + a.u0 + r) : (int)(a.u0 + r)) : INT_MAX;
    }
    __syncthreads();
    const int uid = ids[lane];
    const bool ok = r0 + lane < C && uid >= 0 && uid < a.num_users;
#pragma unroll
    for (int q = 0; q < kAudColsPerWarp; ++q) {
      const int c = warp * kAudColsPerWarp + q;
      if (j0 + c >= M) break;  // warp-uniform
      const uint32_t x = POOL ? ids_mask(a.excl_users, ep[q], ee[q], ids, lane)
                              : list_mask(a.excl_users, ep[q], ee[q], (int)(a.u0 + r0), lane);
      const bool cand = ok && (!((x >> lane) & 1u) || uid == t[q]);  // the target is never excluded
      const unsigned long long key = cand ? topk_key(tile[lane][c], uid) : kNoKey;
      topk_push(aud_smem + (size_t)c * cap, n[q], thr[q], key, cap, k, lane);
    }
    __syncthreads();
  }
#pragma unroll
  for (int q = 0; q < kAudColsPerWarp; ++q) {
    const int c = warp * kAudColsPerWarp + q;
    if (j0 + c < M && n[q] > 0) audience_merge<POOL>(a, w, j0 + c, s, aud_smem + (size_t)c * cap, n[q], cap, lane);
  }
}

// One warp per item: the k smallest keys of its S lists (topk_merge_warp's rule, carrying the raw scores).
__global__ void __launch_bounds__(kTopkThreads) audience_final_kernel(const AudienceArgs a, const AudienceWs w,
                                                                      const int32_t* __restrict__ items,
                                                                      int32_t num_items, int32_t* __restrict__ top_users,
                                                                      float* __restrict__ top_scores,
                                                                      int32_t* __restrict__ pos) {
  const int lane = threadIdx.x & 31;
  const int64_t j = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (j >= a.M) return;  // warp-uniform
  const int k = a.k, S = w.S;
  const bool bad = items != nullptr && (unsigned)__ldg(items + j) >= (unsigned)num_items;
  const int t = a.targets != nullptr ? __ldg(a.targets + j) : -1;
  const size_t mine = ((size_t)j * S + lane) * k;
  int cur = 0, hit = k;
  unsigned long long head = lane < S ? w.keys[mine] : kNoKey;
  for (int i = 0; i < k; ++i) {
    unsigned long long m = head;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long x = __shfl_xor_sync(0xffffffffu, m, o);
      m = x < m ? x : m;
    }
    const bool win = m != kNoKey && head == m;  // distinct keys: one winner at most
    float sc = win ? w.scores[mine + cur] : 0.f;
    const uint32_t wm = __ballot_sync(0xffffffffu, win);
    sc = __shfl_sync(0xffffffffu, sc, wm ? __ffs(wm) - 1 : 0);
    if (win) {
      ++cur;
      head = cur < k ? w.keys[mine + cur] : kNoKey;
    }
    const int user = (m == kNoKey || bad) ? -1 : (int)(uint32_t)m;
    if (lane == (i & 31)) {
      if (top_users != nullptr) top_users[j * k + i] = user;
      if (top_scores != nullptr) top_scores[j * k + i] = user < 0 ? nanf("") : sc;
    }
    if (user >= 0 && user == t && hit == k) hit = i;
  }
  if (pos != nullptr && lane == 0) pos[j] = hit;
}

int launch_audience_init(const AudienceArgs& a, const AudienceState& state, cudaStream_t st) {
  if (a.k > kTopkSmallK) return launch_audience_large_init(a, state.lg, st);
  const AudienceWs& w = state.w;
  MR_CUDA(cudaMemsetAsync(w.keys, 0xff, (size_t)a.M * w.S * a.k * sizeof(unsigned long long), st));
  const size_t smem = (size_t)kAudCols * audience_cap(a.k) * sizeof(unsigned long long);  // <= 128 KB
  MR_CUDA(cudaFuncSetAttribute(audience_chunk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  MR_CUDA(cudaFuncSetAttribute(audience_chunk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  return MR_OK;
}

int launch_audience_chunk(const AudienceArgs& a, const AudienceState& state, cudaStream_t st) {
  if (a.U == 0 || a.M == 0) return MR_OK;
  if (a.k > kTopkSmallK) return launch_audience_large_chunk(a, state.lg, st);
  const AudienceWs& w = state.w;
  const int cap = audience_cap(a.k);
  const size_t smem = (size_t)kAudCols * cap * sizeof(unsigned long long);
  const dim3 grid((unsigned)(((int64_t)a.M + kAudCols - 1) / kAudCols), (unsigned)w.S);
  if (a.users != nullptr) audience_chunk_kernel<true><<<grid, kAudThreads, smem, st>>>(a, w, cap);
  else audience_chunk_kernel<false><<<grid, kAudThreads, smem, st>>>(a, w, cap);
  MR_LAUNCH_CHECK("audience_chunk_kernel");
  return MR_OK;
}

int launch_audience_final(const AudienceArgs& a, const AudienceState& state, const int32_t* items, int32_t num_items,
                          int32_t* top_users, float* top_scores, int32_t* pos, float* sums, cudaStream_t st) {
  if (a.M == 0) {
    if (sums != nullptr) MR_CUDA(cudaMemsetAsync(sums, 0, 2 * sizeof(float), st));
    return MR_OK;
  }
  if (a.k > kTopkSmallK) {
    int32_t* p = pos != nullptr ? pos : (sums != nullptr ? state.lg.pos : nullptr);
    const int rc = launch_audience_large_final(a, state.lg, items, num_items, top_users, top_scores, p, st);
    return rc != MR_OK ? rc : launch_topk_metrics(p, a.M, a.k, sums, st);
  }
  const AudienceWs& w = state.w;
  int32_t* p = pos != nullptr ? pos : (sums != nullptr ? w.pos : nullptr);
  const int wpc = kTopkThreads / 32;
  audience_final_kernel<<<(unsigned)(((int64_t)a.M + wpc - 1) / wpc), kTopkThreads, 0, st>>>(a, w, items, num_items,
                                                                                             top_users, top_scores, p);
  MR_LAUNCH_CHECK("audience_final_kernel");
  return launch_topk_metrics(p, a.M, a.k, sums, st);
}

__global__ void iota_kernel(int32_t* __restrict__ out, int64_t n, int64_t first) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x)
    out[r] = (int32_t)(first + r);
}

int launch_iota(int32_t* out, int64_t n, int64_t first, cudaStream_t st) {
  if (n == 0) return MR_OK;
  int64_t grid = (n + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 8;
  if (grid > cap) grid = cap;
  iota_kernel<<<(unsigned)grid, 256, 0, st>>>(out, n, first);
  MR_LAUNCH_CHECK("iota_kernel");
  return MR_OK;
}

__global__ void tile_list_kernel(int32_t* __restrict__ out, int64_t rows, const int32_t* __restrict__ items, int32_t M) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x)
    out[r] = __ldg(items + r % M);
}

int launch_tile_list(int32_t* out, int64_t rows, const int32_t* items, int32_t M, cudaStream_t st) {
  if (rows == 0) return MR_OK;
  int64_t grid = (rows + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 8;
  if (grid > cap) grid = cap;
  tile_list_kernel<<<(unsigned)grid, 256, 0, st>>>(out, rows, items, M);
  MR_LAUNCH_CHECK("tile_list_kernel");
  return MR_OK;
}

}  // namespace mr
