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
#include <limits.h>

#include "launchers.h"

namespace mr {

constexpr int kTopkThreads = 128;  // four warps per CTA, each with its own buffer
constexpr int kTopkMinSlice = 1024;
constexpr int kTopkMaxSlices = 32;  // one merge lane per slice
constexpr unsigned long long kNoKey = ~0ull;

static int topk_slice_len(int32_t N) {
  int64_t s = ((int64_t)N + kTopkMaxSlices - 1) / kTopkMaxSlices;
  s = (s + 31) / 32 * 32;
  return (int)(s < kTopkMinSlice ? kTopkMinSlice : s);
}
static int topk_slices(int32_t N) { return (int)(((int64_t)N + topk_slice_len(N) - 1) / topk_slice_len(N)); }
static int topk_cap(int k) {  // buffer entries: a power of two >= k + 32 (room for one more warp-wide append)
  int c = 64;
  while (c < k + 32) c <<= 1;
  return c;
}

size_t topk_workspace_bytes(int64_t U, int32_t N, int32_t k) {
  const size_t rows = (size_t)(U < 1 ? 1 : U) * topk_slices(N);
  return align_up(rows * k * sizeof(unsigned long long), 256) + align_up(rows * sizeof(int32_t), 256);
}

__device__ __forceinline__ unsigned long long topk_key(float p, int item) {
  uint32_t b = __float_as_uint(rank_key(p) + 0.0f);
  b = (b & 0x80000000u) ? ~b : (b | 0x80000000u);  // ascending with the float value
  return ((unsigned long long)(~b) << 32) | (uint32_t)item;
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
  // exclusion list: [ep, ee) from the first entry >= lo
  int64_t ep = 0, ee = 0;
  if (a.excl_rowptr != nullptr) {
    const int64_t r = a.excl_ids != nullptr ? (int64_t)__ldg(a.excl_ids + gu) : gu;
    if (r >= 0 && r < a.excl_rows) {
      int64_t b = a.excl_rowptr[r], e = a.excl_rowptr[r + 1];
      ee = e;
      while (b < e) {
        const int64_t mid = (b + e) >> 1;
        if (__ldg(a.excl_items + mid) < lo) b = mid + 1;
        else e = mid;
      }
      ep = b;
    }
  }
  const int t = a.targets != nullptr ? __ldg(a.targets + gu) : -1;
  const bool has_t = (unsigned)t < (unsigned)N;
  const unsigned long long key_t = has_t ? topk_key(__ldg(row + t), t) : 0ull;
  int below = 0, n = 0;
  unsigned long long thr = kNoKey;
  for (int c = lo; c < hi; c += 32) {
    uint32_t xmask = 0;  // excluded items of [c, c + 32)
    for (;;) {           // warp-uniform: lists are sorted, so the entries below c + 32 are a prefix of the lanes
      const int64_t i = ep + lane;
      const int e = i < ee ? __ldg(a.excl_items + i) : INT_MAX;
      const bool in = e < c + 32;
      const int nin = __popc(__ballot_sync(0xffffffffu, in));
      xmask |= __reduce_or_sync(0xffffffffu, (in && e >= c) ? 1u << (e - c) : 0u);
      ep += nin;
      if (nin < 32) break;
    }
    const int item = c + lane;
    const bool cand = item < hi && (!((xmask >> lane) & 1u) || item == t);  // the target is never excluded
    const unsigned long long key = cand ? topk_key(__ldg(row + item), item) : kNoKey;
    below += (has_t && key < key_t) ? 1 : 0;
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
  const unsigned long long* mine = lists + ((size_t)u * S + lane) * k;
  int cur = 0;
  unsigned long long head = lane < S ? mine[0] : kNoKey;
  for (int i = 0; i < k; ++i) {
    unsigned long long m = head;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long x = __shfl_xor_sync(0xffffffffu, m, o);
      m = x < m ? x : m;
    }
    if (m != kNoKey && head == m) {  // keys are distinct: one winner
      ++cur;
      head = cur < k ? mine[cur] : kNoKey;
    }
    if (lane == (i & 31)) {
      const int item = (m == kNoKey || bad_u) ? -1 : (int)(uint32_t)m;
      if (a.top_items != nullptr) a.top_items[gu * k + i] = item;
      if (a.top_scores != nullptr) a.top_scores[gu * k + i] = item < 0 ? nanf("") : __ldg(a.scores + u * N + item);
    }
  }
  if (a.pos != nullptr) {
    int c = lane < S ? counts[u * S + lane] : 0;
    c = warp_sum_int(c);
    const int t = __ldg(a.targets + gu);
    if (lane == 0) a.pos[gu] = (bad_u || (unsigned)t >= (unsigned)N) ? N : c;
  }
}

int launch_topk(const TopkArgs& a, void* ws, cudaStream_t st) {
  if (a.U == 0) return MR_OK;
  const int S = topk_slices(a.N), slice = topk_slice_len(a.N), cap = topk_cap(a.k);
  Carver cv(ws);
  unsigned long long* lists = cv.take<unsigned long long>((size_t)a.U * S * a.k);
  int32_t* counts = cv.take<int32_t>((size_t)a.U * S);
  const int wpc = kTopkThreads / 32;
  const size_t smem = (size_t)wpc * cap * sizeof(unsigned long long);  // <= 16 KB (cap <= 512)
  topk_slice_kernel<<<(unsigned)((a.U * S + wpc - 1) / wpc), kTopkThreads, smem, st>>>(a, S, slice, cap, lists, counts);
  MR_LAUNCH_CHECK("topk_slice_kernel");
  topk_merge_kernel<<<(unsigned)((a.U + wpc - 1) / wpc), kTopkThreads, 0, st>>>(a, S, lists, counts);
  MR_LAUNCH_CHECK("topk_merge_kernel");
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

}  // namespace mr
