// Stable LSD radix sort of (row id, sample index) pairs -- the "sort" of the deterministic
// sort-and-segmented-reduce embedding-gradient path.  8-bit digits; only ceil(key_bits/8) passes run
// (ids are <= num_users / num_items once out-of-range ids are mapped to that sentinel, so 2-3 passes).  Each warp owns a contiguous tile of kKeysPerWarp
// keys and walks it 32 keys at a time in order, ranking equal digits with __match_any_sync, so the
// sort is stable without any block-level synchronisation and without atomics.
#include "launchers.h"

namespace mr {

// Keys per warp tile.  A warp walks its tile 32 keys at a time IN ORDER (that is what makes the sort stable), so
// the tile length is the serial depth of the kernel: at 2048 keys a launch took ~50 us however few keys there
// were (64 dependent iterations, 4 warps per SM at 1.3 M keys).  256 keys = 8 iterations whose loads are all
// issued up front.
constexpr int kKeysPerWarp = 256;
constexpr int kTileIters = kKeysPerWarp / 32;
constexpr int kSortWarps = 4;  // warps per CTA
constexpr int kBins = 256;

__device__ __forceinline__ unsigned digit_of(int32_t key, int shift) { return ((unsigned)key >> shift) & 0xFFu; }

// Key as the sort sees it: keys above `sentinel` (unsigned compare, so negative keys too) become `sentinel`.
// 0xFFFFFFFF leaves every key as it is.
__device__ __forceinline__ int32_t load_key(const int32_t* keys, int64_t i, unsigned sentinel) {
  return (int32_t)min((unsigned)__ldg(keys + i), sentinel);
}

// hist[bin * nwt + wt] = number of keys of warp tile `wt` whose digit is `bin`.
__global__ void __launch_bounds__(kSortWarps * 32) radix_hist_kernel(const int32_t* __restrict__ keys, int64_t n,
                                                                     int shift, unsigned sentinel,
                                                                     unsigned* __restrict__ hist, int64_t nwt) {
  __shared__ unsigned cnt[kSortWarps][kBins];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t wt = (int64_t)blockIdx.x * kSortWarps + w;
  for (int b = lane; b < kBins; b += 32) cnt[w][b] = 0;
  __syncwarp();
  if (wt < nwt) {
    const int64_t base = wt * kKeysPerWarp;
    int32_t kreg[kTileIters];
#pragma unroll
    for (int q = 0; q < kTileIters; ++q) {
      const int64_t i = base + 32 * q + lane;
      kreg[q] = i < n ? load_key(keys, i, sentinel) : 0;
    }
#pragma unroll
    for (int q = 0; q < kTileIters; ++q) {
      const int64_t i = base + 32 * q + lane;
      const bool valid = i < n;
      const unsigned d = valid ? digit_of(kreg[q], shift) : (0x100u | lane);
      const unsigned peers = __match_any_sync(0xffffffffu, d);
      if (valid && (peers & ((1u << lane) - 1)) == 0) cnt[w][d] += __popc(peers);
      __syncwarp();
    }
    for (int b = lane; b < kBins; b += 32) hist[(size_t)b * nwt + wt] = cnt[w][b];
  }
}

// Per-digit exclusive scan over the warp tiles: CTA `bin` scans row hist[bin][0..nwt) in place and
// writes the row total.  256 CTAs run in parallel (a single-CTA scan of the whole matrix cost 0.31 ms
// per pass at 1.3 M keys); the 256 digit bases are folded into the scatter kernel.
__global__ void __launch_bounds__(256) radix_rowscan_kernel(unsigned* __restrict__ hist, int64_t nwt,
                                                            unsigned* __restrict__ totals) {
  __shared__ unsigned warp_tot[8];
  __shared__ unsigned carry;
  unsigned* row = hist + (size_t)blockIdx.x * nwt;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  if (tid == 0) carry = 0;
  __syncthreads();
  for (int64_t t0 = 0; t0 < nwt; t0 += 256) {
    const int64_t i = t0 + tid;
    const unsigned v = i < nwt ? row[i] : 0u;
    unsigned incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) warp_tot[w] = incl;
    __syncthreads();
    unsigned before = carry;
    for (int q = 0; q < w; ++q) before += warp_tot[q];
    if (i < nwt) row[i] = before + incl - v;
    __syncthreads();
    if (tid == 255) carry = before + incl;
    __syncthreads();
  }
  if (tid == 0) totals[blockIdx.x] = carry;
}

// Scatter pass: keys (and their payload index) move to their stable position for this digit.
__global__ void __launch_bounds__(kSortWarps * 32) radix_scatter_kernel(
    const int32_t* __restrict__ keys, const int32_t* __restrict__ index /* null = identity */, int64_t n, int shift,
    unsigned sentinel, const unsigned* __restrict__ hist, const unsigned* __restrict__ totals, int64_t nwt,
    int32_t* __restrict__ out_keys, int32_t* __restrict__ out_index) {
  __shared__ unsigned run[kSortWarps][kBins];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t wt = (int64_t)blockIdx.x * kSortWarps + w;
  if (wt >= nwt) return;
  {
    // digit bases: exclusive scan of the 256 row totals, 8 consecutive digits per lane
    unsigned t[8], s8 = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      t[q] = __ldg(totals + lane * 8 + q);
      s8 += t[q];
    }
    unsigned incl = s8;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned x = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += x;
    }
    unsigned basev = incl - s8;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int b = lane * 8 + q;
      run[w][b] = basev + hist[(size_t)b * nwt + wt];
      basev += t[q];
    }
  }
  __syncwarp();
  const int64_t base = wt * kKeysPerWarp;
  int32_t kreg[kTileIters], vreg[kTileIters];
#pragma unroll
  for (int q = 0; q < kTileIters; ++q) {
    const int64_t i = base + 32 * q + lane;
    kreg[q] = i < n ? load_key(keys, i, sentinel) : 0;
    vreg[q] = i < n ? (index != nullptr ? __ldg(index + i) : (int32_t)i) : 0;
  }
#pragma unroll
  for (int q = 0; q < kTileIters; ++q) {
    const int64_t i = base + 32 * q + lane;
    if (base + 32 * q >= n) break;  // warp-uniform
    const bool valid = i < n;
    const int32_t key = kreg[q];
    const int32_t val = vreg[q];
    const unsigned d = valid ? digit_of(key, shift) : (0x100u | lane);
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const int rank = __popc(peers & ((1u << lane) - 1));
    unsigned pos = 0;
    if (valid) pos = run[w][d] + rank;
    __syncwarp();
    if (valid && rank == 0) run[w][d] += __popc(peers);
    __syncwarp();
    if (valid) {
      out_keys[pos] = key;
      out_index[pos] = val;
    }
  }
}

static int64_t num_warp_tiles(int64_t n) { return (n + kKeysPerWarp - 1) / kKeysPerWarp; }

size_t sort_workspace_bytes(int64_t n) {
  const int64_t nwt = num_warp_tiles(n < 1 ? 1 : n);
  return align_up((size_t)n * 4, 256) * 2 + align_up((size_t)kBins * nwt * 4, 256) + align_up(kBins * 4, 256) + 256;
}

int launch_sort_pairs(const int32_t* keys, int64_t n, int key_bits, int32_t* out_keys, int32_t* out_index,
                      void* ws, size_t ws_bytes, cudaStream_t st, int32_t num_rows) {
  if (n == 0) return MR_OK;
  if (ws_bytes < sort_workspace_bytes(n)) {
    set_error("sort workspace too small: %zu < %zu", ws_bytes, sort_workspace_bytes(n));
    return MR_ERR_WORKSPACE;
  }
  if (n >= (int64_t)1 << 31) {
    set_error("sort: n must be < 2^31");
    return MR_ERR_INVALID;
  }
  const int64_t nwt = num_warp_tiles(n);
  Carver cv(ws);
  int32_t* tmp_keys = cv.take<int32_t>(n);
  int32_t* tmp_index = cv.take<int32_t>(n);
  unsigned* hist = cv.take<unsigned>(kBins * nwt);
  unsigned* totals = cv.take<unsigned>(kBins);
  int passes = (key_bits + 7) / 8;
  if (passes < 1) passes = 1;
  if (passes > 4) passes = 4;
  const unsigned blocks = (unsigned)((nwt + kSortWarps - 1) / kSortWarps);
  const int32_t* src_k = keys;
  const int32_t* src_i = nullptr;
  for (int p = 0; p < passes; ++p) {
    const bool to_out = ((passes - 1 - p) & 1) == 0;
    int32_t* dst_k = to_out ? out_keys : tmp_keys;
    int32_t* dst_i = to_out ? out_index : tmp_index;
    // the first pass maps out-of-range keys to the sentinel and stores them so; later passes read mapped keys
    const unsigned sentinel = (p == 0 && num_rows >= 0) ? (unsigned)num_rows : 0xFFFFFFFFu;
    radix_hist_kernel<<<blocks, kSortWarps * 32, 0, st>>>(src_k, n, 8 * p, sentinel, hist, nwt);
    MR_LAUNCH_CHECK("radix_hist_kernel");
    radix_rowscan_kernel<<<kBins, 256, 0, st>>>(hist, nwt, totals);
    MR_LAUNCH_CHECK("radix_rowscan_kernel");
    radix_scatter_kernel<<<blocks, kSortWarps * 32, 0, st>>>(src_k, src_i, n, 8 * p, sentinel, hist, totals, nwt, dst_k,
                                                             dst_i);
    MR_LAUNCH_CHECK("radix_scatter_kernel");
    src_k = dst_k;
    src_i = dst_i;
  }
  return MR_OK;
}

}  // namespace mr
