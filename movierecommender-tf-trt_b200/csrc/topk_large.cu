// Large-k selection (kTopkSmallK < k <= MR_MAX_TOPK): one CTA per segment -- a row of scores, a ragged list, or an
// audience item's kept list plus its append buffer.  Keys are topk_key's: distinct 64-bit integers, ascending in the
// RankLayer order, so the k smallest are a unique set.  The CTA finds the k-th smallest candidate key by an MSB radix
// select (8-bit digits over the key, integer histograms in shared memory), keeps the candidates at or below it
// (compaction order is irrelevant: the kept set is sorted next), sorts them with a block bitonic sort in shared
// memory (a power of two >= k keys: 32 KB at k = 4096, 48 KB with the audience's 4-byte payload) and writes them.
// The select stops as soon as the boundary bin holds exactly the keys still needed; equal scores fall through to the
// id (or position) bits, which separate every key.  Nothing depends on the order threads meet in: deterministic.
//   rows:      the key pass walks the row next to its exclusion list (per-warp slices, list_mask), stages the keys in
//              the workspace (8 bytes per row: 32 MB per 2^22-row chunk, which stays in L2), counts the candidates
//              below the target's key and builds the first digit's histogram; the radix passes read the staged keys.
//   lists:     keys are recomputed from the scores each pass (key = score bits and position, no exclusion).
//   audiences: per chunk a filter kernel transposes 32 x 32 score tiles (audience_chunk_kernel's reading and
//              exclusion handling) and appends every candidate below its item's threshold (the k-th key of the
//              item's list) to the item's buffer, one warp-aggregated integer atomic per (warp, column, tile); a
//              compaction kernel selects the k best of list + buffer whenever the next chunk could overflow the
//              buffer (cap = k + C, C = users per chunk: about ln(U / k) + 1 compactions per item), and once more
//              after the last chunk, writing the results.
#include "topk_common.cuh"

namespace mr {

constexpr int kLgThreads = 512;
// Rows of at least kLgWideRow items run 1024-thread CTAs: a 2^22-row chunk then has at most 256 rows, too few CTAs to
// fill the GPU, so each CTA's passes need the width (ML-20M: 156 rows of 26,744 per chunk; RANK at k = 1000 drops
// from 163 to 141 ms on a B200).  Shorter rows and lists have CTAs enough, and the wider CTA only adds to each pass.
constexpr int kLgWideThreads = 1024, kLgWideRow = 16384;
constexpr int kLgBits = 8, kLgBins = 1 << kLgBits;
constexpr int kLgAudTargetCtas = 2048;  // filter CTAs per chunk that narrow calls split their row tiles to reach

struct LgState {
  int hist[kLgBins];
  unsigned long long prefix;  // the decided high bits of the k-th smallest candidate key
  int bits;                   // how many high bits are decided
  int need;                   // candidates still needed among those that share the decided bits
  int done;
  int count;                  // candidates of the segment
  int cursor;                 // compaction slots taken
  int below;                  // candidates below the target's key
  int hit;                    // audiences: the target's slot
};

static int lg_cap(int k) {  // sort buffer: a power of two >= k
  int c = 64;
  while (c < k) c <<= 1;
  return c;
}

__device__ void lg_init(LgState& s, int k) {
  for (int i = threadIdx.x; i < kLgBins; i += blockDim.x) s.hist[i] = 0;
  if (threadIdx.x == 0) {
    s.prefix = 0;
    s.bits = 0;
    s.need = k;
    s.done = 0;
    s.count = s.cursor = s.below = 0;
    s.hit = k;
  }
}

// A candidate whose decided high bits equal the prefix's.
__device__ __forceinline__ bool lg_match(unsigned long long key, unsigned long long prefix, int bits) {
  return key != kNoKey && (bits == 0 || (key >> (64 - bits)) == (prefix >> (64 - bits)));
}

// Adds one warp's keys to the histogram of the next digit; lanes with the same bin add once.  Warp-uniform call.
__device__ __forceinline__ void lg_count(int* hist, unsigned long long key, unsigned long long prefix, int bits,
                                         int lane) {
  const bool in = lg_match(key, prefix, bits);
  const int bin = in ? (int)((key >> (64 - kLgBits - bits)) & (kLgBins - 1)) : -1;
  const uint32_t peers = __match_any_sync(0xffffffffu, bin);
  if (in && lane == __ffs(peers) - 1) atomicAdd(hist + bin, __popc(peers));
}

// Warp 0: the bin of the need-th candidate becomes the next digit of the prefix; clears the histogram.  Done when
// the bin holds exactly the candidates still needed, or when all 64 bits are decided: distinct keys always end the
// first way; equal keys (a pool that repeats a user, which the ABI leaves unspecified) end the second, and the
// compaction then keeps k of them.
__device__ void lg_pick(LgState& s, int lane) {
  constexpr int per = kLgBins / 32;
  int c[per], tot = 0;
#pragma unroll
  for (int q = 0; q < per; ++q) {
    c[q] = s.hist[lane * per + q];
    tot += c[q];
  }
  int x = tot;  // inclusive scan over the lanes
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  const int need = s.need;
  __syncwarp();
  if (x - tot < need && need <= x) {  // exactly one lane: need <= the candidates sharing the prefix
    int run = x - tot;
#pragma unroll
    for (int q = 0; q < per; ++q) {
      if (run < need && need <= run + c[q]) {
        s.need = need - run;
        s.prefix |= (unsigned long long)(lane * per + q) << (64 - kLgBits - s.bits);
        s.bits += kLgBits;
        s.done = c[q] == need - run || s.bits == 64;
      }
      run += c[q];
    }
  }
#pragma unroll
  for (int q = 0; q < per; ++q) s.hist[lane * per + q] = 0;
}

// One warp step of the first pass over a segment: counts the candidates, adds them to the first digit's histogram.
__device__ __forceinline__ void lg_first(LgState& s, unsigned long long key, int lane) {
  lg_count(s.hist, key, 0ull, 0, lane);
  const int n = __popc(__ballot_sync(0xffffffffu, key != kNoKey));
  if (lane == 0 && n > 0) atomicAdd(&s.count, n);
}

// The k smallest candidates of key_at(0 .. n) (kNoKey: not a candidate), after a first pass (lg_first) and a
// __syncthreads.  keep(slot, i, key) runs once for each of them, slots 0 .. m - 1 in no particular order; returns
// m = min(k, candidates).  At most 8 radix passes; keep never sees a slot >= k, even when equal keys tie at the k-th
// place.  Block-uniform call; ends with a __syncthreads.
template <class KeyAt, class Keep>
__device__ int lg_select(LgState& s, int64_t n, int k, KeyAt key_at, Keep keep) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int count = s.count;
  if (count > k) {
    for (;;) {
      if (warp == 0) lg_pick(s, lane);
      __syncthreads();
      if (s.done) break;
      const unsigned long long prefix = s.prefix;
      const int bits = s.bits;
      for (int64_t base = (int64_t)warp * 32; base < n; base += blockDim.x) {
        const int64_t i = base + lane;
        lg_count(s.hist, i < n ? key_at(i) : kNoKey, prefix, bits, lane);
      }
      __syncthreads();
    }
  }
  const unsigned long long prefix = s.prefix;  // count <= k: bits = 0, every candidate is kept
  const int bits = s.bits;
  for (int64_t base = (int64_t)warp * 32; base < n; base += blockDim.x) {
    const int64_t i = base + lane;
    const unsigned long long key = i < n ? key_at(i) : kNoKey;
    const bool in = key != kNoKey && (bits == 0 || (key >> (64 - bits)) <= (prefix >> (64 - bits)));
    const uint32_t pm = __ballot_sync(0xffffffffu, in);
    if (pm == 0) continue;
    int slot = 0;
    if (lane == 0) slot = atomicAdd(&s.cursor, __popc(pm));
    slot = __shfl_sync(0xffffffffu, slot, 0) + __popc(pm & ((1u << lane) - 1u));
    if (in && slot < k) keep(slot, i, key);
  }
  __syncthreads();
  return count < k ? count : k;
}

// Pads keys[m, cap) with kNoKey and sorts keys[0, cap) ascending, carrying vals when VALS: the network spans the
// smallest power of two >= m, since the padding beyond it is already in order.
template <bool VALS>
__device__ void lg_sort(unsigned long long* keys, int* vals, int m, int cap) {
  for (int i = m + threadIdx.x; i < cap; i += blockDim.x) keys[i] = kNoKey;
  __syncthreads();
  int span = 1;
  while (span < m) span <<= 1;
  for (int size = 2; size <= span; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = threadIdx.x; i < span / 2; i += blockDim.x) {
        const int x0 = 2 * i - (i & (stride - 1)), x1 = x0 + stride;
        const unsigned long long x = keys[x0], y = keys[x1];
        if ((x > y) == ((x0 & size) == 0)) {
          keys[x0] = y;
          keys[x1] = x;
          if (VALS) {
            const int t = vals[x0];
            vals[x0] = vals[x1];
            vals[x1] = t;
          }
        }
      }
      __syncthreads();
    }
  }
}

// ---- rows --------------------------------------------------------------------------------------------------------
// SKIP_SELF: the row's own id a.users[gu] is never a candidate (similar items / users).  Launched with kLgThreads or
// kLgWideThreads threads.
template <bool SKIP_SELF>
__global__ void __launch_bounds__(kLgWideThreads) topk_large_rows_kernel(const TopkArgs a, int cap,
                                                                     unsigned long long* __restrict__ stage) {
  extern __shared__ unsigned long long lg_keys[];
  __shared__ LgState s;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t u = blockIdx.x, gu = a.u0 + u;
  const int N = a.N, k = a.k;
  const float* row = a.scores + u * N;
  const bool bad_u = a.users != nullptr && (unsigned)__ldg(a.users + gu) >= (unsigned)a.num_users;
  const int t = a.targets != nullptr ? __ldg(a.targets + gu) : -1;
  const bool has_t = (unsigned)t < (unsigned)N;
  lg_init(s, k);
  __syncthreads();
  if (!bad_u) {  // block-uniform
    unsigned long long* keys = stage + u * N;
    const unsigned long long key_t = has_t ? topk_key(__ldg(row + t), t) : 0ull;
    const int nw = blockDim.x / 32;
    const int slice = (int)(((int64_t)N + nw - 1) / nw + 31) / 32 * 32;
    const int lo = (int)min((int64_t)warp * slice, (int64_t)N), hi = (int)min((int64_t)lo + slice, (int64_t)N);
    int64_t ep, ee;
    excl_cursor(a.excl_ids, a.excl_rows, a.excl_rowptr, a.excl_items, gu, lo, ep, ee);
    const int self = SKIP_SELF ? __ldg(a.users + gu) : -1;
    int below = 0;
    for (int c = lo; c < hi; c += 32) {
      const uint32_t xmask = list_mask(a.excl_items, ep, ee, c, lane);
      const int item = c + lane;
      const bool cand = item < hi && (!((xmask >> lane) & 1u) || item == t) &&  // the target is never excluded
                        (!SKIP_SELF || item != self);
      const unsigned long long key = cand ? topk_key(__ldg(row + item), item) : kNoKey;
      if (item < hi) keys[item] = key;
      below += (has_t && key < key_t) ? 1 : 0;
      lg_first(s, key, lane);
    }
    below = warp_sum_int(below);
    if (lane == 0 && below > 0) atomicAdd(&s.below, below);
    __syncthreads();
    const int m = lg_select(s, N, k, [&](int64_t i) { return keys[i]; },
                            [&](int slot, int64_t, unsigned long long key) { lg_keys[slot] = key; });
    lg_sort<false>(lg_keys, nullptr, m, cap);
  }
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    const unsigned long long m = bad_u ? kNoKey : lg_keys[i];
    const int item = m == kNoKey ? -1 : (int)(uint32_t)m;
    if (a.top_items != nullptr) a.top_items[gu * k + i] = item;
    if (a.top_scores != nullptr) a.top_scores[gu * k + i] = item < 0 ? nanf("") : __ldg(row + item);
  }
  if (a.pos != nullptr && threadIdx.x == 0) a.pos[gu] = (bad_u || !has_t) ? N : s.below;
}

size_t topk_large_workspace_bytes(int64_t U, int32_t N) {
  return align_up((size_t)(U < 1 ? 1 : U) * N * sizeof(unsigned long long), 256);
}

int launch_topk_large(const TopkArgs& a, void* ws, cudaStream_t st, bool skip_self) {
  const int cap = lg_cap(a.k);
  const int threads = a.N >= kLgWideRow ? kLgWideThreads : kLgThreads;
  const size_t smem = (size_t)cap * sizeof(unsigned long long);
  unsigned long long* stage = static_cast<unsigned long long*>(ws);
  if (skip_self) topk_large_rows_kernel<true><<<(unsigned)a.U, threads, smem, st>>>(a, cap, stage);
  else topk_large_rows_kernel<false><<<(unsigned)a.U, threads, smem, st>>>(a, cap, stage);
  MR_LAUNCH_CHECK("topk_large_rows_kernel");
  return MR_OK;
}

// ---- ragged lists ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kLgThreads) topk_large_lists_kernel(const TopkListsArgs a, int cap,
                                                                      int32_t* __restrict__ pos) {
  extern __shared__ unsigned long long lg_keys[];
  __shared__ LgState s;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t u = blockIdx.x;
  int64_t b, e;
  list_bounds(a.rowptr, u, a.nnz, b, e);
  const int len = (int)(e - b), k = a.k;
  const float* sc = a.scores + b;
  const bool bad_u = a.users != nullptr && (unsigned)__ldg(a.users + u) >= (unsigned)a.num_users;
  const int t = a.targets != nullptr ? __ldg(a.targets + u) : -1;
  const bool has_t = (unsigned)t < (unsigned)len;
  lg_init(s, k);
  __syncthreads();
  if (!bad_u) {  // block-uniform
    const unsigned long long key_t = has_t ? topk_key(__ldg(sc + t), t) : 0ull;
    auto key_at = [&](int64_t i) { return topk_key(__ldg(sc + i), (int)i); };
    int below = 0;
    for (int base = warp * 32; base < len; base += blockDim.x) {
      const int j = base + lane;
      const unsigned long long key = j < len ? key_at(j) : kNoKey;
      below += (has_t && key < key_t) ? 1 : 0;
      if (len > k) lg_first(s, key, lane);
    }
    below = warp_sum_int(below);
    if (lane == 0 && below > 0) atomicAdd(&s.below, below);
    if (threadIdx.x == 0 && len <= k) s.count = len;  // a list no longer than k is simply sorted
    __syncthreads();
    const int m = lg_select(s, len, k, key_at, [&](int slot, int64_t, unsigned long long key) { lg_keys[slot] = key; });
    lg_sort<false>(lg_keys, nullptr, m, cap);
  }
  for (int i = threadIdx.x; i < k; i += blockDim.x) lists_emit(a, u, b, i, bad_u ? kNoKey : lg_keys[i], bad_u);
  if (pos != nullptr && threadIdx.x == 0) pos[u] = (bad_u || !has_t) ? len : s.below;
}

int launch_topk_lists_large(const TopkListsArgs& a, int32_t* pos, cudaStream_t st) {
  if (a.U == 0) return MR_OK;
  const int cap = lg_cap(a.k);
  topk_large_lists_kernel<<<(unsigned)a.U, kLgThreads, (size_t)cap * sizeof(unsigned long long), st>>>(a, cap, pos);
  MR_LAUNCH_CHECK("topk_large_lists_kernel");
  return MR_OK;
}

// ---- audiences ---------------------------------------------------------------------------------------------------
AudienceLargeWs carve_audience_large(void* ws, int64_t C, int32_t M, int32_t k, size_t& total) {
  AudienceLargeWs w{};
  Carver cv(ws);
  const size_t items = (size_t)(M < 1 ? 1 : M);
  w.cap = k + (C < 1 ? 1 : C);
  w.keys = cv.take<unsigned long long>(items * k);
  w.scores = cv.take<float>(items * k);
  w.bkeys = cv.take<unsigned long long>(items * w.cap);
  w.bscores = cv.take<float>(items * w.cap);
  w.cnt = cv.take<int32_t>(items);
  w.pos = cv.take<int32_t>(items);
  total = cv.off;
  return w;
}

// Per chunk: one CTA per (32 columns, strided group of 32-row tiles); each warp walks 4 columns of every tile, the
// lanes being 32 users, and appends the candidates below the column's threshold to its buffer.
template <bool POOL>
__global__ void __launch_bounds__(256) audience_large_filter_kernel(const AudienceArgs a, const AudienceLargeWs w) {
  constexpr int kCols = 32, kColsPerWarp = kCols / 8;
  __shared__ float tile[32][33];
  __shared__ int ids[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int k = a.k, M = a.M;
  const int64_t C = a.U, first = (int64_t)blockIdx.y * 32, step = (int64_t)32 * gridDim.y;
  if (first >= C) return;  // block-uniform
  const int j0 = blockIdx.x * kCols;
  const int lo_user = POOL ? __ldg(a.users + a.u0 + first) : (int)(a.u0 + first);
  int t[kColsPerWarp];
  unsigned long long thr[kColsPerWarp];
  int64_t ep[kColsPerWarp], ee[kColsPerWarp];
#pragma unroll
  for (int q = 0; q < kColsPerWarp; ++q) {
    const int j = j0 + warp * kColsPerWarp + q;
    t[q] = -1;
    thr[q] = kNoKey;
    ep[q] = ee[q] = 0;
    if (j < M) {
      thr[q] = w.keys[(size_t)j * k + k - 1];
      excl_cursor(a.excl_ids, a.excl_rows, a.excl_rowptr, a.excl_users, j, lo_user, ep[q], ee[q]);
      if (a.targets != nullptr) t[q] = __ldg(a.targets + j);
    }
  }
  for (int64_t r0 = first; r0 < C; r0 += step) {
    const int col = j0 + lane;
    for (int rr = warp; rr < 32; rr += 8) {
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
    for (int q = 0; q < kColsPerWarp; ++q) {
      const int c = warp * kColsPerWarp + q, j = j0 + c;
      if (j >= M) break;  // warp-uniform
      const uint32_t x = POOL ? ids_mask(a.excl_users, ep[q], ee[q], ids, lane)
                              : list_mask(a.excl_users, ep[q], ee[q], (int)(a.u0 + r0), lane);
      const bool cand = ok && (!((x >> lane) & 1u) || uid == t[q]);  // the target is never excluded
      const float p = tile[lane][c];
      const unsigned long long key = cand ? topk_key(p, uid) : kNoKey;
      const bool pass = key < thr[q];
      const uint32_t pm = __ballot_sync(0xffffffffu, pass);
      if (pm == 0) continue;
      int slot = 0;
      if (lane == 0) slot = atomicAdd(w.cnt + j, __popc(pm));
      slot = __shfl_sync(0xffffffffu, slot, 0) + __popc(pm & ((1u << lane) - 1u));
      if (pass) {
        w.bkeys[(size_t)j * w.cap + slot] = key;
        w.bscores[(size_t)j * w.cap + slot] = p;
      }
    }
    __syncthreads();
  }
}

// Persistent CTAs over the items: the k best of an item's list + buffer become its list (FINAL: its results).  Not
// FINAL, an item is compacted only when a chunk of `next` rows could overflow its buffer.
template <bool FINAL>
__global__ void __launch_bounds__(kLgThreads) audience_large_compact_kernel(const AudienceArgs a, const AudienceLargeWs w,
                                                                           int cap, int64_t next,
                                                                           const int32_t* __restrict__ items,
                                                                           int32_t num_items, int32_t* __restrict__ top_users,
                                                                           float* __restrict__ top_scores,
                                                                           int32_t* __restrict__ pos) {
  extern __shared__ unsigned long long lg_keys[];
  __shared__ LgState s;
  int* vals = reinterpret_cast<int*>(lg_keys + cap);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int k = a.k;
  for (int64_t j = blockIdx.x; j < a.M; j += gridDim.x) {
    const int nb = w.cnt[j];
    if (!FINAL && nb + next <= w.cap) continue;  // block-uniform
    const unsigned long long* lk = w.keys + (size_t)j * k;
    const unsigned long long* bk = w.bkeys + (size_t)j * w.cap;
    const float* ls = w.scores + (size_t)j * k;
    const float* bs = w.bscores + (size_t)j * w.cap;
    const int64_t n = (int64_t)k + nb;
    auto key_at = [&](int64_t i) { return i < k ? lk[i] : bk[i - k]; };
    __syncthreads();  // the previous item is done with s and the buffers
    lg_init(s, k);
    __syncthreads();
    for (int64_t base = (int64_t)warp * 32; base < n; base += blockDim.x) {
      const int64_t i = base + lane;
      lg_first(s, i < n ? key_at(i) : kNoKey, lane);
    }
    __syncthreads();
    const int m = lg_select(s, n, k, key_at, [&](int slot, int64_t i, unsigned long long key) {
      lg_keys[slot] = key;
      vals[slot] = (int)i;
    });
    lg_sort<true>(lg_keys, vals, m, cap);
    for (int i = threadIdx.x; i < m; i += blockDim.x) {  // the source slot becomes the raw score
      const int v = vals[i];
      vals[i] = __float_as_int(v < k ? ls[v] : bs[v - k]);
    }
    __syncthreads();  // every old score is read
    if (FINAL) {
      const bool bad = items != nullptr && (unsigned)__ldg(items + j) >= (unsigned)num_items;
      const int tj = a.targets != nullptr ? __ldg(a.targets + j) : -1;
      for (int i = threadIdx.x; i < k; i += blockDim.x) {
        const int user = (i >= m || bad) ? -1 : (int)(uint32_t)lg_keys[i];
        if (top_users != nullptr) top_users[j * k + i] = user;
        if (top_scores != nullptr) top_scores[j * k + i] = user < 0 ? nanf("") : __int_as_float(vals[i]);
        if (user >= 0 && user == tj) s.hit = i;  // distinct users: one slot at most
      }
      __syncthreads();
      if (pos != nullptr && threadIdx.x == 0) pos[j] = s.hit;
    } else {
      unsigned long long* lkw = w.keys + (size_t)j * k;
      float* lsw = w.scores + (size_t)j * k;
      for (int i = threadIdx.x; i < k; i += blockDim.x) {
        lkw[i] = lg_keys[i];
        lsw[i] = i < m ? __int_as_float(vals[i]) : 0.f;
      }
      if (threadIdx.x == 0) w.cnt[j] = 0;
    }
  }
}

static unsigned audience_large_ctas(int32_t M) {
  const int64_t g = (int64_t)sm_count() * 4;
  return (unsigned)(M < g ? M : g);
}

static size_t audience_large_smem(int k) { return (size_t)lg_cap(k) * (sizeof(unsigned long long) + sizeof(int)); }

int launch_audience_large_init(const AudienceArgs& a, const AudienceLargeWs& w, cudaStream_t st) {
  MR_CUDA(cudaMemsetAsync(w.keys, 0xff, (size_t)a.M * a.k * sizeof(unsigned long long), st));
  MR_CUDA(cudaMemsetAsync(w.cnt, 0, (size_t)a.M * sizeof(int32_t), st));
  const int smem = (int)audience_large_smem(a.k);  // <= 48 KB
  MR_CUDA(cudaFuncSetAttribute(audience_large_compact_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  MR_CUDA(cudaFuncSetAttribute(audience_large_compact_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  return MR_OK;
}

int launch_audience_large_chunk(const AudienceArgs& a, const AudienceLargeWs& w, cudaStream_t st) {
  const int cap = lg_cap(a.k);
  if (a.u0 + a.U > w.cap) {  // before that no buffer can hold more than u0 entries
    audience_large_compact_kernel<false><<<audience_large_ctas(a.M), kLgThreads, audience_large_smem(a.k), st>>>(
        a, w, cap, a.U, nullptr, 0, nullptr, nullptr, nullptr);
    MR_LAUNCH_CHECK("audience_large_compact_kernel");
  }
  const int64_t blocks = ((int64_t)a.M + 31) / 32, tiles = (a.U + 31) / 32;
  int64_t y = (kLgAudTargetCtas + blocks - 1) / blocks;
  if (y > tiles) y = tiles;
  const dim3 grid((unsigned)blocks, (unsigned)(y < 1 ? 1 : y));
  if (a.users != nullptr) audience_large_filter_kernel<true><<<grid, 256, 0, st>>>(a, w);
  else audience_large_filter_kernel<false><<<grid, 256, 0, st>>>(a, w);
  MR_LAUNCH_CHECK("audience_large_filter_kernel");
  return MR_OK;
}

int launch_audience_large_final(const AudienceArgs& a, const AudienceLargeWs& w, const int32_t* items,
                                int32_t num_items, int32_t* top_users, float* top_scores, int32_t* pos, cudaStream_t st) {
  audience_large_compact_kernel<true><<<audience_large_ctas(a.M), kLgThreads, audience_large_smem(a.k), st>>>(
      a, w, lg_cap(a.k), 0, items, num_items, top_users, top_scores, pos);
  MR_LAUNCH_CHECK("audience_large_compact_kernel");
  return MR_OK;
}

}  // namespace mr
