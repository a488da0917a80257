// Deterministic segmented reduction of staged per-sample embedding-row gradients, fused with the
// row update -- the "segmented-reduce scatter-add, with no atomics, feeding a fused sparse-row Adam
// update" of the train step.  Input: sample indices stably sorted by row id (radix_sort.cu), so the
// samples of one row are contiguous and in batch order.
//
// Load-balanced by recursive chunking.  Level 0: every warp owns exactly 32 consecutive sorted
// entries, sums each run of equal row ids inside its chunk (entries added in order), and
//   * applies the row update at once when the run neither continues from the previous chunk nor
//     into the next one (the whole segment is inside the chunk), or
//   * emits a partial sum into one of the chunk's two output slots (slot 0: the run that continues
//     from the previous chunk, slot 1: the run that continues into the next one).
// The emitted (row id, partial row) list is again a sequence in which equal ids are contiguous, 16x
// shorter, and the same kernel reduces it (now reading rows directly); after log32(n) levels one chunk
// is left and everything has been applied.  Popular rows (MovieLens item popularity is Zipf-like: one
// item can own 10^4..10^5 samples of a batch) therefore cost a balanced tree instead of one warp's
// serial loop, and the summation tree depends only on positions -> bit-identical on every run.
// Unused slots carry the key kSkip; a chunk that is one single continuing run emits (id, sum) and
// (id, zeros) so that equal ids stay contiguous across chunk boundaries.
//
// GMF-recompute form of level 0 (the fused train kernel's item side): the staged rows hold only the d0 columns of
// dZ1, and columns [d0, d0 + d1) of an entry -- the GMF item gradient (dz * w_out[c]) * gmf_u[user][c] -- are formed
// here from the row's dz and its user's GMF row, with the same two roundings as the staging they replace, so the sums
// are bit for bit those of the staged layout.  The d1 columns cost 4 B of dz per row plus a gather of the user's GMF
// row (a 35 MB table at the ML-20M shape) instead of 256 B written by the fused kernel and read back here.
#include "launchers.h"

namespace mr {

constexpr int kSkip = -1;     // empty slot
constexpr int kPastEnd = -2;  // lane beyond n
constexpr int kNoNeighbour = -3;
constexpr int kBatch = 8;     // rows loaded per lane before they are added (level 0: thousands of chunks in flight)
constexpr int kBatchUpper = 16;  // upper levels: few chunks, so a chunk's own latency is the launch's duration --
                                 // deeper batches and one warp per 128-column slab (gridDim.y) cut its serial
                                 // load rounds from 8 to 2 (ncu: every upper-level launch took 20-25 us)

__device__ __forceinline__ void apply_row_value(const RowUpdate& u, int row, int c, float g) {
  float *p, *m, *v, *gt;
  int d, col;
  if (c < u.d0) {
    p = u.p0; m = u.m0; v = u.v0; gt = u.g0; d = u.d0; col = c;
  } else {
    p = u.p1; m = u.m1; v = u.v1; gt = u.g1; d = u.d1; col = c - u.d0;
  }
  const size_t at = (size_t)row * d + col;
  if (u.mode == MR_TABLES_DENSE) {
    gt[at] = g;  // the dense Adam sweep (optimizer.cu) consumes the gradient table
  } else if (u.optimizer == MR_OPT_ADAM) {
    const float mn = u.beta_1 * m[at] + (1.f - u.beta_1) * g;
    const float vn = u.beta_2 * v[at] + (1.f - u.beta_2) * g * g;
    m[at] = mn;
    v[at] = vn;
    p[at] = p[at] - u.lr_t * mn / (sqrtf(vn) + u.epsilon);
  } else {
    p[at] = p[at] - u.lr * g;
  }
}

// Four consecutive columns c..c+3 of one table (the vector path guarantees d0 % 4 == 0 and c % 4 == 0, so the
// four never straddle the two tables): 128-bit accesses instead of four scalar read-modify-writes per lane.
__device__ __forceinline__ void apply_row_value4(const RowUpdate& u, int row, int c, float4 g) {
  float *p, *m, *v, *gt;
  int d, col;
  if (c < u.d0) {
    p = u.p0; m = u.m0; v = u.v0; gt = u.g0; d = u.d0; col = c;
  } else {
    p = u.p1; m = u.m1; v = u.v1; gt = u.g1; d = u.d1; col = c - u.d0;
  }
  const size_t at = (size_t)row * d + col;
  if ((d & 3) != 0) {  // rows of this table are not 16-byte aligned: scalar path
    apply_row_value(u, row, c, g.x);
    apply_row_value(u, row, c + 1, g.y);
    apply_row_value(u, row, c + 2, g.z);
    apply_row_value(u, row, c + 3, g.w);
    return;
  }
  if (u.mode == MR_TABLES_DENSE) {
    *reinterpret_cast<float4*>(gt + at) = g;
  } else if (u.optimizer == MR_OPT_ADAM) {
    const float4 m0 = *reinterpret_cast<const float4*>(m + at), v0 = *reinterpret_cast<const float4*>(v + at);
    float4 pw = *reinterpret_cast<const float4*>(p + at);
    float4 mn, vn;
    mn.x = u.beta_1 * m0.x + (1.f - u.beta_1) * g.x; vn.x = u.beta_2 * v0.x + (1.f - u.beta_2) * g.x * g.x;
    mn.y = u.beta_1 * m0.y + (1.f - u.beta_1) * g.y; vn.y = u.beta_2 * v0.y + (1.f - u.beta_2) * g.y * g.y;
    mn.z = u.beta_1 * m0.z + (1.f - u.beta_1) * g.z; vn.z = u.beta_2 * v0.z + (1.f - u.beta_2) * g.z * g.z;
    mn.w = u.beta_1 * m0.w + (1.f - u.beta_1) * g.w; vn.w = u.beta_2 * v0.w + (1.f - u.beta_2) * g.w * g.w;
    pw.x = pw.x - u.lr_t * mn.x / (sqrtf(vn.x) + u.epsilon);
    pw.y = pw.y - u.lr_t * mn.y / (sqrtf(vn.y) + u.epsilon);
    pw.z = pw.z - u.lr_t * mn.z / (sqrtf(vn.z) + u.epsilon);
    pw.w = pw.w - u.lr_t * mn.w / (sqrtf(vn.w) + u.epsilon);
    *reinterpret_cast<float4*>(m + at) = mn;
    *reinterpret_cast<float4*>(v + at) = vn;
    *reinterpret_cast<float4*>(p + at) = pw;
  } else {
    float4 pw = *reinterpret_cast<const float4*>(p + at);
    pw.x -= u.lr * g.x; pw.y -= u.lr * g.y; pw.z -= u.lr * g.z; pw.w -= u.lr * g.w;
    *reinterpret_cast<float4*>(p + at) = pw;
  }
}

struct ChunkInfo {
  int nvalid;       // entries of the chunk that exist
  bool first_inc;   // run starting at entry 0 continues from the previous chunk
  bool last_inc;    // run ending at the last entry continues into the next chunk
  int64_t chunk;
  int ld;
  float* out_rows;
};

// A run [s, t) of row id `key` has been summed into acc (VEC: 4 columns c..c+3, else 1 column c).  DENSE: u.mode is
// MR_TABLES_DENSE (the row is written into the gradient table; no optimizer code in the kernel).
template <bool VEC, bool DENSE = false>
__device__ __forceinline__ void flush_run(const RowUpdate& u, const ChunkInfo& ci, int key, int s, int t, int c,
                                          bool on, float4 acc) {
  if (key == kSkip || !on || (unsigned)key >= (unsigned)u.num_rows) return;
  const bool inc_first = (s == 0) && ci.first_inc;
  const bool inc_last = (t == ci.nvalid) && ci.last_inc;
  if (!inc_first && !inc_last) {
    if (DENSE) {
      const bool t0 = c < u.d0;
      *reinterpret_cast<float4*>((t0 ? u.g0 : u.g1) + (size_t)key * (t0 ? u.d0 : u.d1) + (t0 ? c : c - u.d0)) = acc;
    } else if (VEC) {
      apply_row_value4(u, key, c, acc);
    } else {
      apply_row_value(u, key, c, acc.x);
    }
    return;
  }
  float* slot0 = ci.out_rows + (size_t)(2 * ci.chunk) * ci.ld + c;
  float* slot1 = slot0 + ci.ld;
  if (VEC) {
    if (inc_first) {
      *reinterpret_cast<float4*>(slot0) = acc;
      if (inc_last) *reinterpret_cast<float4*>(slot1) = make_float4(0.f, 0.f, 0.f, 0.f);
    } else {
      *reinterpret_cast<float4*>(slot1) = acc;
    }
  } else {
    if (inc_first) {
      *slot0 = acc.x;
      if (inc_last) *slot1 = 0.f;
    } else {
      *slot1 = acc.x;
    }
  }
}

// keys[n]; INDIRECT: row of entry e is rows[index[e]], else rows[e].  out_keys/out_rows hold two slots
// per chunk (may be NULL when there is a single chunk: then nothing can be incomplete).  GMF (level 0, VEC only):
// rows are d0 wide and columns [d0, ld) are formed from g (see the top of this file).
template <bool INDIRECT, bool VEC, int KB, bool GMF>
__global__ void __launch_bounds__(256) segreduce_level_kernel(const int32_t* __restrict__ keys,
                                                              const int32_t* __restrict__ index, int64_t n,
                                                              const float* __restrict__ rows, int32_t* __restrict__ out_keys,
                                                              float* __restrict__ out_rows, const RowUpdate u,
                                                              const GmfRows g) {
  static_assert(!GMF || (INDIRECT && VEC), "the GMF columns are formed at level 0, four per lane");
  const int lane = threadIdx.x & 31;
  const int64_t chunk = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t base = chunk * 32;
  if (base >= n) return;  // warp-uniform
  const int ld = u.d0 + u.d1;
  const int rs = GMF ? u.d0 : ld;  // floats between staged rows
  const int64_t e = base + lane;
  const int key = e < n ? __ldg(keys + e) : kPastEnd;
  const int64_t src = e < n ? (INDIRECT ? (int64_t)__ldg(index + e) : e) : 0;
  const bool ok = e < n && key != kSkip;
  // GMF: this lane's entry's dz and user (-1: out of range, its GMF row reads as zeros as in the fused kernel)
  float dz_e = 0.f;
  int user_e = -1;
  if (GMF && ok) {
    dz_e = __ldg(g.dz + src);
    const int usr = __ldg(g.group_users + src / g.group);
    user_e = (unsigned)usr < (unsigned)g.num_users ? usr : -1;
  }
  const int kprev = base > 0 ? __ldg(keys + base - 1) : kNoNeighbour;
  const int knext = base + 32 < n ? __ldg(keys + base + 32) : kNoNeighbour;
  int kup = __shfl_up_sync(0xffffffffu, key, 1);
  const unsigned starts = __ballot_sync(0xffffffffu, e < n && (lane == 0 || key != kup));

  ChunkInfo ci;
  ci.nvalid = (int)min((int64_t)32, n - base);
  const int key0 = __shfl_sync(0xffffffffu, key, 0);
  const int keyl = __shfl_sync(0xffffffffu, key, ci.nvalid - 1);
  ci.first_inc = key0 != kSkip && kprev == key0;
  ci.last_inc = ci.nvalid == 32 && keyl != kSkip && knext == keyl;
  ci.chunk = chunk;
  ci.ld = ld;
  ci.out_rows = out_rows;
  if (out_keys != nullptr && lane == 0 && blockIdx.y == 0) {
    out_keys[2 * chunk] = ci.first_inc ? key0 : kSkip;
    out_keys[2 * chunk + 1] = ci.last_inc ? keyl : kSkip;
  }

  constexpr int W = VEC ? 4 : 1;
  static_assert(!GMF || 32 % (2 * KB) == 0, "the formed pass takes 2 KB entries per step");
  for (int cb = blockIdx.y * 32 * W; cb < ld; cb += gridDim.y * 32 * W) {
    // GMF: the pass over the formed columns (warp-uniform: the launcher requires d0 % 128 == 0 and d1 <= 64).  Their
    // d1 / 4 <= 16 lanes fit a half-warp, so both halves gather -- entries j0 .. j0 + KB - 1 and the KB after them,
    // same columns -- and the low half sums all 2 KB in order: twice the gathers in flight per warp.
    const bool formed = GMF && cb >= u.d0;
    const int half = formed ? lane >> 4 : 0;
    const int c = formed ? u.d0 + 4 * (lane & 15) : cb + lane * W;
    const bool col = c < ld;                 // a column of the table
    const bool on = col && half == 0;        // ... that this lane sums and flushes
    const float4 w4 = formed && col ? ldg4(g.w + (c - u.d0)) : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int run_key = key0, run_start = 0;
    auto take = [&](int j, const float4& x) {  // entry j of the chunk, in order
      if (j < ci.nvalid) {
        if (j > 0 && ((starts >> j) & 1u)) {  // a new run starts: close the previous one
          flush_run<VEC, GMF>(u, ci, run_key, run_start, j, c, on, acc);
          acc = make_float4(0.f, 0.f, 0.f, 0.f);
          run_start = j;
          run_key = __shfl_sync(0xffffffffu, key, j);
        }
        acc.x += x.x;
        if (VEC) {
          acc.y += x.y;
          acc.z += x.z;
          acc.w += x.w;
        }
      }
    };
    for (int j0 = 0; j0 < ci.nvalid; j0 += formed ? 2 * KB : KB) {
      float4 v[KB];
      if (formed) {  // (dz * w) * gmf_u, rounded after each product like the staged value; __fmul_rn keeps the second
                     // product out of an FMA with the run's add
#pragma unroll
        for (int q = 0; q < KB; ++q) {
          const int j = j0 + KB * half + q;  // < 32: j0 is a multiple of 2 KB
          const float dz = __shfl_sync(0xffffffffu, dz_e, j);
          const int usr = __shfl_sync(0xffffffffu, user_e, j);
          const bool okj = __shfl_sync(0xffffffffu, (int)ok, j) != 0;
          // unconditional loads from a valid address, zeros selected afterwards: a branch around each load made the
          // compiler consume every load before issuing the next
          float4 gu = ldg4(g.user_gmf + (size_t)(usr >= 0 ? usr : 0) * u.d1 + (col ? c - u.d0 : 0));
          if (usr < 0) gu = make_float4(0.f, 0.f, 0.f, 0.f);
          v[q] = make_float4(__fmul_rn(dz * w4.x, gu.x), __fmul_rn(dz * w4.y, gu.y), __fmul_rn(dz * w4.z, gu.z),
                             __fmul_rn(dz * w4.w, gu.w));
          if (!okj) v[q] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int q = 0; q < KB; ++q) take(j0 + q, v[q]);
#pragma unroll
        for (int q = 0; q < KB; ++q) {  // the high half's entries, same columns
          const float4 hi = make_float4(__shfl_down_sync(0xffffffffu, v[q].x, 16), __shfl_down_sync(0xffffffffu, v[q].y, 16),
                                        __shfl_down_sync(0xffffffffu, v[q].z, 16), __shfl_down_sync(0xffffffffu, v[q].w, 16));
          take(j0 + KB + q, hi);
        }
      } else {
#pragma unroll
        for (int q = 0; q < KB; ++q) {
          const int j = j0 + q;  // j < 32 always (nvalid <= 32, KB divides 32)
          const int64_t sj = __shfl_sync(0xffffffffu, src, j);
          const bool okj = __shfl_sync(0xffffffffu, (int)ok, j) != 0;
          v[q] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (okj && on) {
            if (VEC) v[q] = ld_stream4(rows + (size_t)sj * rs + c);
            else v[q].x = __ldg(rows + (size_t)sj * rs + c);
          }
        }
#pragma unroll
        for (int q = 0; q < KB; ++q) take(j0 + q, v[q]);
      }
    }
    flush_run<VEC, GMF>(u, ci, run_key, run_start, ci.nvalid, c, on, acc);
  }
}

static int64_t level_entries(int64_t n) { return 2 * ((n + 31) / 32); }

size_t segreduce_workspace_bytes(int64_t n, int ld) {
  const int64_t n1 = level_entries(n < 1 ? 1 : n), n2 = level_entries(n1);
  return align_up((size_t)n1 * 4, 256) + align_up((size_t)n2 * 4, 256) + align_up((size_t)n1 * ld * 4, 256) +
         align_up((size_t)n2 * ld * 4, 256);
}

int launch_segreduce(const int32_t* sorted_keys, const int32_t* sorted_index, int64_t n, const float* staged,
                     const RowUpdate& u, void* ws, size_t ws_bytes, cudaStream_t st, const GmfRows* gmf,
                     const std::function<int()>& after_level0) {
  if (n == 0) return after_level0 ? after_level0() : MR_OK;
  const int ld = u.d0 + u.d1;
  if (ws_bytes < segreduce_workspace_bytes(n, ld)) {
    set_error("segreduce workspace too small: %zu < %zu", ws_bytes, segreduce_workspace_bytes(n, ld));
    return MR_ERR_WORKSPACE;
  }
  const int64_t n1 = level_entries(n), n2 = level_entries(n1);
  Carver cv(ws);
  int32_t* kbuf[2] = {cv.take<int32_t>(n1), cv.take<int32_t>(n2)};
  float* rbuf[2] = {cv.take<float>((size_t)n1 * ld), cv.take<float>((size_t)n2 * ld)};
  uintptr_t align = reinterpret_cast<uintptr_t>(staged);
  for (const float* q : {u.p0, u.m0, u.v0, u.g0, u.p1, u.m1, u.v1, u.g1}) align |= reinterpret_cast<uintptr_t>(q);
  if (gmf != nullptr)
    for (const float* q : {gmf->w, gmf->user_gmf}) align |= reinterpret_cast<uintptr_t>(q);
  const bool vec = (ld & 3) == 0 && (u.d0 & 3) == 0 && (align & 15) == 0;
  if (gmf != nullptr && !(vec && u.d0 % 128 == 0 && u.d1 <= 64 && u.mode == MR_TABLES_DENSE && gmf->group > 0)) {
    set_error("segreduce: the GMF columns need 16-byte aligned rows, d0 %% 128 == 0, d1 <= 64, dense tables and a group size");
    return MR_ERR_INVALID;
  }
  const GmfRows g = gmf != nullptr ? *gmf : GmfRows{};

  const int32_t* keys = sorted_keys;
  const float* rows = staged;
  int64_t cur = n;
  for (int level = 0;; ++level) {
    const int64_t nchunks = (cur + 31) / 32;
    const bool last = nchunks == 1;
    int32_t* ok = last ? nullptr : kbuf[level & 1];
    float* orows = last ? nullptr : rbuf[level & 1];
    const unsigned blocks = (unsigned)((nchunks + 7) / 8);
    if (level == 0) {
      if (gmf != nullptr)  // (96 registers: 256-thread blocks fit 16 warps per SM, 64-thread blocks 20; measured
                           // on a B200 at 1000 W: the segreduce phase 0.50 -> 0.46 ms)
        segreduce_level_kernel<true, true, kBatch, true><<<(unsigned)((nchunks + 1) / 2), 64, 0, st>>>(
            keys, sorted_index, cur, rows, ok, orows, u, g);
      else if (vec)
        segreduce_level_kernel<true, true, kBatch, false><<<blocks, 256, 0, st>>>(keys, sorted_index, cur, rows, ok, orows, u, g);
      else
        segreduce_level_kernel<true, false, kBatch, false><<<blocks, 256, 0, st>>>(keys, sorted_index, cur, rows, ok, orows, u, g);
    } else {
      const int per = vec ? 128 : 32;  // columns a warp covers per pass
      const dim3 grid(blocks, (unsigned)((ld + per - 1) / per));
      if (vec) segreduce_level_kernel<false, true, kBatchUpper, false><<<grid, 256, 0, st>>>(keys, nullptr, cur, rows, ok, orows, u, g);
      else segreduce_level_kernel<false, false, kBatchUpper, false><<<grid, 256, 0, st>>>(keys, nullptr, cur, rows, ok, orows, u, g);
    }
    MR_LAUNCH_CHECK("segreduce_level_kernel");
    if (level == 0 && after_level0) {
      const int rc = after_level0();
      if (rc != MR_OK) return rc;
    }
    if (last) break;
    keys = ok;
    rows = orows;
    cur = 2 * nchunks;
  }
  return MR_OK;
}

}  // namespace mr
