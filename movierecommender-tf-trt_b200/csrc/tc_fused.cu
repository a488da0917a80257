// Fused per-tile train kernel of the projected NeuMF tower (BASELINE config 3: layers 256-128-64, GMF 64, grouped
// batches of 1 positive + negs negatives per user).  ONE persistent kernel covers, for every tile of rows,
//
//   H1 = relu(Pi[item] + Pu[user])                       gather + add + ReLU            (model.py:161-176)
//   H2 = relu(H1 . W2 + b2)                              tcgen05, accumulator in TMEM   (model.py:175-181)
//   z  = w_out . [gmf_u * gmf_i | H2] + b_out, p, BCE    epilogue, thread = row         (model.py:184-188, 213-215)
//   dZ2 = dz * w_out[f:] * (H2 > 0)                      written back as an MMA operand
//   dW2 += H1^T . dZ2 ,  dZ1 = (dZ2 . W2^T) * (H1 > 0)   tcgen05 from the SAME shared-memory tiles
//   staged rows dZ1 and dz per row and [sum_group dZ1 | d gmf_u] per group, d w_out, d b_out, d b2, loss
//
// so that H1, H2, dZ2 never exist in HBM; the per-row HBM traffic is the staged gradient rows (which the sorted
// segmented reduction needs) plus the L2-resident projection / GMF rows.  The GMF item gradient of a row,
// (dz * w_out[:f]) * gmf_u, is not staged: the item-side reduction forms it from dz and the user's GMF row
// (segreduce.cu), which saves 256 B written and 256 B read per row.
//
// fp32 accuracy on the tensor cores: every operand is split into THREE bf16 parts (round to nearest, x = b1 + b2 + b3
// up to 2^-24 |x|) and a product keeps the six part products down to 2^-16: b1.b1' + b1.b2' + b2.b1' + b1.b3' + b3.b1'
// + b2.b2' (fp32 accumulation in TMEM).  Same tensor-pipe time as 3xTF32 (six K=16 MMAs instead of three K=8 MMAs
// per sixteen K elements), 25 % fewer operand bytes, and -- the reason it is used here -- for 16-bit operands the
// SWIZZLE_128B shared-memory layout is the SAME bytes whether a tile is read K-major (reduction over its columns:
// forward / backward) or MN-major (reduction over its rows: weight gradient).  A tile X[row][col] is stored as
// 64-column panels of [rows x 128 B], the 16-byte chunks of a row XOR-ed with (row % 8):
//     K-major  view: M/N index = row, K = col   (SBO = 1024 B between 8-row groups, K-step of 16 = +32 B)
//     MN-major view: M/N index = col, K = row   (LBO = panel stride, SBO = 1024 B, K-step of 16 rows = +2048 B)
// H1 (96 KB), dZ2 (48 KB) and W2 (48 KB) therefore live ONCE in shared memory, all resident.
//
// Tile = 4 TMEM lane quarters x RQ rows, RQ = (32 / GROUP) * GROUP whole groups per quarter (GROUP = 5: 30 rows, two
// zero padding lanes per quarter), so every per-group sum stays inside one warp.
//   warps 0-7   producers: thread = (group, 16-byte piece): loads Pu once and Pi for the GROUP rows, ReLU bits by
//               ballot, bf16 split, st.shared (swizzled); then the GMF branch of the same rows in the same mapping
//               (dot product before the epilogue, row gradients after it)
//   warp  8     one elected thread issues all tcgen05.mma (forward as the H1 halves land; weight gradient, then
//               backward once dZ2 is in shared memory)
//   warps 9-12  epilogue 1 (H2 -> z, p, loss, dz, dZ2 operand, column sums) and epilogue 2 (dZ1 mask, staged rows,
//               group sums), thread = row = TMEM lane
// Everything is single-buffered; the overlap is producers(t + 1) under backward + epilogue 2 of tile t.
#include "launchers.h"
#include "tc_bf16x3.cuh"
#include "tc_common.cuh"

namespace mr {
namespace fz {

constexpr int kD1 = 128, kD2 = 64, kF = 64;
constexpr int kThreads = 16 * 32;
constexpr int kProdThreads = 256;
constexpr int kE1Warp0 = 8, kE2Warp0 = 12;  // epilogue-1 warps 8-11 (warp 8 also issues the MMAs), epilogue-2 warps 12-15
constexpr uint32_t kPanel = 16384;        // [128 rows x 64 bf16], rows of 128 bytes
constexpr uint32_t kH1Part = 2 * kPanel;  // two feature panels per part
constexpr int kEpiLd = 36;                // floats per row of an epilogue warp's 32 x 32 staging tile

// shared-memory map (bytes from the 1024-aligned base)
constexpr uint32_t oH1 = 0;                              // 3 parts x 2 panels
constexpr uint32_t oZ2 = oH1 + 3 * kH1Part;              // 3 parts x 1 panel
constexpr uint32_t oW2 = oZ2 + 3 * kPanel;               // 3 parts x 1 panel
constexpr uint32_t oStage = oW2 + 3 * kPanel;            // 4 warps x 32 x kEpiLd floats (end of kernel: reductions)
constexpr uint32_t oBits = oStage + 4 * 32 * kEpiLd * 4; // 2 buffers x 128 slots x 16 B: four ReLU bits per 16-byte piece
constexpr uint32_t oIds = oBits + 2 * 128 * 16;          // 2 buffers x (128 items + 32 users + 128 labels)
constexpr uint32_t oGdot = oIds + 2 * 288 * 4;           // GMF part of the logit, per slot
constexpr uint32_t oDz = oGdot + 512;                    // dz per slot
constexpr uint32_t oFlag = oDz + 512;                    // per slot: 0 = no row, 1 = row, 2 = row with an id out of range
constexpr uint32_t oConst = oFlag + 512;                 // b2[64] | w_out[f:][64] | w_out[:f][64] | b_out
constexpr uint32_t oRedG = oConst + 1024;                // end of kernel: the producers' d w_out[:f] partials (256 x float4)
constexpr uint32_t oRedE = oRedG + 4096;                 // end of kernel: the epilogue-1 warps' column sums, 4 x 160 floats
constexpr uint32_t kSmemBytes = oRedE + 4 * 160 * 4;

// TMEM columns
//   cFwd / cBwd: forward / backward accumulators of the tile; cWg: dW2 of the tile.  The tensor core's fp32
//   accumulation truncates: n chained MMAs leave ~n x 2^-24 of relative error (measured, tests/test_gpu_tc.py), so a
//   chain over all of a CTA's tiles (3,500 MMAs at the ML-20M batch) would cost 4e-5 -- every tile's dW2 is
//   therefore added to cWgSum by the epilogue-2 warps with ordinary round-to-nearest adds (48 MMAs per chain);
//   cCs: per-lane column sums of dz * H2 (64 columns) and of dZ2 (64), accumulated over the tiles by the epilogue
//   threads themselves (read-modify-write of their own lane: no shuffles per tile, one reduction at the end)
//   cWgSum: dW2 summed over the tiles in fp32 registers (below)
constexpr uint32_t cFwd = 0, cWg = 64, cBwd = 128, cCs = 256, cWgSum = 384, kTmemCols = 512;

// Sum of v[c] over the 32 lanes for every c: lane l returns the total of column l.  31 shuffles, fixed order.
__device__ __forceinline__ float warp_transpose_sum32(float (&v)[32], int lane) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool up = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < off; ++i) {
      const float send = up ? v[i] : v[i + off];
      const float keep = up ? v[i + off] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

__device__ __forceinline__ void cp_async4(void* dst_smem, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(tc::smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ void bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Diagnostics build (-DMR_FUSED_TIMING, tools/fused_timing.py): one thread per role accumulates clock64 deltas per
// segment of its tile loop; g_fused_timing[cta][role * 16 + segment].
#ifdef MR_FUSED_TIMING
__device__ long long g_fused_timing[256 * 48];
#define FZ_T_DECL long long tz_[16] = {0}; long long tz_last_ = clock64();
#define FZ_T(seg) { const long long n_ = clock64(); tz_[seg] += n_ - tz_last_; tz_last_ = n_; }
#define FZ_T_FLUSH(role, cond) if (cond) { for (int q_ = 0; q_ < 16; ++q_) g_fused_timing[blockIdx.x * 48 + (role) * 16 + q_] = tz_[q_]; }
#else
#define FZ_T_DECL
#define FZ_T(seg)
#define FZ_T_FLUSH(role, cond)
#endif

struct FusedParams {
  const float* Pi;        // [num_items x 128]  E_item . W1[item rows]
  const float* Pu;        // [num_users x 128]  E_user . W1[user rows] + b1
  const float* user_gmf;  // [num_users x 64]
  const float* item_gmf;  // [num_items x 64]
  const int32_t* users;   // one id per row (equal inside a group: checked by check_grouped_kernel)
  const int32_t* items;
  const float* labels;
  int32_t num_users, num_items;
  int64_t rows;
  const uint16_t* w2_image;  // pack_w2_bf16x3_kernel output: 3 parts x [128 x 64] bf16, swizzled
  const float* b2;
  const float* w_out;     // [f + 64]
  const float* b_out;
  float inv_batch;
  float* probs;           // [rows]
  float* stage_i;         // [rows x si]: columns [0, 128) dZ1
  float* dz_rows;         // [rows]
  float* stage_u;         // [rows / GROUP x su]: columns [0, 128) group sums of dZ1, [128, 192) d gmf_u
  int32_t si, su;
  float* partial;         // this launch's dense-gradient partial rows: row = CTA, stride partial_stride
  int64_t partial_stride;
  int64_t off_w2, off_b2, off_wout, off_bout;  // offsets of W2, b2, w_out, b_out inside a partial row
  float* loss_partial;    // [grid]
  int32_t* flags;         // bit 0: an id out of range was seen
};

template <int GROUP>
__global__ void __launch_bounds__(kThreads, 1) neumf_fused_train_kernel(const FusedParams p) {
  constexpr int GQ = 32 / GROUP, RQ = GQ * GROUP, GT = 4 * GQ, TR = 4 * RQ;
  constexpr int NT = GT * 16;                 // (group, 16-byte piece of a 64-feature half) tasks per half
  static_assert((2 * NT) % kProdThreads == 0, "H1 tasks must divide evenly over the producer threads");
  constexpr int SLOTS = 2 * NT / kProdThreads;
  constexpr int GSLOTS = (NT + kProdThreads - 1) / kProdThreads;

  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t h1_full[2], fwd_done, gmf_ready, dz2_full, h1_free, bwd_done, e2_done, wg_read, w2_bar;
  __shared__ uint32_t tmem_slot;
  // 1024-byte alignment of the operand tiles, computed in the shared window so that the compiler keeps treating
  // `smem` as shared memory (through a uintptr_t round trip every access became a generic LD / ST: ncu showed the
  // producers' stores and the epilogues' staging loads on the long scoreboard)
  uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t ntiles = (p.rows + TR - 1) / TR;
  float* gdot_s = reinterpret_cast<float*>(smem + oGdot);
  float* dz_s = reinterpret_cast<float*>(smem + oDz);
  int32_t* flag_s = reinterpret_cast<int32_t*>(smem + oFlag);
  float* const_s = reinterpret_cast<float*>(smem + oConst);

  // ---- one-time setup ------------------------------------------------------------------------------------
  for (uint32_t e = tid; e < oW2 / 16; e += kThreads) reinterpret_cast<uint4*>(smem)[e] = make_uint4(0u, 0u, 0u, 0u);
  for (int e = tid; e < 128; e += kThreads) {
    gdot_s[e] = 0.f;
    dz_s[e] = 0.f;
    flag_s[e] = 0;
  }
  for (int e = tid; e < 64; e += kThreads) {
    const_s[e] = __ldg(p.b2 + e);
    const_s[64 + e] = __ldg(p.w_out + kF + e);
    const_s[128 + e] = __ldg(p.w_out + e);
  }
  if (tid == 0) {
    const_s[192] = __ldg(p.b_out);
    tc::mbar_init(&h1_full[0], 8);
    tc::mbar_init(&h1_full[1], 8);
    tc::mbar_init(&fwd_done, 1);
    tc::mbar_init(&gmf_ready, 8);
    tc::mbar_init(&dz2_full, 4);
    tc::mbar_init(&h1_free, 1);
    tc::mbar_init(&bwd_done, 1);
    tc::mbar_init(&e2_done, 4);
    tc::mbar_init(&wg_read, 4);
    tc::mbar_init(&w2_bar, 1);
    tc::mbar_init_fence();
  }
  if (warp == kE1Warp0) tc::tmem_alloc(&tmem_slot, kTmemCols);
  tc::fence_proxy_async();  // the zero fill must be visible to the tensor core (padding rows are never written again)
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_base = tmem_slot;
  if (tid == 0) {  // the W2 operand image, once per CTA
    tc::mbar_arrive_expect_tx(&w2_bar, 3 * kPanel);
    tc::bulk_g2s(smem + oW2, p.w2_image, 3 * kPanel, &w2_bar);
  }

  if (warp < 8) {
    // ================================ producers / GMF branch =================================================
    const float4 wg4 = *reinterpret_cast<const float4*>(const_s + 128 + 4 * (tid & 15));
    float4 accg = make_float4(0.f, 0.f, 0.f, 0.f);  // d w_out[:f] of this thread's four columns
    int32_t* ids_s = reinterpret_cast<int32_t*>(smem + oIds);
    auto load_ids = [&](int64_t tile, int buf, bool async) {
      const int64_t row0 = tile * TR;
      int32_t* dst = ids_s + buf * 288;
      if (tid < TR) {
        const int64_t r = row0 + tid;
        if (r < p.rows) {
          if (async) cp_async4(dst + tid, p.items + r);
          else dst[tid] = __ldg(p.items + r);
        } else {
          dst[tid] = 0;
        }
      } else if (tid >= 128 && tid < 128 + GT) {
        const int64_t r = row0 + (int64_t)(tid - 128) * GROUP;
        if (r < p.rows) {
          if (async) cp_async4(dst + tid, p.users + r);
          else dst[tid] = __ldg(p.users + r);
        } else {
          dst[tid] = 0;
        }
      }
      if (tid >= 128 && tid < 128 + TR) {  // the labels of the tile's rows, read by the epilogue warps
        const int64_t r = row0 + (tid - 128);
        float* ldst = reinterpret_cast<float*>(dst) + 160 + (tid - 128);
        if (r < p.rows) {
          if (async) cp_async4(ldst, p.labels + r);
          else *ldst = __ldg(p.labels + r);
        } else {
          *ldst = 0.f;
        }
      }
    };
    if (blockIdx.x < ntiles) load_ids(blockIdx.x, 0, false);
    bar_sync(1, kProdThreads);
    bool any_bad = false;
    int64_t it = 0;
    FZ_T_DECL
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
      const int buf = (int)(it & 1);
      const int64_t row0 = tile * TR;
      const int32_t* ids = ids_s + buf * 288;
      FZ_T(0)
      if (tile + gridDim.x < ntiles) load_ids(tile + gridDim.x, buf ^ 1, true);

      // the task indices below are re-derived from an opaque copy of the thread index every tile: left to itself the
      // compiler hoisted ~40 per-task shared-memory offsets out of the tile loop and spilled them (their reloads sat
      // on the long scoreboard inside the conversion loop)
      int tidv = tid;
      asm volatile("" : "+r"(tidv));
      // ---- H1 = relu(Pi[item] + Pu[user]) and the GMF dot products, software-pipelined over the thread's tasks: the
      // loads of task s + 2 are issued before task s + 1 is converted, so two tasks (12 x 16 B per thread, 48 KB per
      // SM) are in flight and at most two tasks' rows are live in registers (the first version issued all 18 loads of
      // a tile up front: ptxas spilled the loaded rows and every spill store waited for its load)
      auto h1_issue = [&](int s, float4& xu, float4 (&xi)[GROUP]) {
        const int T = tidv + kProdThreads * s;
        const int ps = T >= NT ? 1 : 0, idx = T - ps * NT;
        const int gt = idx >> 4, pc = idx & 15;
        const int col = 64 * ps + 4 * pc;
        const bool gvalid = row0 + (int64_t)gt * GROUP < p.rows;
        const int u = ids[128 + gt];
        const bool uok = gvalid && (unsigned)u < (unsigned)p.num_users;
        xu = uok ? ldg4(p.Pu + (size_t)u * kD1 + col) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int j = 0; j < GROUP; ++j) {
          const int itm = ids[gt * GROUP + j];
          const bool iok = uok && (unsigned)itm < (unsigned)p.num_items;
          xi[j] = iok ? ldg4(p.Pi + (size_t)itm * kD1 + col) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      };
      uint8_t* bits_b = smem + oBits + buf * (128 * 16);
      auto h1_store = [&](int s, const float4& xu, const float4 (&xi)[GROUP]) {
        const int T = tidv + kProdThreads * s;
        const int ps = T >= NT ? 1 : 0, idx = T - ps * NT;
        const int gt = idx >> 4, pc = idx & 15;
        const int sl0 = 32 * (gt / GQ) + GROUP * (gt % GQ);
#pragma unroll
        for (int j = 0; j < GROUP; ++j) {
          const int sl = sl0 + j;
          const float4 a = xi[j], b = xu;
          const float v0 = fmaxf(a.x + b.x, 0.f), v1 = fmaxf(a.y + b.y, 0.f), v2 = fmaxf(a.z + b.z, 0.f),
                      v3 = fmaxf(a.w + b.w, 0.f);
          // four ReLU bits of this 16-byte piece; two neighbouring pieces share a byte (epilogue 2 reads the slot's
          // 16 bytes).  One shuffle per row: the four ballots + field extraction of the first version cost 3x this.
          const uint32_t nib = (v0 > 0.f ? 1u : 0u) | (v1 > 0.f ? 2u : 0u) | (v2 > 0.f ? 4u : 0u) | (v3 > 0.f ? 8u : 0u);
          const uint32_t nib_hi = __shfl_xor_sync(0xffffffffu, nib, 1);
          if (!(pc & 1)) bits_b[sl * 16 + 8 * ps + (pc >> 1)] = (uint8_t)(nib | (nib_hi << 4));
          uint32_t w1a, w2a, w3a, w1b, w2b, w3b;
          split3(v0, v1, w1a, w2a, w3a);
          split3(v2, v3, w1b, w2b, w3b);
          const uint32_t off = oH1 + ps * kPanel + (uint32_t)sl * 128 + ((((pc >> 1) ^ (sl & 7)) << 4) | ((pc & 1) << 3));
          *reinterpret_cast<uint2*>(smem + off) = make_uint2(w1a, w1b);
          *reinterpret_cast<uint2*>(smem + off + kH1Part) = make_uint2(w2a, w2b);
          *reinterpret_cast<uint2*>(smem + off + 2 * kH1Part) = make_uint2(w3a, w3b);
        }
      };
      auto h1_arrive = [&](int half) {
        tc::fence_proxy_async();
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&h1_full[half]);
      };
      auto gmf_issue = [&](int s, float4& gu, float4 (&gi)[GROUP]) {
        const int idx = tidv + kProdThreads * s;
        const int gt = idx >> 4, pc = idx & 15;
        const bool gvalid = row0 + (int64_t)gt * GROUP < p.rows;
        const int u = ids[128 + gt];
        const bool uok = gvalid && (unsigned)u < (unsigned)p.num_users;
        gu = uok ? ldg4(p.user_gmf + (size_t)u * kF + 4 * pc) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int j = 0; j < GROUP; ++j) {
          const int itm = ids[gt * GROUP + j];
          const bool iok = uok && (unsigned)itm < (unsigned)p.num_items;
          gi[j] = iok ? ldg4(p.item_gmf + (size_t)itm * kF + 4 * pc) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      };
      auto gmf_dot = [&](int s, const float4& gu, const float4 (&gi)[GROUP]) {
        const int idx = tidv + kProdThreads * s;
        const int gt = idx >> 4, pc = idx & 15;
        const int sl0 = 32 * (gt / GQ) + GROUP * (gt % GQ);
        const bool gvalid = row0 + (int64_t)gt * GROUP < p.rows;
        const bool uok = (unsigned)ids[128 + gt] < (unsigned)p.num_users;
#pragma unroll
        for (int j = 0; j < GROUP; ++j) {
          float sdot = wg4.x * (gu.x * gi[j].x);
          sdot = fmaf(wg4.y, gu.y * gi[j].y, sdot);
          sdot = fmaf(wg4.z, gu.z * gi[j].z, sdot);
          sdot = fmaf(wg4.w, gu.w * gi[j].w, sdot);
          sdot += __shfl_xor_sync(0xffffffffu, sdot, 1);
          sdot += __shfl_xor_sync(0xffffffffu, sdot, 2);
          sdot += __shfl_xor_sync(0xffffffffu, sdot, 4);
          sdot += __shfl_xor_sync(0xffffffffu, sdot, 8);
          if (pc == 0) {
            const bool bad = gvalid && !(uok && (unsigned)ids[gt * GROUP + j] < (unsigned)p.num_items);
            any_bad |= bad;
            gdot_s[sl0 + j] = sdot;
            flag_s[sl0 + j] = gvalid ? (bad ? 2 : 1) : 0;
          }
        }
      };
      static_assert(SLOTS >= 2, "the producer pipeline keeps two tasks in flight");
      static_assert(NT >= kProdThreads, "every producer warp must own a task of the first half (its h1_full[0] arrival)");
      // which half a task belongs to is warp-uniform: T = tid + 256 s >= NT; a warp's LAST task of half 0 is followed
      // by its arrival on h1_full[0], its last task overall by h1_full[1]
      const bool g1_live = tid + kProdThreads < NT;  // second GMF task (GSLOTS == 2): warp-uniform
      static_assert(GSLOTS <= 2, "two GMF tasks per thread at most");
      float4 xu[2], xi[2][GROUP];
      float4 gu[GSLOTS], gi[GSLOTS][GROUP];
      h1_issue(0, xu[0], xi[0]);
      h1_issue(1, xu[1], xi[1]);
      FZ_T(1)
      if (it > 0) {  // the weight-gradient MMAs of the previous tile have read H1
        tc::mbar_wait(&h1_free, (uint32_t)((it - 1) & 1));
      }
      FZ_T(2)
#pragma unroll
      for (int s = 0; s < SLOTS; ++s) {
        h1_store(s, xu[s & 1], xi[s & 1]);
        const bool last_of_half0 = (tidv + kProdThreads * s < NT) && (tidv + kProdThreads * (s + 1) >= NT);
        if (last_of_half0) h1_arrive(0);
        // at most two tasks' rows live at any time: the next H1 task takes the registers just converted; the GMF rows
        // follow once the H1 loads are all issued
        if (s + 2 < SLOTS) h1_issue(s + 2, xu[s & 1], xi[s & 1]);
        else if (s + 2 == SLOTS) gmf_issue(0, gu[0], gi[0]);
        else if (GSLOTS > 1 && g1_live) gmf_issue(1, gu[GSLOTS - 1], gi[GSLOTS - 1]);
      }
      h1_arrive(1);
      FZ_T(4)
      // ---- GMF branch, part 1: gmf_u * gmf_i . w_out[:f] per row (the rows stay in registers for part 2)
      gmf_dot(0, gu[0], gi[0]);
      if (GSLOTS > 1 && g1_live) gmf_dot(1, gu[GSLOTS - 1], gi[GSLOTS - 1]);
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&gmf_ready);
      FZ_T(5)

      // ---- GMF branch, part 2 (after the epilogue has dz): dz per row and the group's d gmf_u, straight to the staged
      // rows, and the d w_out[:f] partials
      tc::mbar_wait(&dz2_full, (uint32_t)(it & 1));
      FZ_T(6)
#pragma unroll
      for (int s = 0; s < GSLOTS; ++s) {
        const int idx = tidv + kProdThreads * s;
        if (s > 0 && !g1_live) continue;
        const int gt = idx >> 4, pc = idx & 15;
        const int sl0 = 32 * (gt / GQ) + GROUP * (gt % GQ);
        const int64_t grow0 = row0 + (int64_t)gt * GROUP;
        const bool gvalid = grow0 < p.rows;
        float4 ga = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int j = 0; j < GROUP; ++j) {
          const float dz = dz_s[sl0 + j];
          // (here rather than in epilogue 1, where the store made ptxas spill more of the kernel)
          if (gvalid && pc == 0) p.dz_rows[grow0 + j] = dz;
          const float4 g = make_float4(dz * wg4.x, dz * wg4.y, dz * wg4.z, dz * wg4.w);
          const float4 u4 = gu[s], i4 = gi[s][j];
          accg.x = fmaf(dz, u4.x * i4.x, accg.x);
          accg.y = fmaf(dz, u4.y * i4.y, accg.y);
          accg.z = fmaf(dz, u4.z * i4.z, accg.z);
          accg.w = fmaf(dz, u4.w * i4.w, accg.w);
          ga.x = fmaf(g.x, i4.x, ga.x);
          ga.y = fmaf(g.y, i4.y, ga.y);
          ga.z = fmaf(g.z, i4.z, ga.z);
          ga.w = fmaf(g.w, i4.w, ga.w);
        }
        if (gvalid) *reinterpret_cast<float4*>(p.stage_u + (size_t)(grow0 / GROUP) * p.su + kD1 + 4 * pc) = ga;
      }
      FZ_T(7)
      cp_async_wait_all();
      bar_sync(1, kProdThreads);  // the next tile's ids are in place; gdot / flags / dz may be rewritten
      FZ_T(8)
    }
    FZ_T_FLUSH(0, tid == 0)
    if (any_bad) atomicOr(p.flags, 1);
    *reinterpret_cast<float4*>(smem + oRedG + 16 * tid) = accg;
  } else if (warp < kE2Warp0) {
    // ================================ epilogue 1 (thread = row = TMEM lane) + the MMA issuer =================
    // Warp kE1Warp0 also issues every tcgen05.mma of the CTA, through one elected lane, in the two windows in which
    // the epilogue-1 warps have nothing to do anyway: before the forward accumulator is ready (forward MMAs) and
    // after dZ2 has been handed over (weight gradient, backward).  A dedicated issuer warp would be the 17th warp.
    const int quarter = warp & 3;
    const int slot = 32 * quarter + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * quarter) << 16);
    const float b_out = const_s[192];
    const bool issuer = warp == kE1Warp0;
    const uint32_t s0 = tc::smem_u32(smem);
    const uint64_t dk = tc::smem_desc(0, 16, 1024, kLayoutSw128);        // K-major view (LBO unused)
    const uint64_t dmn = tc::smem_desc(0, kPanel, 1024, kLayoutSw128);   // MN-major view, 64-column blocks kPanel apart
    const uint32_t id_fwd = idesc_bf16(128, kD2, 0, 1);   // H1 (K-major) x W2 (MN-major: N = output unit)
    const uint32_t id_bwd = idesc_bf16(128, kD1, 0, 0);   // dZ2 (K-major) x W2 (K-major: N = input unit)
    const uint32_t id_wg = idesc_bf16(128, kD2, 1, 1);    // H1^T (MN-major) x dZ2 (MN-major)
    // the six part products of a 3 x bf16 split product (a part, b part)
    constexpr int PA[6] = {0, 0, 1, 0, 2, 1}, PB[6] = {0, 1, 0, 2, 0, 1};
    {  // zero this lane's column-sum accumulators
      float zero[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) zero[i] = 0.f;
#pragma unroll
      for (int c = 0; c < 4; ++c) tmem_st32(lane_addr + cCs + 32 * c, zero);
    }
    float accb = 0.f, accl = 0.f;
    int64_t it = 0;
    FZ_T_DECL
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
      const uint32_t ph = (uint32_t)(it & 1);
      const int64_t row0 = tile * TR;
      const int64_t row = row0 + quarter * RQ + lane;
      const bool live = lane < RQ && row < p.rows;

      if (issuer) {
        // forward: acc_fwd[slot][j] = sum_i H1[slot][i] W2[i][j], one 64-feature half as soon as it has landed
        if (tc::elect_one()) {
          if (it == 0) tc::mbar_wait(&w2_bar, 0);
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            tc::mbar_wait(&h1_full[half], ph);
            tc::fence_after_sync();
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
              for (int q = 0; q < 6; ++q) {
                const uint32_t a = s0 + oH1 + PA[q] * kH1Part + half * kPanel + ks * 32;
                const uint32_t b = s0 + oW2 + PB[q] * kPanel + (4 * half + ks) * 2048;
                mma_bf16(tmem_base + cFwd, dk + (a >> 4), dmn + (b >> 4), id_fwd, (half | ks | q) != 0);
              }
            }
          }
          tc::mma_commit(&fwd_done);
        }
        __syncwarp();
      }

      tc::mbar_wait(&fwd_done, ph);
      tc::fence_after_sync();
      FZ_T(0)
      // two passes over the accumulator (TMEM reads are cheap, registers are not): the logit first, then -- once dz
      // is known -- H2 again, 32 columns at a time, for dZ2 and the column sums
      float zdot = 0.f;
#pragma unroll
      for (int cb = 0; cb < 2; ++cb) {
        float h[32];
        tmem_ld32(lane_addr + cFwd + 32 * cb, h);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float4 bv = *reinterpret_cast<const float4*>(const_s + 32 * cb + 4 * q);
          const float4 wv = *reinterpret_cast<const float4*>(const_s + 64 + 32 * cb + 4 * q);
          zdot = fmaf(fmaxf(h[4 * q + 0] + bv.x, 0.f), wv.x, zdot);
          zdot = fmaf(fmaxf(h[4 * q + 1] + bv.y, 0.f), wv.y, zdot);
          zdot = fmaf(fmaxf(h[4 * q + 2] + bv.z, 0.f), wv.z, zdot);
          zdot = fmaf(fmaxf(h[4 * q + 3] + bv.w, 0.f), wv.w, zdot);
        }
      }
      FZ_T(1)
      tc::mbar_wait(&gmf_ready, ph);
      FZ_T(2)
      const int flag = flag_s[slot];
      // (the label arrived with the tile's ids: a global load here was sunk to its first use by the compiler and
      // sat on the long scoreboard in the middle of the epilogue)
      const float y = live ? reinterpret_cast<const float*>(smem + oIds)[(it & 1) * 288 + 160 + quarter * RQ + lane] : 0.f;
      const float z = zdot + gdot_s[slot] + b_out;
      const float pr = sigmoidf_stable(z);
      if (live) p.probs[row] = flag == 2 ? nanf("") : pr;
      const float dz = (live && flag == 1) ? (pr - y) * p.inv_batch : 0.f;
      if (live && flag == 1) accl += bce_logits(z, y);
      accb += dz;
      dz_s[slot] = dz;
#pragma unroll
      for (int cb = 0; cb < 2; ++cb) {
        float h[32], g[32];
        tmem_ld32(lane_addr + cFwd + 32 * cb, h);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float4 bv = *reinterpret_cast<const float4*>(const_s + 32 * cb + 4 * q);
          const float4 wv = *reinterpret_cast<const float4*>(const_s + 64 + 32 * cb + 4 * q);
          h[4 * q + 0] = fmaxf(h[4 * q + 0] + bv.x, 0.f);
          h[4 * q + 1] = fmaxf(h[4 * q + 1] + bv.y, 0.f);
          h[4 * q + 2] = fmaxf(h[4 * q + 2] + bv.z, 0.f);
          h[4 * q + 3] = fmaxf(h[4 * q + 3] + bv.w, 0.f);
          g[4 * q + 0] = h[4 * q + 0] > 0.f ? dz * wv.x : 0.f;
          g[4 * q + 1] = h[4 * q + 1] > 0.f ? dz * wv.y : 0.f;
          g[4 * q + 2] = h[4 * q + 2] > 0.f ? dz * wv.z : 0.f;
          g[4 * q + 3] = h[4 * q + 3] > 0.f ? dz * wv.w : 0.f;
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {  // 16-byte chunk 4 * cb + c of the slot's 128-byte row, in each part
          uint32_t w1[4], w2[4], w3[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) split3(g[8 * c + 2 * e], g[8 * c + 2 * e + 1], w1[e], w2[e], w3[e]);
          const uint32_t off = oZ2 + (uint32_t)slot * 128 + ((((4 * cb + c) ^ (slot & 7))) << 4);
          *reinterpret_cast<uint4*>(smem + off) = make_uint4(w1[0], w1[1], w1[2], w1[3]);
          *reinterpret_cast<uint4*>(smem + off + kPanel) = make_uint4(w2[0], w2[1], w2[2], w2[3]);
          *reinterpret_cast<uint4*>(smem + off + 2 * kPanel) = make_uint4(w3[0], w3[1], w3[2], w3[3]);
        }
        // column sums for d w_out[f:] (dz * H2) and d b2 (dZ2): this lane's running sums live in TMEM
        float acc[32];
        tmem_ld32(lane_addr + cCs + 32 * cb, acc);
#pragma unroll
        for (int i = 0; i < 32; ++i) acc[i] = fmaf(dz, h[i], acc[i]);
        tmem_st32(lane_addr + cCs + 32 * cb, acc);
        tmem_ld32(lane_addr + cCs + 64 + 32 * cb, acc);
#pragma unroll
        for (int i = 0; i < 32; ++i) acc[i] += g[i];
        tmem_st32(lane_addr + cCs + 64 + 32 * cb, acc);
      }
      tc::fence_proxy_async();
      tc::fence_before_sync();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&dz2_full);
      FZ_T(3)

      if (issuer) {
        // weight gradient first (it frees H1 for the producers), then backward
        if (tc::elect_one()) {
          tc::mbar_wait(&dz2_full, ph);
          // epilogue 2 of the previous tile has read its accumulator (and long since its ReLU bits), and the previous
          // tile's dW2 has been taken out of cWg
          if (it > 0) {
            tc::mbar_wait(&e2_done, (uint32_t)((it - 1) & 1));
            tc::mbar_wait(&wg_read, (uint32_t)((it - 1) & 1));
          }
          tc::fence_after_sync();
#pragma unroll
          for (int ks = 0; ks < 8; ++ks) {
#pragma unroll
            for (int q = 0; q < 6; ++q) {
              const uint32_t a = s0 + oH1 + PA[q] * kH1Part + ks * 2048;
              const uint32_t b = s0 + oZ2 + PB[q] * kPanel + ks * 2048;
              mma_bf16(tmem_base + cWg, dmn + (a >> 4), dmn + (b >> 4), id_wg, (ks | q) != 0);
            }
          }
          tc::mma_commit(&h1_free);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
#pragma unroll
            for (int q = 0; q < 6; ++q) {
              const uint32_t a = s0 + oZ2 + PA[q] * kPanel + ks * 32;
              const uint32_t b = s0 + oW2 + PB[q] * kPanel + ks * 32;
              mma_bf16(tmem_base + cBwd, dk + (a >> 4), dk + (b >> 4), id_bwd, (ks | q) != 0);
            }
          }
          tc::mma_commit(&bwd_done);
        }
        __syncwarp();
      }
      FZ_T(4)
    }
    FZ_T_FLUSH(1, warp == kE1Warp0 && lane == 0)
    // this warp's column sums: the 32 lanes' TMEM accumulators folded once, fixed order; scratch = oRedE (per warp)
    float* red = reinterpret_cast<float*>(smem + oRedE) + (warp - kE1Warp0) * 160;
#pragma unroll
    for (int c = 0; c < 4; ++c) {  // c = 0, 1: d w_out[f:] columns 32 c ..; c = 2, 3: d b2 columns 32 (c - 2) ..
      float v[32];
      tmem_ld32(lane_addr + cCs + 32 * c, v);
      red[32 * c + lane] = warp_transpose_sum32(v, lane);
    }
    accb = warp_sum(accb);
    accl = warp_sum(accl);
    if (lane == 0) {
      red[128] = accb;
      red[129] = accl;
    }
  } else {
    // ================================ epilogue 2 (thread = row = TMEM lane) =====================================
    // dZ1 = acc_bwd * (H1 > 0) -> staged item rows; group sums -> staged user rows.  Its own four warps: it runs
    // under the producers' work on the next tile and never delays epilogue 1.
    const int quarter = warp & 3;
    const int slot = 32 * quarter + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(32 * quarter) << 16);
    float* tile_s = reinterpret_cast<float*>(smem + oStage) + (size_t)(warp - kE2Warp0) * (32 * kEpiLd);
    {  // zero this lane's (= input unit's) row of the dW2 sum
      float zero[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) zero[i] = 0.f;
      tmem_st32(lane_addr + cWgSum, zero);
      tmem_st32(lane_addr + cWgSum + 32, zero);
    }
    int64_t it = 0;
    FZ_T_DECL
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
      const uint32_t ph = (uint32_t)(it & 1);
      const int64_t row0 = tile * TR;
      // this tile's dW2 out of the tensor core's accumulator as soon as its MMAs are done (h1_free), into the sum
      tc::mbar_wait(&h1_free, ph);
      tc::fence_after_sync();
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        float w[32], acc[32];
        tmem_ld32(lane_addr + cWg + 32 * c, w);
        if (c == 1) {  // cWg is in registers: the next tile's weight-gradient MMAs may overwrite it
          tc::fence_before_sync();
          __syncwarp();
          if (lane == 0) tc::mbar_arrive(&wg_read);
        }
        tmem_ld32(lane_addr + cWgSum + 32 * c, acc);
#pragma unroll
        for (int i = 0; i < 32; ++i) acc[i] += w[i];
        tmem_st32(lane_addr + cWgSum + 32 * c, acc);
      }
      tc::mbar_wait(&bwd_done, ph);
      tc::fence_after_sync();
      FZ_T(0)
      const uint4 bw = *reinterpret_cast<const uint4*>(smem + oBits + (it & 1) * (128 * 16) + slot * 16);
      const uint32_t bwv[4] = {bw.x, bw.y, bw.z, bw.w};  // nibble = piece (4 columns): word cb holds columns 32 cb ..
      const int64_t qrow0 = row0 + quarter * RQ;          // first row of this warp's quarter
      const int64_t qgrp0 = tile * GT + quarter * GQ;     // its first group
#pragma unroll
      for (int cb = 0; cb < 4; ++cb) {
        float v[32];
        tmem_ld32(lane_addr + cBwd + 32 * cb, v);
        if (cb == 3) {  // the accumulator is in registers: the next backward pass may overwrite it
          tc::fence_before_sync();
          __syncwarp();
          if (lane == 0) tc::mbar_arrive(&e2_done);
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) {  // column 32 cb + i: piece 8 cb + i / 4 = nibble i / 4 of word cb, bit i % 4
          if (!((bwv[cb] >> i) & 1u)) v[i] = 0.f;
        }
#pragma unroll
        for (int q = 0; q < 8; ++q)
          *reinterpret_cast<float4*>(tile_s + lane * kEpiLd + 4 * q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int idx = lane + 32 * j, r = idx >> 3, c4 = idx & 7;
          if (r < RQ && qrow0 + r < p.rows)
            *reinterpret_cast<float4*>(p.stage_i + (size_t)(qrow0 + r) * p.si + 32 * cb + 4 * c4) =
                *reinterpret_cast<const float4*>(tile_s + r * kEpiLd + 4 * c4);
        }
#pragma unroll
        for (int gq = 0; gq < GQ; ++gq) {
          float s = 0.f;
#pragma unroll
          for (int j = 0; j < GROUP; ++j) s += tile_s[(gq * GROUP + j) * kEpiLd + lane];
          if ((qgrp0 + gq) * GROUP < p.rows) p.stage_u[(size_t)(qgrp0 + gq) * p.su + 32 * cb + lane] = s;
        }
        __syncwarp();
      }
      FZ_T(1)
    }
    FZ_T_FLUSH(2, warp == kE2Warp0 && lane == 0)
    // ---- end of the CTA's tiles: dW2 (TMEM lane = input unit) into this CTA's partial row
    if (it > 0) {
      float* dst = p.partial + (size_t)blockIdx.x * p.partial_stride + p.off_w2 + (size_t)slot * kD2;
#pragma unroll
      for (int cb = 0; cb < 2; ++cb) {
        float v[32];
        tmem_ld32(lane_addr + cWgSum + 32 * cb, v);
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          float4 o = *reinterpret_cast<float4*>(dst + 32 * cb + 4 * q);
          o.x += v[4 * q];
          o.y += v[4 * q + 1];
          o.z += v[4 * q + 2];
          o.w += v[4 * q + 3];
          *reinterpret_cast<float4*>(dst + 32 * cb + 4 * q) = o;
        }
      }
    }
  }

  // ---- per-CTA sums into this CTA's partial row, fixed order ---------------------------------------------------
  // scratch: the epilogue-1 warps' column sums (160 floats each) at oRedE, the producers' d w_out[:f] float4 at oRedG
  tc::fence_before_sync();
  __syncthreads();
  {
    const float* red = reinterpret_cast<const float*>(smem + oRedE);
    const float4* redg = reinterpret_cast<const float4*>(smem + oRedG);
    constexpr int RS = 160;  // floats between the epilogue-1 warps' scratch rows
    float* prow = p.partial + (size_t)blockIdx.x * p.partial_stride;
    if (tid < 64) {  // d w_out[:f]: column tid = piece tid / 4 of the 16 threads tid/4 + 16 k
      float s = 0.f;
      for (int k = 0; k < 16; ++k) {
        const float4 v = redg[(tid >> 2) + 16 * k];
        s += (tid & 3) == 0 ? v.x : (tid & 3) == 1 ? v.y : (tid & 3) == 2 ? v.z : v.w;
      }
      prow[p.off_wout + tid] += s;
    } else if (tid < 128) {  // d w_out[f:]
      const int j = tid - 64;
      float s = 0.f;
      for (int w = 0; w < 4; ++w) s += red[w * RS + j];
      prow[p.off_wout + kF + j] += s;
    } else if (tid < 192) {  // d b2
      const int j = tid - 128;
      float s = 0.f;
      for (int w = 0; w < 4; ++w) s += red[w * RS + 64 + j];
      prow[p.off_b2 + j] += s;
    } else if (tid == 192) {
      float sb = 0.f, sl = 0.f;
      for (int w = 0; w < 4; ++w) {
        sb += red[w * RS + 128];
        sl += red[w * RS + 129];
      }
      prow[p.off_bout] += sb;
      p.loss_partial[blockIdx.x] = sl;
    }
  }
  __syncthreads();
  if (warp == kE1Warp0) tc::tmem_dealloc(tmem_base, kTmemCols);
}

// W2 (128 x 64, Keras (in, out) layout) -> the shared-memory operand image: 3 bf16 parts x [128 rows x 128 B], swizzled.
__global__ void pack_w2_bf16x3_kernel(const float* __restrict__ W, uint16_t* __restrict__ dst) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;  // pair index
  if (e >= kD1 * kD2 / 2) return;
  const int i = e / (kD2 / 2), j = 2 * (e - i * (kD2 / 2));
  uint32_t w1, w2, w3;
  split3(__ldg(W + (size_t)i * kD2 + j), __ldg(W + (size_t)i * kD2 + j + 1), w1, w2, w3);
  const uint32_t off = sw128_off(i, j);
  uint8_t* d = reinterpret_cast<uint8_t*>(dst);
  *reinterpret_cast<uint32_t*>(d + off) = w1;
  *reinterpret_cast<uint32_t*>(d + kPanel + off) = w2;
  *reinterpret_cast<uint32_t*>(d + 2 * kPanel + off) = w3;
}

}  // namespace fz

bool fused_train_supported(const MrModel& m, int group) {
  return m.n_layers == 3 && m.L[0] == 2 * fz::kD1 && m.L[1] == fz::kD1 && m.L[2] == fz::kD2 && m.mf_dim == fz::kF && group == 5;
}

size_t fused_w2_image_bytes() { return 3 * fz::kPanel; }

int launch_fused_train(const FusedTrainArgs& a, cudaStream_t st, int* grid_out) {
  if (a.group != 5) {
    set_error("fused train kernel: unsupported group %d", a.group);
    return MR_ERR_INVALID;
  }
  fz::pack_w2_bf16x3_kernel<<<(fz::kD1 * fz::kD2 / 2 + 255) / 256, 256, 0, st>>>(a.W2, a.w2_image);
  MR_LAUNCH_CHECK("pack_w2_bf16x3_kernel");
  fz::FusedParams p{};
  p.Pi = a.Pi;
  p.Pu = a.Pu;
  p.user_gmf = a.user_gmf;
  p.item_gmf = a.item_gmf;
  p.users = a.users;
  p.items = a.items;
  p.labels = a.labels;
  p.num_users = a.num_users;
  p.num_items = a.num_items;
  p.rows = a.rows;
  p.w2_image = a.w2_image;
  p.b2 = a.b2;
  p.w_out = a.w_out;
  p.b_out = a.b_out;
  p.inv_batch = a.inv_batch;
  p.probs = a.probs;
  p.stage_i = a.stage_i;
  p.dz_rows = a.dz_rows;
  p.stage_u = a.stage_u;
  p.si = a.si;
  p.su = a.su;
  p.partial = a.partial;
  p.partial_stride = a.partial_stride;
  p.off_w2 = a.off_w2;
  p.off_b2 = a.off_b2;
  p.off_wout = a.off_wout;
  p.off_bout = a.off_bout;
  p.loss_partial = a.loss_partial;
  p.flags = a.flags;
  constexpr int TR = 4 * (32 / 5) * 5;
  const int64_t ntiles = (a.rows + TR - 1) / TR;
  int64_t grid = sm_count();
  if (grid > ntiles) grid = ntiles;
  if (grid_out) *grid_out = (int)grid;
  if (grid == 0) return MR_OK;
  auto kern = fz::neumf_fused_train_kernel<5>;
  const size_t smem = fz::kSmemBytes + 1024;
  MR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<(unsigned)grid, fz::kThreads, smem, st>>>(p);
  MR_LAUNCH_CHECK("neumf_fused_train_kernel");
  return MR_OK;
}

#ifdef MR_FUSED_TIMING
extern "C" int mr_fused_timing_read(long long* out_host) {
  return cudaMemcpyFromSymbol(out_host, fz::g_fused_timing, sizeof(long long) * 256 * 48) == cudaSuccess ? 0 : -1;
}
#endif

}  // namespace mr
