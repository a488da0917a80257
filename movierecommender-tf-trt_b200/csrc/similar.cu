// Similar items and similar users: exact k nearest neighbours of rows of one side in the model's scoring space.
//
//   representation of row x:  r_x = concat(p_x / |p_x|, g_x / |g_x|) / sqrt(n_parts)
//     p_x = E_s[x] . W1_s      what the first hidden layer sees of x (linear, no bias; only with a hidden layer)
//     g_x = w_out[0:f] * G_s[x] what the GMF head sees of x (only with mf_dim > 0)
//   A part with zero norm stays zero.  similarity(a, b) = r_a . r_b, the mean of the two per-part cosines.
//
// similar_pack_kernel writes the representation of every row of the side (or of a chunk's query rows, gathered by id)
// as the K-major core-matrix operand image pack_weights_kernel makes for weights (tc_common.cuh): [D/32 chunks][hi, lo]
// [rows x 32], each value split into TF32 hi + lo once.  similar_gemm_kernel then computes S = R_q . R^T for a chunk
// of queries on the tensor cores (3xTF32, fp32 accumulate) with both operands landing in shared memory by bulk copies:
//   warp 0     one thread issues the four bulk copies (A hi / lo, B hi / lo) of every K-chunk of 32
//   warp 1     one elected thread issues tcgen05.mma: acc += Ahi.Bhi + Alo.Bhi + Ahi.Blo per K-step of 8
//   warps 2-9  epilogue: tcgen05.ld the 128 x 256 accumulator (double-buffered in TMEM, 2 x 256 columns), transpose
//              32 x 32 blocks through shared memory and store 128-byte row segments of the row-major score chunk
// Persistent CTAs over tiles of 128 queries x 256 candidates.  Every score is the same MMA sequence over K whatever its
// tile or chunk, so a query's scores do not depend on the other queries of a call or on chunking.
#include "launchers.h"
#include "tc_common.cuh"

namespace mr {

constexpr int kSimKC = 32;       // K elements per pipeline stage
constexpr int kSimStages = 2;    // 96 KB each
constexpr int kSimEpiWarps = 8;  // two per TMEM lane quarter, alternate 32-column blocks
constexpr int kSimThreads = 32 * (2 + kSimEpiWarps);
constexpr int kSimEpiLd = 33;    // floats per row of an epilogue warp's 32 x 32 staging block (conflict-free both ways)
constexpr uint32_t kSimABytes = kSimTileQ * kSimKC * 4;  // one of hi / lo
constexpr uint32_t kSimBBytes = kSimTileC * kSimKC * 4;
constexpr uint32_t kSimStageBytes = 2 * kSimABytes + 2 * kSimBBytes;
constexpr size_t kSimSmem = (size_t)kSimStages * kSimStageBytes + (size_t)kSimEpiWarps * 32 * kSimEpiLd * sizeof(float);

// Row n < rows_pad of the image: the representation of table row id = ids ? ids[n] : n when n < count and the id lies
// in [0, num_rows), else zeros.  One warp per row; the norms are fixed-order warp sums, so a row's image is the same
// whichever call or position writes it.
__global__ void __launch_bounds__(256) similar_pack_kernel(const float* __restrict__ P, int L1,
                                                           const float* __restrict__ G, const float* __restrict__ w_gmf,
                                                           int f, int32_t num_rows, const int32_t* __restrict__ ids,
                                                           int64_t count, int64_t rows_pad, int Dpad, float part_scale,
                                                           float* __restrict__ img) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x / 32);
  for (int64_t n = (int64_t)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5); n < rows_pad; n += warps) {
    int64_t id = -1;
    if (n < count) id = ids != nullptr ? (int64_t)__ldg(ids + n) : n;
    const bool valid = id >= 0 && id < num_rows;  // warp-uniform
    const float* p = valid ? P + id * L1 : nullptr;
    const float* g = valid ? G + id * f : nullptr;
    float sp = 0.f, sg = 0.f;
    if (valid) {
      for (int c = lane; c < L1; c += 32) {
        const float x = __ldg(p + c);
        sp = fmaf(x, x, sp);
      }
      for (int c = lane; c < f; c += 32) {
        const float x = __ldg(w_gmf + c) * __ldg(g + c);
        sg = fmaf(x, x, sg);
      }
    }
    sp = warp_sum(sp);
    sg = warp_sum(sg);
    const float scp = sp > 0.f ? part_scale / sqrtf(sp) : 0.f;
    const float scg = sg > 0.f ? part_scale / sqrtf(sg) : 0.f;
    for (int k = lane; k < Dpad; k += 32) {
      float x = 0.f;
      if (valid) {
        if (k < L1) x = __ldg(p + k) * scp;
        else if (k < L1 + f) x = (__ldg(w_gmf + (k - L1)) * __ldg(g + (k - L1))) * scg;
      }
      float hi, lo;
      tc::split_tf32(x, hi, lo);
      const int c = k / kSimKC, kc = k - c * kSimKC;
      const size_t base = (size_t)c * 2 * rows_pad * kSimKC;
      const size_t off = (size_t)(n >> 3) * (8 * kSimKC) + tc::core_off_rg_major((int)(n & 7), kc, kSimKC / 4) / 4;
      img[base + off] = hi;
      img[base + (size_t)rows_pad * kSimKC + off] = lo;
    }
  }
}

struct SimGemmParams {
  const float* a_img;  // [nchunks][hi, lo][a_rows x 32]: the chunk's queries
  const float* b_img;  // [nchunks][hi, lo][b_rows x 32]: every row of the side
  int64_t a_rows, b_rows;
  int nchunks;
  int64_t C;           // valid query rows
  int32_t N;           // valid candidates
  float* out;          // C x N row-major
};

__global__ void __launch_bounds__(kSimThreads, 1) similar_gemm_kernel(const SimGemmParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ uint64_t full_bar[kSimStages], empty_bar[kSimStages], acc_full[2], acc_empty[2];
  __shared__ uint32_t tmem_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t mt = (p.C + kSimTileQ - 1) / kSimTileQ, nt = ((int64_t)p.N + kSimTileC - 1) / kSimTileC;
  const int64_t ntiles = mt * nt;  // tile t = (query tile t % mt, candidate tile t / mt): neighbours share B
  const int nchunks = p.nchunks;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kSimStages; ++s) {
      tc::mbar_init(&full_bar[s], 1);
      tc::mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      tc::mbar_init(&acc_full[b], 1);
      tc::mbar_init(&acc_empty[b], kSimEpiWarps);
    }
    tc::mbar_init_fence();
  }
  if (warp == 1) tc::tmem_alloc(&tmem_slot, 2 * kSimTileC);
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem_base = tmem_slot;

  if (warp == 0) {
    // ================================ bulk copies ===============================================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t tq = tile % mt, tcand = tile / mt;
        for (int c = 0; c < nchunks; ++c) {
          tc::mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* s = smem + (size_t)stage * kSimStageBytes;
          tc::mbar_arrive_expect_tx(&full_bar[stage], kSimStageBytes);
          const float* a = p.a_img + (size_t)c * 2 * p.a_rows * kSimKC + (size_t)tq * kSimTileQ * kSimKC;
          const float* b = p.b_img + (size_t)c * 2 * p.b_rows * kSimKC + (size_t)tcand * kSimTileC * kSimKC;
          tc::bulk_g2s(s, a, kSimABytes, &full_bar[stage]);
          tc::bulk_g2s(s + kSimABytes, a + (size_t)p.a_rows * kSimKC, kSimABytes, &full_bar[stage]);
          tc::bulk_g2s(s + 2 * kSimABytes, b, kSimBBytes, &full_bar[stage]);
          tc::bulk_g2s(s + 2 * kSimABytes + kSimBBytes, b + (size_t)p.b_rows * kSimKC, kSimBBytes, &full_bar[stage]);
          if (++stage == kSimStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ================================================
    if (tc::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t idesc = tc::idesc_tf32(kSimTileQ, kSimTileC, 0, 0);
      const uint64_t dbase = tc::smem_desc(0, 128, 1024);  // address field added per operand (smem < 256 KB: no carry)
      const uint32_t s0 = tc::smem_u32(smem);
      int64_t it = 0;
      for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
        const int b = (int)(it & 1);
        tc::mbar_wait(&acc_empty[b], (uint32_t)((it >> 1) & 1) ^ 1);
        tc::fence_after_sync();
        const uint32_t d_tmem = tmem_base + (uint32_t)b * kSimTileC;
        for (int c = 0; c < nchunks; ++c) {
          tc::mbar_wait(&full_bar[stage], phase);
          tc::fence_after_sync();
          const uint32_t sa = s0 + (uint32_t)stage * kSimStageBytes;
          const uint32_t sb = sa + 2 * kSimABytes;
          const uint64_t ah = dbase + (sa >> 4), al = dbase + ((sa + kSimABytes) >> 4);
          const uint64_t bh = dbase + (sb >> 4), bl = dbase + ((sb + kSimBBytes) >> 4);
#pragma unroll
          for (int kk = 0; kk < kSimKC / 8; ++kk) {  // one K=8 step = two 128-byte core matrices = 256 bytes
            tc::mma_tf32(d_tmem, ah + 16 * kk, bh + 16 * kk, idesc, (c | kk) != 0);
            tc::mma_tf32(d_tmem, al + 16 * kk, bh + 16 * kk, idesc, 1);
            tc::mma_tf32(d_tmem, ah + 16 * kk, bl + 16 * kk, idesc, 1);
          }
          tc::mma_commit(&empty_bar[stage]);  // stage reusable once these MMAs have read it
          if (c == nchunks - 1) tc::mma_commit(&acc_full[b]);
          if (++stage == kSimStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else {
    // ================================ epilogue ==================================================
    const int e = warp - 2, quarter = warp & 3, half = e >> 2;  // TMEM lane quarter this warp may access
    float* blk = reinterpret_cast<float*>(smem + (size_t)kSimStages * kSimStageBytes) + (size_t)e * 32 * kSimEpiLd;
    int64_t it = 0;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
      const int b = (int)(it & 1);
      const int64_t tq = tile % mt, tcand = tile / mt;
      const int64_t row0 = tq * kSimTileQ + 32 * quarter;
      tc::mbar_wait(&acc_full[b], (uint32_t)((it >> 1) & 1));
      tc::fence_after_sync();
      if (row0 < p.C) {  // warp-uniform: quarters past the chunk's last query hold padding rows only
        const uint32_t taddr = tmem_base + (uint32_t)b * kSimTileC + ((uint32_t)(32 * quarter) << 16);
        for (int cb = half; cb < kSimTileC / 32; cb += 2) {
          const int64_t col0 = tcand * kSimTileC + 32 * cb;
          if (col0 >= p.N) break;  // warp-uniform
          float v[32];
          tc::tmem_ld16(taddr + 32 * cb, v);
          tc::tmem_ld16(taddr + 32 * cb + 16, v + 16);
#pragma unroll
          for (int j = 0; j < 32; ++j) blk[lane * kSimEpiLd + j] = v[j];
          __syncwarp();
          const int64_t col = col0 + lane;
          const int rows = (int)min((int64_t)32, p.C - row0);
          if (col < p.N) {
            float* dst = p.out + (size_t)row0 * p.N + col;
            for (int r = 0; r < rows; ++r) dst[(size_t)r * p.N] = blk[r * kSimEpiLd + lane];
          }
          __syncwarp();
        }
      }
      tc::fence_before_sync();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&acc_empty[b]);
    }
  }
  tc::fence_before_sync();
  __syncthreads();
  if (warp == 1) tc::tmem_dealloc(tmem_base, 2 * kSimTileC);
}

// ---- host ------------------------------------------------------------------------------------------

int launch_similar_pack(const float* P, int L1, const float* G, const float* w_gmf, int f, int32_t num_rows,
                        const int32_t* ids, int64_t count, int64_t rows_pad, int Dpad, int n_parts, float* img,
                        cudaStream_t st) {
  if (rows_pad == 0) return MR_OK;
  int64_t blocks = (rows_pad + 7) / 8;
  const int64_t cap = (int64_t)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  similar_pack_kernel<<<(unsigned)blocks, 256, 0, st>>>(P, L1, G, w_gmf, f, num_rows, ids, count, rows_pad, Dpad,
                                                        1.f / sqrtf((float)n_parts), img);
  MR_LAUNCH_CHECK("similar_pack_kernel");
  return MR_OK;
}

int launch_similar_gemm(const float* a_img, int64_t a_rows, const float* b_img, int64_t b_rows, int Dpad, int64_t C,
                        int32_t N, float* out, cudaStream_t st) {
  if (C == 0 || N == 0) return MR_OK;
  if (Dpad % kSimKC || a_rows % kSimTileQ || b_rows % kSimTileC || a_rows < C || b_rows < N) {
    set_error("similar gemm: unsupported shape D=%d a_rows=%lld b_rows=%lld", Dpad, (long long)a_rows, (long long)b_rows);
    return MR_ERR_INVALID;
  }
  SimGemmParams p{};
  p.a_img = a_img;
  p.b_img = b_img;
  p.a_rows = a_rows;
  p.b_rows = b_rows;
  p.nchunks = Dpad / kSimKC;
  p.C = C;
  p.N = N;
  p.out = out;
  MR_CUDA(cudaFuncSetAttribute(similar_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSimSmem));
  const int64_t ntiles = ((C + kSimTileQ - 1) / kSimTileQ) * (((int64_t)N + kSimTileC - 1) / kSimTileC);
  int64_t grid = sm_count();
  if (grid > ntiles) grid = ntiles;
  similar_gemm_kernel<<<(unsigned)grid, kSimThreads, kSimSmem, st>>>(p);
  MR_LAUNCH_CHECK("similar_gemm_kernel");
  return MR_OK;
}

}  // namespace mr
