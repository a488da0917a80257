// On-device negative sampler (replaces MovieLensDataGenerator._get_random_negatives_and_positive,
// movierec/data_pipeline.py:99-113, and the batch layout of __getitem__, :136-150).
//
// One thread per positive; the draws of a positive (Philox4x32-10 keyed by seed, epoch and the positive's global
// index, exact sampling without replacement among the unseen items) are negative_draw.cuh's, which the fold-in kernel
// shares.  oracle/movierec_oracle.py:device_sample_group restates them bit for bit.
#include "launchers.h"
#include "negative_draw.cuh"

namespace mr {

__global__ void __launch_bounds__(128) sample_negatives_kernel(
    const int64_t* __restrict__ rowptr, const int32_t* __restrict__ csr, int32_t num_items,
    const int32_t* __restrict__ pos_users, const int32_t* __restrict__ pos_items, int64_t P, int64_t first_index,
    int negs, uint64_t seed, uint64_t epoch, int32_t* __restrict__ out_users, int32_t* __restrict__ out_items,
    float* __restrict__ out_labels) {
  int picked[MR_MAX_NEGS + 1];  // sorted candidate ranks already taken (local memory)
  const int group = negs + 1;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += (int64_t)gridDim.x * blockDim.x) {
    const int u = __ldg(pos_users + p);
    const int64_t lo = __ldg(rowptr + u), hi = __ldg(rowptr + u + 1);
    draw_negatives(csr + lo, (int)(hi - lo), num_items, negs, (uint64_t)(first_index + p), seed, epoch, picked,
                   [&](int j, int item) {
                     if (out_items != nullptr) out_items[p * group + j] = item;
                     if (out_users != nullptr) out_users[p * group + j] = u;
                     if (out_labels != nullptr) out_labels[p * group + j] = 0.f;
                   });
    if (out_items != nullptr) out_items[p * group + negs] = __ldg(pos_items + p);
    if (out_users != nullptr) out_users[p * group + negs] = u;
    if (out_labels != nullptr) out_labels[p * group + negs] = 1.f;
  }
}

int launch_sample_negatives(const int64_t* rowptr, const int32_t* csr_items, int32_t num_items,
                            const int32_t* pos_users, const int32_t* pos_items, int64_t P, int64_t first_index,
                            int negs, uint64_t seed, uint64_t epoch, int32_t* out_users, int32_t* out_items,
                            float* out_labels, cudaStream_t st) {
  if (P == 0) return MR_OK;
  int64_t blocks = (P + 127) / 128;
  const int64_t cap = (int64_t)sm_count() * 16;
  if (blocks > cap) blocks = cap;
  sample_negatives_kernel<<<(unsigned)blocks, 128, 0, st>>>(rowptr, csr_items, num_items, pos_users, pos_items, P,
                                                            first_index, negs, seed, epoch, out_users, out_items,
                                                            out_labels);
  MR_LAUNCH_CHECK("sample_negatives_kernel");
  return MR_OK;
}

}  // namespace mr
