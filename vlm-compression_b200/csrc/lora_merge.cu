// K14: SparseLoRA masked merge  W <- (W + scaling * B A) (.) M  in one pass.
//
// Replaces lavis/peft/src/peft/tuners/lora.py:384-387 (Linear.merge, sparse branch)
//   self.weight.data += (B @ A * scaling) * mask        (fp32 math, one rounding to W's dtype)
// fused with the re-mask of train.py:634-637
//   module.weight.data[~module.mask] = 0
// The reference materialises an fp32 [R, C] temporary and makes ~5 passes; here a thread
// owns 16 B of one row, the A columns it needs sit in registers for all rows of its tile,
// the B row is a broadcast load.  HBM-bound: 5 B/weight (read W + mask, write W).
#include "lora_tile.cuh"

namespace vlmc {

// ---- one or many LoRA linears (16 per launch) as ONE list of work units ------------------------------------------------
// train.py:626-637 merges module by module; the matrices are 34-90 MB, so one launch per linear spends a third of its
// time ramping up and draining.  The linears are one list of work units (kLtUnitRows rows x 1024 columns) that a fully
// resident grid strides over; vlmc_sparselora_merge is the same kernel with a list of one.
constexpr int kMbMax = 16;
struct MergeBatchItem {
  void* W; int64_t ldw; int R, C; const float* A; const float* B; int rank; float scaling;
  const uint8_t* mask; int64_t ldm; int coltiles;
};
struct MergeBatch { MergeBatchItem it[kMbMax]; int unit_begin[kMbMax + 1]; int count; };

template <typename T>
__global__ void __launch_bounds__(kLtThreads, 5)
lora_merge_batch_kernel(const __grid_constant__ MergeBatch b, int remask) {
  constexpr int V = Elem<T>::kVec;
  extern __shared__ __align__(16) float4 lt_sA[];
  const int total = b.unit_begin[b.count];
  // contiguous span of units per CTA; units of an item are ordered column tile major, row blocks fastest
  const int u0 = (int)((int64_t)blockIdx.x * total / gridDim.x), u1 = (int)((int64_t)(blockIdx.x + 1) * total / gridDim.x);
  int staged_item = -1, staged_ct = -1, p = 0;
  for (int unit = u0; unit < u1; ++unit) {
    while (unit >= b.unit_begin[p + 1]) ++p;
    const MergeBatchItem& it = b.it[p];
    const int local = unit - b.unit_begin[p];
    const int rowblocks = (it.R + kLtUnitRows - 1) / kLtUnitRows;
    const int ct = local / rowblocks, rb = local - ct * rowblocks;
    const int col0 = ct * kLtThreads * V;
    if (p != staged_item || ct != staged_ct) {
      __syncthreads();                                 // the previous tile's readers are done with sA
      lt_stage_a<T>(lt_sA, it.A, it.rank, it.C, col0);
      __syncthreads();
      staged_item = p; staged_ct = ct;
    }
    const int col = col0 + threadIdx.x * V;
    if (col >= it.C) continue;
    const int row_end = (rb + 1) * kLtUnitRows < it.R ? (rb + 1) * kLtUnitRows : it.R;
    const float scaling = it.scaling;
    T* W = reinterpret_cast<T*>(it.W);
    lt_rows<T>(W, it.ldw, W, it.ldw, col, rb * kLtUnitRows, row_end, it.B, it.rank, it.mask, it.ldm, lt_sA,
               [&](float (&f)[V], const float (&acc)[V], const uint32_t (&mb)[2]) { lt_merge<T>(f, acc, mb, scaling, remask); });
  }
}

static int merge_batch_launch(const vlmc_merge_item* items, int count, int dtype, int remask, cudaStream_t st) {
  if (!items || count < 1 || count > kMbMax) return VLMC_ERR_BAD_ARG;
  if (dtype != VLMC_F32 && dtype != VLMC_F16 && dtype != VLMC_BF16) return VLMC_ERR_BAD_ARG;
  const int V = dtype == VLMC_F32 ? 4 : 8;
  MergeBatch b;
  b.count = count;
  b.unit_begin[0] = 0;
  int max_rank = 1;
  for (int i = 0; i < count; ++i) {
    const vlmc_merge_item& s = items[i];
    if (!s.W || !s.A || !s.B || !s.keep_mask || s.R < 1 || s.C < 1 || s.rank < 1 || s.ldw < s.C || s.ldm < s.C) return VLMC_ERR_BAD_ARG;
    if (s.rank > kLtMaxRank) return VLMC_ERR_UNSUPPORTED;
    if (s.C % V != 0 || s.ldw % V != 0 || s.ldm % V != 0 || ((uintptr_t)s.W & 15) != 0 || ((uintptr_t)s.keep_mask & 7) != 0 ||
        ((uintptr_t)s.A & 15) != 0 || s.C % 4 != 0)
      return VLMC_ERR_UNSUPPORTED;
    if (!is_device_ptr(s.W) || !is_device_ptr(s.A) || !is_device_ptr(s.B) || !is_device_ptr(s.keep_mask)) return VLMC_ERR_NOT_DEVICE;
    MergeBatchItem& it = b.it[i];
    it.W = s.W; it.ldw = s.ldw; it.R = s.R; it.C = s.C; it.A = s.A; it.B = s.B; it.rank = s.rank; it.scaling = s.scaling;
    it.mask = s.keep_mask; it.ldm = s.ldm;
    it.coltiles = (s.C / V + kLtThreads - 1) / kLtThreads;
    const int64_t units = (int64_t)it.coltiles * ((s.R + kLtUnitRows - 1) / kLtUnitRows);
    if (b.unit_begin[i] + units > 0x7fffffff) return VLMC_ERR_UNSUPPORTED;
    b.unit_begin[i + 1] = b.unit_begin[i] + (int)units;
    max_rank = s.rank > max_rank ? s.rank : max_rank;
  }
  const int total = b.unit_begin[count];
  VLMC_DISPATCH_DTYPE(dtype, {
    auto kern = lora_merge_batch_kernel<scalar_t>;
    const size_t smem = lt_smem_bytes<scalar_t>(max_rank);
    static size_t attr = 0;
    if (smem > attr) {
      if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lt_smem_bytes<scalar_t>(kLtMaxRank)) != cudaSuccess)
        return check_launch();
      attr = lt_smem_bytes<scalar_t>(kLtMaxRank);
    }
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kLtThreads, smem);
    int grid = kNumSMs * (per_sm < 1 ? 1 : per_sm);
    if (grid > total) grid = total;
    kern<<<grid, kLtThreads, smem, st>>>(b, remask);
  });
  return check_launch();
}

}  // namespace vlmc

extern "C" int vlmc_sparselora_merge(void* W, int dtype, int R, int C, int64_t ldw,
                                     const float* A, const float* B, int rank, float scaling,
                                     const uint8_t* keep_mask, int64_t ldm, int remask, void* stream) {
  vlmc_merge_item it;
  it.W = W; it.ldw = ldw; it.R = R; it.C = C; it.A = A; it.B = B; it.rank = rank; it.scaling = scaling;
  it.keep_mask = keep_mask; it.ldm = ldm;
  return vlmc::merge_batch_launch(&it, 1, dtype, remask, (cudaStream_t)stream);
}

extern "C" int vlmc_sparselora_merge_batch(const vlmc_merge_item* items, int count, int dtype, int remask, void* stream) {
  return vlmc::merge_batch_launch(items, count, dtype, remask, (cudaStream_t)stream);
}
