// K28 / K30: SparseLoRA on a compressed 2:4 weight whose kept set is the layer's mask (K27, sparse24.cu).
//
// The reference fine-tunes a pruned model through the masked forward (lavis/peft/src/peft/tuners/lora.py:364-375) and
// merges with a re-mask (lora.py:384-394, train.py:634-637) on a dense frozen weight plus a bool mask: 3 B / weight
// resident.  A 2:4 mask is exactly the meta of the compressed format, so the layer can keep values + meta instead
// (1.125 B / weight).  Both kernels run the K14 / K15 tile loop with a compressed loader (lt_rows_sp24, sparse24.cuh):
//   K28  vlmc_sparse24_lora_effective_weight   values + meta -> W_eff [R, C] dense, bit-identical to K15 on
//                                              (decompress(values, meta), mask = meta); 3.125 B / weight
//   K30  vlmc_sparse24_lora_merge              values <- round(values + s * B A) at the stored slots, in place, bit-
//                                              identical to K14 with remask on the same pair; 2.25 B / weight
// K29 (the LoRA gradients) lives beside K16 in lora_forward.cu: the same kernels with a meta mask source.
#include "sparse24.cuh"

namespace vlmc {

// kMerge = false: K28 (out = the effective weight); true: K30 (values merged in place, out unused)
template <typename T, bool kMerge>
__global__ void __launch_bounds__(kLtThreads, 5)
sparse24_lora_tile_kernel(uint16_t* values, int64_t ldv, const uint16_t* __restrict__ meta, int64_t ldm, int R, int C,
                          const float* __restrict__ A, const float* __restrict__ B, int rank, float scaling, int sparse,
                          T* __restrict__ out, int64_t ldo, int units) {
  constexpr int V = Elem<T>::kVec;
  extern __shared__ __align__(16) float4 lt_sA[];
  // K15's schedule: a contiguous span of units per CTA, column tile major / row blocks fastest
  const int rowblocks = (R + kLtUnitRows - 1) / kLtUnitRows;
  const int u0 = (int)((int64_t)blockIdx.x * units / gridDim.x), u1 = (int)((int64_t)(blockIdx.x + 1) * units / gridDim.x);
  int staged_ct = -1;
  for (int unit = u0; unit < u1; ++unit) {
    const int ct = unit / rowblocks, rb = unit - ct * rowblocks;
    const int col0 = ct * kLtThreads * V;
    if (ct != staged_ct) {
      __syncthreads();
      lt_stage_a<T>(lt_sA, A, rank, C, col0);
      __syncthreads();
      staged_ct = ct;
    }
    const int col = col0 + threadIdx.x * V;
    if (col >= C) continue;
    const int row_end = (rb + 1) * kLtUnitRows < R ? (rb + 1) * kLtUnitRows : R;
    if (kMerge)
      lt_rows_sp24<T, true>(values, ldv, meta, ldm, out, ldo, col, rb * kLtUnitRows, row_end, B, rank, lt_sA,
                            [&](float (&f)[V], const float (&acc)[V], const uint32_t (&mb)[2]) { lt_merge<T>(f, acc, mb, scaling, 1); });
    else
      lt_rows_sp24<T, false>(values, ldv, meta, ldm, out, ldo, col, rb * kLtUnitRows, row_end, B, rank, lt_sA,
                             [&](float (&f)[V], const float (&acc)[V], const uint32_t (&mb)[2]) { lt_effective<T>(f, acc, mb, scaling, sparse); });
  }
}

template <typename T, bool kMerge>
static int sparse24_lora_launch(void* values, int64_t ldv, const uint16_t* meta, int64_t ldm, int R, int C, const float* A,
                                const float* B, int rank, float scaling, int sparse, void* out, int64_t ldo,
                                cudaStream_t st) {
  constexpr int V = Elem<T>::kVec;
  const int coltiles = (C / V + kLtThreads - 1) / kLtThreads;
  const int64_t units64 = (int64_t)coltiles * ((R + kLtUnitRows - 1) / kLtUnitRows);
  if (units64 > 0x7fffffff) return VLMC_ERR_UNSUPPORTED;
  const int units = (int)units64;
  auto kern = sparse24_lora_tile_kernel<T, kMerge>;
  const size_t smem = lt_smem_bytes<T>(rank);
  static size_t attr = 0;
  if (smem > attr) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lt_smem_bytes<T>(kLtMaxRank)) != cudaSuccess)
      return check_launch();
    attr = lt_smem_bytes<T>(kLtMaxRank);
  }
  int per_sm = 1;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kLtThreads, smem);
  int grid = kNumSMs * (per_sm < 1 ? 1 : per_sm);
  if (grid > units) grid = units;
  kern<<<grid, kLtThreads, smem, st>>>(static_cast<uint16_t*>(values), ldv, meta, ldm, R, C, A, B, rank, scaling, sparse,
                                       static_cast<T*>(out), ldo, units);
  return check_launch();
}

// the checks K28 and K30 share: 16-bit values, C % 16 == 0, 8-byte value rows (4 values per 8 columns), A 16-byte aligned
static int sparse24_lora_check(const void* values, int dtype, int R, int C, int64_t ldv, const uint16_t* meta, int64_t ldm,
                               const float* A, const float* B, int rank) {
  if (!values || !meta || !A || !B || R < 1 || C < 16 || rank < 1 || ldv < C / 2 || ldm < C / 16) return VLMC_ERR_BAD_ARG;
  if (dtype != VLMC_F16 && dtype != VLMC_BF16) return dtype == VLMC_F32 ? VLMC_ERR_UNSUPPORTED : VLMC_ERR_BAD_ARG;
  if (C % 16 != 0 || rank > kLtMaxRank || ldv % 4 != 0 || ((uintptr_t)values & 7) != 0 || ((uintptr_t)meta & 1) != 0 ||
      ((uintptr_t)A & 15) != 0)
    return VLMC_ERR_UNSUPPORTED;
  if (!is_device_ptr(values) || !is_device_ptr(meta) || !is_device_ptr(A) || !is_device_ptr(B)) return VLMC_ERR_NOT_DEVICE;
  return VLMC_OK;
}

}  // namespace vlmc

extern "C" int vlmc_sparse24_lora_effective_weight(const void* values, int dtype, int R, int C, int64_t ldv,
                                                   const uint16_t* meta, int64_t ldm, const float* A, const float* B,
                                                   int rank, float scaling, int sparse, void* out, int64_t ldo,
                                                   void* stream) {
  using namespace vlmc;
  int rc = sparse24_lora_check(values, dtype, R, C, ldv, meta, ldm, A, B, rank);
  if (rc) return rc;
  if (!out || ldo < C) return VLMC_ERR_BAD_ARG;
  if (ldo % 8 != 0 || ((uintptr_t)out & 15) != 0) return VLMC_ERR_UNSUPPORTED;
  if (!is_device_ptr(out)) return VLMC_ERR_NOT_DEVICE;
  void* v = const_cast<void*>(values);        // read only: the K28 instantiation never stores to values
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == VLMC_F16) return sparse24_lora_launch<__half, false>(v, ldv, meta, ldm, R, C, A, B, rank, scaling, sparse, out, ldo, st);
  return sparse24_lora_launch<__nv_bfloat16, false>(v, ldv, meta, ldm, R, C, A, B, rank, scaling, sparse, out, ldo, st);
}

extern "C" int vlmc_sparse24_lora_merge(void* values, int dtype, int R, int C, int64_t ldv, const uint16_t* meta,
                                        int64_t ldm, const float* A, const float* B, int rank, float scaling,
                                        void* stream) {
  using namespace vlmc;
  int rc = sparse24_lora_check(values, dtype, R, C, ldv, meta, ldm, A, B, rank);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == VLMC_F16) return sparse24_lora_launch<__half, true>(values, ldv, meta, ldm, R, C, A, B, rank, scaling, 1, nullptr, 0, st);
  return sparse24_lora_launch<__nv_bfloat16, true>(values, ldv, meta, ldm, R, C, A, B, rank, scaling, 1, nullptr, 0, st);
}
