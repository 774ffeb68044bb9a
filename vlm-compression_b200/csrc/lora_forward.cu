// K15 / K16: the SparseLoRA masked training forward and its LoRA gradients (SURVEY 8f-2).
//
// Replaces lavis/peft/src/peft/tuners/lora.py:359-382 (Linear.forward, r > 0, not merged)
//   sparse:      F.linear(x, (W + (B @ A).to(W.dtype) * scaling) * mask)        (:364-369)
//   not sparse:  F.linear(x,  W * mask + (B @ A).to(W.dtype) * scaling)         (:370-375)
// which re-materialises a dense [R, C] weight EVERY training step through ~5 elementwise passes (fp32 product,
// cast, scale, add, mask) and whose autograd backward makes as many again (mask, scale, cast to fp32) before two
// rank-r GEMMs.  Here
//   K15  vlmc_sparselora_effective_weight   the effective weight in one pass: read W + mask, write W_eff (5 B / weight),
//                                           rank-r dot in registers, the reference's three roundings in W's dtype
//   K16  vlmc_sparselora_lora_grads         dB = E A^T and dA = B^T E with E = (G (.) mask) * scaling rounded like the
//                                           reference's backward (W dtype, then fp32): one read of G + mask per output,
//                                           fp32 accumulation in a fixed order (deterministic)
//   K29  vlmc_sparse24_lora_grads           K16 with the mask taken from a compressed 2:4 weight's meta (4.25 B / weight)
// The two dense GEMMs of the step (y = x W_eff^T, G = dy^T x) stay library GEMMs (cuBLAS through torch).
#include "lora_tile.cuh"
#include "sparse24.cuh"

namespace vlmc {

constexpr int kFwdThreads = 128;

// ---- K15 -------------------------------------------------------------------------------------------------
// Same streaming tile loop as K14 (lora_tile.cuh): A staged in shared memory once per unit, four rows in flight per thread.
template <typename T>
__global__ void __launch_bounds__(kLtThreads, 5)
lora_effective_weight_kernel(const T* __restrict__ W, int64_t ldw, int R, int C, const float* __restrict__ A,
                             const float* __restrict__ B, int rank, float scaling, const uint8_t* __restrict__ mask,
                             int64_t ldm, int sparse, T* __restrict__ out, int64_t ldo, int coltiles, int units) {
  constexpr int V = Elem<T>::kVec;
  extern __shared__ __align__(16) float4 lt_sA[];
  // contiguous span of units per CTA, column tile major / row blocks fastest: A is staged once or twice per CTA
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
    lt_rows<T>(W, ldw, out, ldo, col, rb * kLtUnitRows, row_end, B, rank, mask, ldm, lt_sA,
               [&](float (&f)[V], const float (&acc)[V], const uint32_t (&mb)[2]) { lt_effective<T>(f, acc, mb, scaling, sparse); });
  }
}

// ---- K16 -------------------------------------------------------------------------------------------------
constexpr int kGradMaxRank = 16;

// E[i][j] = float( round_dt( G[i][j] * mask * scaling ) )   (the reference's backward: mask and scale in W's dtype,
// then .to(float32) for the rank-r products)
template <typename T>
__device__ __forceinline__ void grad_e(const uint4& gv, const uint32_t (&mb)[2], int sparse, float scaling, float* e) {
  constexpr int V = Elem<T>::kVec;
  float g[V];
  Elem<T>::unpack(gv, g);
#pragma unroll
  for (int q = 0; q < V; ++q) {
    const bool keep = !sparse || ((mb[q / 4] >> (8 * (q % 4))) & 0xffu);
    e[q] = keep ? round_dt<T>(__fmul_rn(g[q], scaling)) : 0.f;
  }
}

// Where the kernels read the mask of row `row`, columns [col, col + V), as mask bytes: a bool mask (K16) or the meta of
// a compressed 2:4 weight whose kept set is the mask (K29; sparse24.cuh).  Everything else is the same code.
struct MaskBytes {
  const uint8_t* p; int64_t ld;
  template <int V> __device__ __forceinline__ void load(int row, int col, uint32_t (&mb)[2]) const {
    const uint8_t* mp = p + (int64_t)row * ld + col;
    if (V == 8) { const uint2 t = *reinterpret_cast<const uint2*>(mp); mb[0] = t.x; mb[1] = t.y; }
    else mb[0] = *reinterpret_cast<const uint32_t*>(mp);
  }
};
struct MaskMeta24 {
  const uint16_t* p; int64_t ld;
  template <int V> __device__ __forceinline__ void load(int row, int col, uint32_t (&mb)[2]) const {
    sp_meta_mask<V>(p, ld, row, col, mb);
  }
};

// dB[i][k] = sum_j E[i][j] A[k][j]: one warp per row, lanes stride the 16-byte vectors of the row, fixed-order warp
// reduction.  A (rank x C fp32) is read through L1 / L2 (32-128 KB, shared by every row).
template <typename T, int RK, class Mask>
__global__ void __launch_bounds__(256)
lora_grad_b_kernel(const T* __restrict__ G, int64_t ldg, int R, int C, const Mask mask, int sparse,
                   const float* __restrict__ A, int rank, float scaling, float* __restrict__ dB) {
  constexpr int V = Elem<T>::kVec;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nvec = C / V;
  for (int row = blockIdx.x * 8 + warp; row < R; row += gridDim.x * 8) {
    float acc[RK];
#pragma unroll
    for (int k = 0; k < RK; ++k) acc[k] = 0.f;
    for (int j = lane; j < nvec; j += 32) {
      const uint4 gv = ld_stream(G + (int64_t)row * ldg + j * V);
      uint32_t mb[2] = {0x01010101u, 0x01010101u};
      if (sparse) mask.template load<V>(row, j * V, mb);
      float e[V];
      grad_e<T>(gv, mb, sparse, scaling, e);
#pragma unroll
      for (int k = 0; k < RK; ++k) {
        if (k < rank) {
          const float* ap = A + (int64_t)k * C + j * V;
#pragma unroll
          for (int q = 0; q < V; q += 4) {
            const float4 av = __ldg(reinterpret_cast<const float4*>(ap + q));
            acc[k] = fmaf(e[q], av.x, acc[k]); acc[k] = fmaf(e[q + 1], av.y, acc[k]);
            acc[k] = fmaf(e[q + 2], av.z, acc[k]); acc[k] = fmaf(e[q + 3], av.w, acc[k]);
          }
        }
      }
    }
#pragma unroll
    for (int k = 0; k < RK; ++k) {
      if (k < rank) {
        const float s = warp_sum(acc[k]);
        if (lane == 0) dB[(int64_t)row * rank + k] = s;
      }
    }
  }
}

// dA[k][j] = sum_i B[i][k] E[i][j]: a thread owns 16 bytes of columns, CTAs split the rows into chunks, partial sums
// go to the workspace [chunk][rank][C] and a second kernel adds the chunks in order.
template <typename T, int RK, class Mask>
__global__ void __launch_bounds__(kFwdThreads)
lora_grad_a_partial_kernel(const T* __restrict__ G, int64_t ldg, int R, int C, const Mask mask, int sparse,
                           const float* __restrict__ B, int rank, float scaling, int rows_per_chunk,
                           float* __restrict__ part) {
  constexpr int V = Elem<T>::kVec;
  const int col = (blockIdx.x * kFwdThreads + threadIdx.x) * V;
  if (col >= C) return;
  const int r0 = blockIdx.y * rows_per_chunk;
  const int r1 = r0 + rows_per_chunk < R ? r0 + rows_per_chunk : R;
  float acc[RK][V];
#pragma unroll
  for (int k = 0; k < RK; ++k)
#pragma unroll
    for (int q = 0; q < V; ++q) acc[k][q] = 0.f;
  for (int row = r0; row < r1; ++row) {
    const uint4 gv = ld_stream(G + (int64_t)row * ldg + col);
    uint32_t mb[2] = {0x01010101u, 0x01010101u};
    if (sparse) mask.template load<V>(row, col, mb);
    float e[V];
    grad_e<T>(gv, mb, sparse, scaling, e);
    const float* brow = B + (int64_t)row * rank;
#pragma unroll
    for (int k = 0; k < RK; ++k) {
      if (k < rank) {
        const float b = __ldg(brow + k);
#pragma unroll
        for (int q = 0; q < V; ++q) acc[k][q] = fmaf(b, e[q], acc[k][q]);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < RK; ++k) {
    if (k < rank) {
      float* pp = part + ((int64_t)blockIdx.y * rank + k) * C + col;
#pragma unroll
      for (int q = 0; q < V; q += 4)
        *reinterpret_cast<float4*>(pp + q) = make_float4(acc[k][q], acc[k][q + 1], acc[k][q + 2], acc[k][q + 3]);
    }
  }
}

__global__ void __launch_bounds__(256)
lora_grad_a_reduce_kernel(const float* __restrict__ part, int nchunks, int64_t n, float* __restrict__ dA) {
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int c = 0; c < nchunks; ++c) s += part[(int64_t)c * n + i];
  dA[i] = s;
}

static int grad_chunks(int R) {
  int chunks = kNumSMs * 2;                 // with C / (128 * V) column tiles this fills the GPU for every shape on the path
  if (chunks > (R + 15) / 16) chunks = (R + 15) / 16;
  return chunks < 1 ? 1 : chunks;
}

// the launches of K16 / K29 (the mask source is the only difference): dB, the dA partials, the ordered chunk sum
template <class Mask>
static int lora_grads_launch(const void* G, int dtype, int R, int C, int64_t ldg, const Mask mask, int sparse,
                             const float* A, const float* B, int rank, float scaling, float* dA, float* dB, void* ws,
                             cudaStream_t st) {
  const int V = dtype == VLMC_F32 ? 4 : 8;
  float* part = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + VLMC_WS_COUNTER_BYTES);
  int bgrid = (R + 7) / 8;
  if (bgrid > kNumSMs * 8) bgrid = kNumSMs * 8;
  const int chunks = grad_chunks(R);
  const int rows_per_chunk = (R + chunks - 1) / chunks;
  const int nchunks = (R + rows_per_chunk - 1) / rows_per_chunk;
  dim3 agrid((C / V + kFwdThreads - 1) / kFwdThreads, nchunks);
#define VLMC_GRADS(RK)                                                                                                  \
  VLMC_DISPATCH_DTYPE(dtype, {                                                                                          \
    lora_grad_b_kernel<scalar_t, RK, Mask><<<bgrid, 256, 0, st>>>(reinterpret_cast<const scalar_t*>(G), ldg, R, C,     \
                                                                  mask, sparse, A, rank, scaling, dB);                  \
    lora_grad_a_partial_kernel<scalar_t, RK, Mask><<<agrid, kFwdThreads, 0, st>>>(                                      \
        reinterpret_cast<const scalar_t*>(G), ldg, R, C, mask, sparse, B, rank, scaling, rows_per_chunk, part);         \
  })
  if (rank <= 4) { VLMC_GRADS(4); }
  else if (rank <= 8) { VLMC_GRADS(8); }
  else { VLMC_GRADS(16); }
#undef VLMC_GRADS
  const int64_t n = (int64_t)rank * C;
  lora_grad_a_reduce_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(part, nchunks, n, dA);
  return check_launch();
}

}  // namespace vlmc

extern "C" int vlmc_sparselora_effective_weight(const void* W, int dtype, int R, int C, int64_t ldw, const float* A,
                                                const float* B, int rank, float scaling, const uint8_t* keep_mask,
                                                int64_t ldm, int sparse, void* out, int64_t ldo, void* stream) {
  using namespace vlmc;
  if (!W || !A || !B || !keep_mask || !out || R < 1 || C < 1 || rank < 1 || ldw < C || ldm < C || ldo < C) return VLMC_ERR_BAD_ARG;
  if (dtype != VLMC_F32 && dtype != VLMC_F16 && dtype != VLMC_BF16) return VLMC_ERR_BAD_ARG;
  const int V = dtype == VLMC_F32 ? 4 : 8;
  if (C % V != 0 || ldw % V != 0 || ldm % V != 0 || ldo % V != 0 || ((uintptr_t)W & 15) != 0 || ((uintptr_t)out & 15) != 0 ||
      ((uintptr_t)keep_mask & 7) != 0)
    return VLMC_ERR_UNSUPPORTED;
  if (!is_device_ptr(W) || !is_device_ptr(A) || !is_device_ptr(B) || !is_device_ptr(keep_mask) || !is_device_ptr(out))
    return VLMC_ERR_NOT_DEVICE;
  if (rank > kLtMaxRank) return VLMC_ERR_UNSUPPORTED;
  if (((uintptr_t)A & 15) != 0 || C % 4 != 0) return VLMC_ERR_UNSUPPORTED;
  const int coltiles = (C / V + kLtThreads - 1) / kLtThreads;
  const int64_t units64 = (int64_t)coltiles * ((R + kLtUnitRows - 1) / kLtUnitRows);
  if (units64 > 0x7fffffff) return VLMC_ERR_UNSUPPORTED;
  const int units = (int)units64;
  cudaStream_t st = (cudaStream_t)stream;
  VLMC_DISPATCH_DTYPE(dtype, {
    auto kern = lora_effective_weight_kernel<scalar_t>;
    const size_t smem = lt_smem_bytes<scalar_t>(rank);
    static size_t attr = 0;
    if (smem > attr) {
      if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lt_smem_bytes<scalar_t>(kLtMaxRank)) != cudaSuccess)
        return check_launch();
      attr = lt_smem_bytes<scalar_t>(kLtMaxRank);
    }
    int per_sm = 1;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kLtThreads, smem);
    int grid = kNumSMs * (per_sm < 1 ? 1 : per_sm);
    if (grid > units) grid = units;
    kern<<<grid, kLtThreads, smem, st>>>(reinterpret_cast<const scalar_t*>(W), ldw, R, C, A, B, rank, scaling, keep_mask, ldm,
                                         sparse, reinterpret_cast<scalar_t*>(out), ldo, coltiles, units);
  });
  return check_launch();
}

extern "C" size_t vlmc_sparselora_lora_grads_workspace_bytes(int R, int C, int rank) {
  using namespace vlmc;
  if (R < 1 || C < 1 || rank < 1) return 0;
  return VLMC_WS_COUNTER_BYTES + (size_t)grad_chunks(R) * rank * C * sizeof(float);
}

extern "C" int vlmc_sparselora_lora_grads(const void* G, int dtype, int R, int C, int64_t ldg, const uint8_t* keep_mask,
                                          int64_t ldm, int sparse, const float* A, const float* B, int rank,
                                          float scaling, float* dA, float* dB, void* ws, size_t ws_bytes, void* stream) {
  using namespace vlmc;
  if (!G || !A || !B || !dA || !dB || !ws || R < 1 || C < 1 || rank < 1 || ldg < C) return VLMC_ERR_BAD_ARG;
  if (sparse && (!keep_mask || ldm < C)) return VLMC_ERR_BAD_ARG;
  if (rank > kGradMaxRank) return VLMC_ERR_UNSUPPORTED;
  if (dtype != VLMC_F32 && dtype != VLMC_F16 && dtype != VLMC_BF16) return VLMC_ERR_BAD_ARG;
  const int V = dtype == VLMC_F32 ? 4 : 8;
  if (C % V != 0 || ldg % V != 0 || (sparse && ldm % V != 0) || ((uintptr_t)G & 15) != 0 || ((uintptr_t)A & 15) != 0 ||
      (sparse && ((uintptr_t)keep_mask & 7) != 0))
    return VLMC_ERR_UNSUPPORTED;
  if (!is_device_ptr(G) || !is_device_ptr(A) || !is_device_ptr(B) || !is_device_ptr(dA) || !is_device_ptr(dB) ||
      !is_device_ptr(ws) || (sparse && !is_device_ptr(keep_mask)))
    return VLMC_ERR_NOT_DEVICE;
  if (ws_bytes < vlmc_sparselora_lora_grads_workspace_bytes(R, C, rank)) return VLMC_ERR_WORKSPACE;
  return lora_grads_launch(G, dtype, R, C, ldg, MaskBytes{keep_mask, ldm}, sparse, A, B, rank, scaling, dA, dB, ws,
                           (cudaStream_t)stream);
}

// K29: K16 with the mask read from the meta of a mask-driven compressed 2:4 weight (K27), same kernels and workspace
extern "C" int vlmc_sparse24_lora_grads(const void* G, int dtype, int R, int C, int64_t ldg, const uint16_t* meta,
                                        int64_t ldm, int sparse, const float* A, const float* B, int rank, float scaling,
                                        float* dA, float* dB, void* ws, size_t ws_bytes, void* stream) {
  using namespace vlmc;
  if (!G || !A || !B || !dA || !dB || !ws || R < 1 || C < 16 || rank < 1 || ldg < C) return VLMC_ERR_BAD_ARG;
  if (sparse && (!meta || ldm < C / 16)) return VLMC_ERR_BAD_ARG;
  if (dtype != VLMC_F16 && dtype != VLMC_BF16) return dtype == VLMC_F32 ? VLMC_ERR_UNSUPPORTED : VLMC_ERR_BAD_ARG;
  if (rank > kGradMaxRank) return VLMC_ERR_UNSUPPORTED;
  if (C % 16 != 0 || ldg % 8 != 0 || ((uintptr_t)G & 15) != 0 || ((uintptr_t)A & 15) != 0 || ((uintptr_t)meta & 1) != 0)
    return VLMC_ERR_UNSUPPORTED;
  if (!is_device_ptr(G) || !is_device_ptr(A) || !is_device_ptr(B) || !is_device_ptr(dA) || !is_device_ptr(dB) ||
      !is_device_ptr(ws) || (sparse && !is_device_ptr(meta)))
    return VLMC_ERR_NOT_DEVICE;
  if (ws_bytes < vlmc_sparselora_lora_grads_workspace_bytes(R, C, rank)) return VLMC_ERR_WORKSPACE;
  return lora_grads_launch(G, dtype, R, C, ldg, MaskMeta24{meta, ldm}, sparse, A, B, rank, scaling, dA, dB, ws,
                           (cudaStream_t)stream);
}
