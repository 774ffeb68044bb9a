// K31 vlmc_sparse24_linear_sp_forward: y[T, R] = x[T, C] . W^T (+ bias) on the sparse tensor cores, reading the
// compressed 2:4 weight (include/vlmc.h, "Compressed 2:4 weights") as stored.  The weight is the sparse A operand
// (M = 128 weight rows), the tokens are B (N <= 192): tcgen05.mma.sp.kind::f16 multiplies only the two positions meta
// names in every group of four, at twice the dense rate.  No expansion, no split-K: one CTA owns an output tile and walks
// K in order, so equal inputs give equal bits.
//
// Per K stage (128 dense columns): values 128 rows x 64 = one SW128 atom (the compressed A of four K = 32 MMAs, 32 B
// apart), meta 128 rows x 8 words (16 B a row: a stack of 8-row x 16 B core matrices, no swizzle), x 2 SW128 atoms of
// N tokens x 64 columns.  Meta goes shared -> TMEM with tcgen05.cp .128x128b (16 B of the tile per TMEM lane), one
// 32-bit column per K = 32 MMA.  The sparse MMA reads that column interleaved over 16-row blocks: for rows r and r + 8
// of a block (r < 8), lane r holds their first words (columns 0-15 of the MMA's 32) in its low / high half, lane r + 8
// their second words.  The tile TMA lands is row-major (lane = row, the stored order), so the guard warp swaps the
// 16-bit halves of each such row pair in place before the copy: no reordered copy of meta exists outside the chip.
// The MMA names its metadata column as an even column plus a selector (idesc bits 0-1) for the odd one.
//
// Warp roles (224 threads, 1 CTA / SM, persistent over tiles = (row tile, token tile), row tiles innermost):
//   warp 0       TMA producer: 3 stages of {x, values, meta}
//   warp 1       TMEM allocator + MMA issuer (one thread): tcgen05.cp of the stage's meta, then its four sparse MMAs
//   warps 2-5    drain: tcgen05.ld -> (+ bias, one rounding) -> y; two accumulators, so a drain overlaps the next tile
//   warp 6       meta guard: the row-pair interleave above, and every all-zero 4-bit code (not a 2:4 pattern: TMA
//                zero-fills rows past R) becomes {0, 1}, whose values are +0 there, before the stage goes to the MMA
#include "tc.cuh"

namespace vlmc {

constexpr int kSmRows = 128;                               // weight rows per tile (UMMA M)
constexpr int kSmK = 128;                                  // dense columns per stage
constexpr int kSmMaxN = 192;                               // tokens per tile (UMMA N)
constexpr int kSmStages = 3;
constexpr uint32_t kSmXAtom = kSmMaxN * 128;               // N tokens x 64 columns x 2 B, SW128
constexpr uint32_t kSmValBytes = kSmRows * 128;            // 128 rows x 64 values x 2 B, SW128
constexpr uint32_t kSmMetaBytes = kSmRows * 16;            // 128 rows x 8 uint16 words
constexpr uint32_t kSmStage = 2 * kSmXAtom + kSmValBytes + kSmMetaBytes;
constexpr int kSmDrWarp0 = 2, kSmDrWarps = 4, kSmGuardWarp = 6;
constexpr int kSmThreads = (kSmGuardWarp + 1) * 32;
constexpr uint32_t kSmTmemCols = 512;                      // accumulators at columns 0 and 256, meta ring from 448
constexpr uint32_t kSmAccStride = 256, kSmMetaCol = 448;
static_assert(kSmDrWarp0 + kSmDrWarps == kSmGuardWarp, "drain warps 2-5 cover the four TMEM lane quarters");
static_assert(kSmStage % 1024 == 0, "SW128 atoms need 1024-byte alignment");
static_assert(kSmMetaCol + 4 * kSmStages <= kSmTmemCols && kSmMaxN <= kSmMetaCol - kSmAccStride, "TMEM budget");

struct __align__(8) SmBarriers {
  uint64_t full[kSmStages], meta_ok[kSmStages], empty[kSmStages];
  uint64_t tmem_full[2], tmem_empty[2];
  uint32_t tmem_base;
};
constexpr size_t kSmSmem = 1024 + kSmStages * kSmStage + sizeof(SmBarriers);

struct SmParams {
  void* y;
  int64_t ldy;
  const void* bias;
  int T, R, C, N, nrt, nks, ntiles;
};

// K-major 16-bit operand, 128-byte swizzle: rows 128 B apart, 8-row groups 1024 B apart (SBO)
__device__ __forceinline__ uint64_t sm_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3ffff) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// no swizzle, 8-row x 16 B core matrices 128 B apart along the rows.  There is one core matrix along K, so the leading
// offset is unused; it is set equal to the stride offset
__device__ __forceinline__ uint64_t sm_desc_meta(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3ffff) >> 4);
  d |= (uint64_t)(128 >> 4) << 16;
  d |= (uint64_t)(128 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}

__device__ __forceinline__ void tc_cp_128x128b(uint32_t taddr, uint64_t sdesc) {
  asm volatile("tcgen05.cp.cta_group::1.128x128b [%0], %1;" :: "r"(taddr), "l"(sdesc) : "memory");
}
__device__ __forceinline__ void tc_mma_sp_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t meta_tmem,
                                              uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "tcgen05.mma.sp.cta_group::1.kind::f16 [%0], %1, %2, [%3], %4, p;\n\t"
      "}" :: "r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(meta_tmem), "r"(idesc), "r"(accumulate) : "memory");
}

// every all-zero 4-bit code of a meta word -> 0b0100 (indices 0, 1)
__device__ __forceinline__ uint32_t sm_guard_word(uint32_t w) {
  uint32_t nz = w | (w >> 1);
  nz |= nz >> 2;
  return w | ((~nz & 0x11111111u) << 2);
}

template <typename T> __device__ __forceinline__ uint16_t sm_round(float v);
template <> __device__ __forceinline__ uint16_t sm_round<__half>(float v) { return __half_as_ushort(__float2half_rn(v)); }
template <> __device__ __forceinline__ uint16_t sm_round<__nv_bfloat16>(float v) {
  return __bfloat16_as_ushort(__float2bfloat16_rn(v));
}
template <typename T> __device__ __forceinline__ float sm_float(uint16_t v);
template <> __device__ __forceinline__ float sm_float<__half>(uint16_t v) { return __half2float(__ushort_as_half(v)); }
template <> __device__ __forceinline__ float sm_float<__nv_bfloat16>(uint16_t v) { return __uint_as_float((uint32_t)v << 16); }

template <typename T>
__global__ void __launch_bounds__(kSmThreads, 1)
sparse24_mma_sp_kernel(const __grid_constant__ CUtensorMap xmap, const __grid_constant__ CUtensorMap vmap,
                       const __grid_constant__ CUtensorMap mmap, const SmParams p, const uint32_t idesc) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  SmBarriers* bars = reinterpret_cast<SmBarriers*>(ring + kSmStages * kSmStage);
  // stage layout: x atom 0, x atom 1, values, meta
  constexpr uint32_t kOffVal = 2 * kSmXAtom, kOffMeta = kOffVal + kSmValBytes;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" :: "l"(&xmap) : "memory");
    asm volatile("prefetch.tensormap [%0];" :: "l"(&vmap) : "memory");
    asm volatile("prefetch.tensormap [%0];" :: "l"(&mmap) : "memory");
    for (int s = 0; s < kSmStages; ++s) {
      mbar_init(&bars->full[s], 1);
      mbar_init(&bars->meta_ok[s], 1);
      mbar_init(&bars->empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) { mbar_init(&bars->tmem_full[s], 1); mbar_init(&bars->tmem_empty[s], kSmDrWarps); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 :: "r"(smem_u32(&bars->tmem_base)), "r"(kSmTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  if (warp == 0) {
    // ===== TMA producer (the x atom past C of a partial last stage is not loaded) =====
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      for (int u = blockIdx.x; u < p.ntiles; u += gridDim.x) {
        const int n0 = (u % p.nrt) * kSmRows, t0 = (u / p.nrt) * p.N;
        for (int ks = 0; ks < p.nks; ++ks) {
          const int k0 = ks * kSmK, na = p.C - k0 > 64 ? 2 : 1;
          mbar_wait(&bars->empty[s], ph ^ 1);
          uint8_t* st = ring + s * kSmStage;
          mbar_expect_tx(&bars->full[s], (uint32_t)(na * p.N * 128) + kSmValBytes + kSmMetaBytes);
          for (int a = 0; a < na; ++a) tma_load_2d(st + a * kSmXAtom, &xmap, &bars->full[s], k0 + 64 * a, t0);
          tma_load_2d(st + kOffVal, &vmap, &bars->full[s], k0 / 2, n0);
          tma_load_2d(st + kOffMeta, &mmap, &bars->full[s], k0 / 16, n0);
          if (++s == kSmStages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == kSmGuardWarp) {
    // ===== meta guard: 2 KB per stage, two row pairs (r, r + 8) of 16 B per lane, rewritten in place =====
    int s = 0; uint32_t ph = 0;
    for (int u = blockIdx.x; u < p.ntiles; u += gridDim.x) {
      for (int ks = 0; ks < p.nks; ++ks) {
        mbar_wait(&bars->full[s], ph);
        uint4* m = reinterpret_cast<uint4*>(ring + s * kSmStage + kOffMeta);
#pragma unroll
        for (int i = 0; i < kSmRows / 2 / 32; ++i) {
          const int pr = i * 32 + lane, r0 = (pr >> 3) * 16 + (pr & 7);
          const uint4 a = m[r0], b = m[r0 + 8];
          m[r0] = make_uint4(sm_guard_word(__byte_perm(a.x, b.x, 0x5410)), sm_guard_word(__byte_perm(a.y, b.y, 0x5410)),
                             sm_guard_word(__byte_perm(a.z, b.z, 0x5410)), sm_guard_word(__byte_perm(a.w, b.w, 0x5410)));
          m[r0 + 8] = make_uint4(sm_guard_word(__byte_perm(a.x, b.x, 0x7632)), sm_guard_word(__byte_perm(a.y, b.y, 0x7632)),
                                 sm_guard_word(__byte_perm(a.z, b.z, 0x7632)), sm_guard_word(__byte_perm(a.w, b.w, 0x7632)));
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars->meta_ok[s]);
        if (++s == kSmStages) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (one thread): the meta copy and the MMAs that read it are issued in order by this thread =====
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      int it = 0;
      for (int u = blockIdx.x; u < p.ntiles; u += gridDim.x, ++it) {
        const int ab = it & 1;
        mbar_wait(&bars->tmem_empty[ab], ((it >> 1) & 1) ^ 1);       // the drain has emptied this accumulator
        tc_fence_after();
        const uint32_t acc = tmem_base + ab * kSmAccStride;
        for (int ks = 0; ks < p.nks; ++ks) {
          const int nk = min(4, (p.C - ks * kSmK) / 32);
          mbar_wait(&bars->meta_ok[s], ph);
          tc_fence_after();
          const uint32_t st = smem_u32(ring + s * kSmStage);
          // the meta slot of stage s (4 columns, 4-aligned) is free: its previous MMAs completed before the producer
          // could refill the stage
          const uint32_t mt = tmem_base + kSmMetaCol + 4 * s;
          tc_cp_128x128b(mt, sm_desc_meta(st + kOffMeta));
          for (int kk = 0; kk < nk; ++kk)
            tc_mma_sp_f16(acc, sm_desc_sw128(st + kOffVal + kk * 32),
                          sm_desc_sw128(st + (kk >> 1) * kSmXAtom + (kk & 1) * 64), mt + (kk & 2),
                          idesc | (uint32_t)(kk & 1), (ks > 0 || kk > 0) ? 1u : 0u);
          tc_commit(&bars->empty[s]);
          if (++s == kSmStages) { s = 0; ph ^= 1; }
        }
        tc_commit(&bars->tmem_full[ab]);
      }
    }
  } else {
    // ===== drain =====
    const int q = warp & 3;                 // TMEM lane quarter this warp may touch
    const int row = q * 32 + lane;
    uint16_t* y = reinterpret_cast<uint16_t*>(p.y);
    const uint16_t* bias = reinterpret_cast<const uint16_t*>(p.bias);
    int it = 0;
    for (int u = blockIdx.x; u < p.ntiles; u += gridDim.x, ++it) {
      const int ab = it & 1;
      const int r = (u % p.nrt) * kSmRows + row, t0 = (u / p.nrt) * p.N;
      const float b = (bias && r < p.R) ? sm_float<T>(bias[r]) : 0.f;
      mbar_wait(&bars->tmem_full[ab], (it >> 1) & 1);
      tc_fence_after();
      for (int c0 = 0; c0 < p.N; c0 += 32) {
        uint32_t v[32];
        tc_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + ab * kSmAccStride + c0, v);
        tc_wait_ld();
        if (r < p.R) {
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const int t = t0 + c0 + e;
            if (c0 + e < p.N && t < p.T) y[(int64_t)t * p.ldy + r] = sm_round<T>(__uint_as_float(v[e]) + b);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars->tmem_empty[ab]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(kSmTmemCols) : "memory");
  }
}

static int sm_map(CUtensorMap* map, CUtensorMapDataType type, const void* base, uint64_t inner, uint64_t outer, int64_t ld,
                  uint32_t box_inner, uint32_t box_outer, CUtensorMapSwizzle swizzle) {
  EncodeTiledFn encode = get_encode_fn();
  if (!encode) return VLMC_ERR_CUDA;
  const cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  const cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  const cuuint32_t box[2] = {box_inner, box_outer};
  const cuuint32_t estr[2] = {1, 1};
  CUresult cr = encode(map, type, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle,
                       CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) { g_last_cuda_error = (int)cr; return VLMC_ERR_CUDA; }
  return VLMC_OK;
}

template <typename T>
static int sm_launch(const CUtensorMap& xmap, const CUtensorMap& vmap, const CUtensorMap& mmap, const SmParams& p,
                     uint32_t idesc, cudaStream_t st) {
  auto kern = sparse24_mma_sp_kernel<T>;
  static bool attr_set = false;
  if (!attr_set) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmSmem) != cudaSuccess)
      return check_launch();
    attr_set = true;
  }
  const int grid = p.ntiles < kNumSMs ? p.ntiles : kNumSMs;
  kern<<<grid, kSmThreads, kSmSmem, st>>>(xmap, vmap, mmap, p, idesc);
  return check_launch();
}

static bool sm_aligned16(const void* ptr) { return ((uintptr_t)ptr & 15) == 0; }

}  // namespace vlmc

extern "C" int vlmc_sparse24_linear_sp_forward(const void* x, int dtype, int64_t T, int C, int64_t ldx, const void* values,
                                               int64_t ldv, const uint16_t* meta, int64_t ldm, int R, const void* bias,
                                               void* y, int64_t ldy, void* stream) {
  using namespace vlmc;
  if (!x || !values || !meta || !y || T < 0 || R < 1 || C < 32 || C % 32 != 0 || ldx < C || ldv < C / 2 ||
      ldm < C / 16 || ldy < R)
    return VLMC_ERR_BAD_ARG;
  if (dtype != VLMC_F16 && dtype != VLMC_BF16) return dtype == VLMC_F32 ? VLMC_ERR_UNSUPPORTED : VLMC_ERR_BAD_ARG;
  if (T == 0) return VLMC_OK;
  if (T > 0x7fffffff) return VLMC_ERR_UNSUPPORTED;
  // TMA: 16-byte aligned bases and row pitches
  if (ldx % 8 != 0 || ldv % 8 != 0 || ldm % 8 != 0 || !sm_aligned16(x) || !sm_aligned16(values) || !sm_aligned16(meta))
    return VLMC_ERR_UNSUPPORTED;
  if (!is_device_ptr(x) || !is_device_ptr(values) || !is_device_ptr(meta) || !is_device_ptr(y) ||
      (bias && !is_device_ptr(bias)))
    return VLMC_ERR_NOT_DEVICE;

  const int64_t n16 = (T + 15) / 16 * 16;
  const int N = (int)(n16 < kSmMaxN ? n16 : kSmMaxN);
  const int64_t ntt = (T + N - 1) / N, nrt = (R + kSmRows - 1) / kSmRows;
  if (ntt * nrt > 0x7fffffff) return VLMC_ERR_UNSUPPORTED;
  const CUtensorMapDataType dt = dtype == VLMC_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  CUtensorMap xmap, vmap, mmap;
  int rc = sm_map(&xmap, dt, x, (uint64_t)C, (uint64_t)T, ldx, 64, (uint32_t)N, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  rc = sm_map(&vmap, dt, values, (uint64_t)(C / 2), (uint64_t)R, ldv, kSmK / 2, kSmRows, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  rc = sm_map(&mmap, CU_TENSOR_MAP_DATA_TYPE_UINT16, meta, (uint64_t)(C / 16), (uint64_t)R, ldm, kSmK / 16, kSmRows,
              CU_TENSOR_MAP_SWIZZLE_NONE);
  if (rc) return rc;

  SmParams p;
  p.y = y; p.ldy = ldy; p.bias = bias;
  p.T = (int)T; p.R = R; p.C = C; p.N = N; p.nrt = (int)nrt;
  p.nks = (C + kSmK - 1) / kSmK;
  p.ntiles = (int)(ntt * nrt);
  // instruction descriptor (cute::UMMA::InstrDescriptor): sparse, fp32 accumulate, A (weights) and B (tokens) K-major,
  // M = 128
  const uint32_t fmt = dtype == VLMC_F16 ? 0u : 1u;
  const uint32_t idesc = (1u << 2) | (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(N >> 3) << 17) |
                         ((uint32_t)(kSmRows >> 4) << 24);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == VLMC_F16) return sm_launch<__half>(xmap, vmap, mmap, p, idesc, st);
  return sm_launch<__nv_bfloat16>(xmap, vmap, mmap, p, idesc, st);
}
