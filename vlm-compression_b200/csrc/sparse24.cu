// K24-K26: compressed 2:4 weights for pruned models (format: include/vlmc.h, "Compressed 2:4 weights").
//
// K24 vlmc_sparse24_compress    W [R, C] -> values [R, C/2] + meta [R, C/16] uint16, one pass, a thread per 16-column word
// K27 vlmc_sparse24_compress_masked  W + bool mask -> values + meta: the kept set is the mask (SparseLoRA layers keep
//     their pruned weights unzeroed), exactly two per group
// K25 vlmc_sparse24_decompress  values + meta -> dense W (+0 at pruned positions); the expand step of the large-T path
// K26 vlmc_sparse24_linear_forward  y[T, R] = x[T, C] . W^T (+ bias) reading the COMPRESSED weight: 1.125 B per weight of
//     HBM instead of 2, which is what decode-sized token counts pay for.  Each 128-row x 128-column weight slice is expanded
//     on chip into the dense SW128 operand the kind::f16 tensor core takes (bit-identical to decompress()), and fed to
//     tcgen05.mma with the weight rows as M = 128 and the tokens as N (16..128).
//
// K26 warp roles (352 threads, 1 CTA / SM, persistent over units = (row tile, token tile, k split)):
//   warp 0       TMA producer, raw ring: 5 x {values 128 x 64, meta 128 x 8 words} = 18 KB (90 KB in flight per SM)
//   warp 1       TMEM allocator + MMA issuer (one thread), two accumulators so that a drain overlaps the next unit
//   warp 2       TMA producer, x ring: 2 x {2 atoms of N tokens x 64 columns}, SW128, out-of-bounds rows / columns zero
//   warps 3-6    converters: raw slice -> dense 2 x (128 x 64) SW128 tile (a scatter of two values into four slots),
//                fence.proxy.async, arrive
//   warps 7-10   drain: tcgen05.ld -> (+ bias, one rounding) -> y, or fp32 partial -> workspace; the last CTA of a tile
//                (ticket) sums the partials in split order, so the result does not depend on which CTA finishes last
#include "tc.cuh"
#include "sparse24.cuh"

namespace vlmc {

constexpr int kSpRows = 128;                              // weight rows per tile (UMMA M)
constexpr int kSpK = 128;                                 // columns per stage: the meta of a row slice is 16 B (TMA minimum)
constexpr int kSpMaxN = 128;                              // tokens per tile (UMMA N)
constexpr int kSpRawStages = 5, kSpDenseStages = 2, kSpXStages = 2;
constexpr uint32_t kSpValBytes = kSpRows * kSpK;          // 128 rows x 64 values x 2 B
constexpr uint32_t kSpRawStage = kSpValBytes + kSpRows * 16;
constexpr uint32_t kSpAtom = kSpRows * 128;               // 128 rows x 64 columns x 2 B, SW128
constexpr uint32_t kSpDenseStage = 2 * kSpAtom;
constexpr uint32_t kSpXAtom = kSpMaxN * 128;
constexpr uint32_t kSpXStage = 2 * kSpXAtom;
constexpr int kSpCvtWarp0 = 3, kSpCvtWarps = 4, kSpDrWarp0 = 7, kSpDrWarps = 4;
constexpr int kSpCvtThreads = kSpCvtWarps * 32, kSpDrThreads = kSpDrWarps * 32;
constexpr int kSpThreads = (kSpDrWarp0 + kSpDrWarps) * 32;
constexpr int kSpMaxSplit = 32;
constexpr int kSpMaxTickets = VLMC_WS_COUNTER_BYTES / 4;

struct __align__(8) SpBarriers {
  uint64_t full_raw[kSpRawStages], empty_raw[kSpRawStages];
  uint64_t conv[kSpDenseStages], empty_dense[kSpDenseStages];
  uint64_t full_x[kSpXStages], empty_x[kSpXStages];
  uint64_t tmem_full[2], tmem_empty[2];
  uint32_t tmem_base;
  int last;
};
constexpr size_t kSpSmem = 1024 + kSpXStages * kSpXStage + kSpDenseStages * kSpDenseStage + kSpRawStages * kSpRawStage +
                           sizeof(SpBarriers);

struct SpParams {
  void* y;
  int64_t ldy;
  const void* bias;
  float* part;              // [tiles][S][N][128] fp32 split-K partials (S > 1)
  unsigned int* tickets;    // one per tile, zero on entry and on exit
  int T, R, C, N, nrt, S, nsl, nunits;
  uint32_t acc_cols;
};

struct SpUnit {
  int tile, s, n0, t0, ks0, ks1;
};
__device__ __forceinline__ SpUnit sp_unit(const SpParams& p, int u) {
  SpUnit w;
  w.s = u % p.S;
  w.tile = u / p.S;
  const int rt = w.tile % p.nrt, tt = w.tile / p.nrt;
  w.n0 = rt * kSpRows;
  w.t0 = tt * p.N;
  w.ks0 = (int)((int64_t)w.s * p.nsl / p.S);
  w.ks1 = (int)((int64_t)(w.s + 1) * p.nsl / p.S);
  return w;
}

// K-major 16-bit operand, 128-byte swizzle: rows 128 B apart, 8-row groups 1024 B apart (SBO); LBO unused
__device__ __forceinline__ uint64_t sp_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3ffff) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

template <typename T> __device__ __forceinline__ uint16_t sp_round(float v);
template <> __device__ __forceinline__ uint16_t sp_round<__half>(float v) { return __half_as_ushort(__float2half_rn(v)); }
template <> __device__ __forceinline__ uint16_t sp_round<__nv_bfloat16>(float v) {
  return __bfloat16_as_ushort(__float2bfloat16_rn(v));
}
template <typename T> __device__ __forceinline__ float sp_float(uint16_t v);
template <> __device__ __forceinline__ float sp_float<__half>(uint16_t v) { return __half2float(__ushort_as_half(v)); }
template <> __device__ __forceinline__ float sp_float<__nv_bfloat16>(uint16_t v) { return __uint_as_float((uint32_t)v << 16); }

template <typename T>
__global__ void __launch_bounds__(kSpThreads, 1)
sparse24_linear_kernel(const __grid_constant__ CUtensorMap xmap, const __grid_constant__ CUtensorMap vmap,
                       const __grid_constant__ CUtensorMap mmap, const SpParams p, const uint32_t idesc) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* xring = smem;
  uint8_t* dring = xring + kSpXStages * kSpXStage;
  uint8_t* rring = dring + kSpDenseStages * kSpDenseStage;
  SpBarriers* bars = reinterpret_cast<SpBarriers*>(rring + kSpRawStages * kSpRawStage);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" :: "l"(&xmap) : "memory");
    asm volatile("prefetch.tensormap [%0];" :: "l"(&vmap) : "memory");
    asm volatile("prefetch.tensormap [%0];" :: "l"(&mmap) : "memory");
    for (int s = 0; s < kSpRawStages; ++s) { mbar_init(&bars->full_raw[s], 1); mbar_init(&bars->empty_raw[s], kSpCvtThreads); }
    for (int s = 0; s < kSpDenseStages; ++s) { mbar_init(&bars->conv[s], kSpCvtThreads); mbar_init(&bars->empty_dense[s], 1); }
    for (int s = 0; s < kSpXStages; ++s) { mbar_init(&bars->full_x[s], 1); mbar_init(&bars->empty_x[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&bars->tmem_full[s], 1); mbar_init(&bars->tmem_empty[s], kSpDrWarps); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                 :: "r"(smem_u32(&bars->tmem_base)), "r"(2 * p.acc_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  if (warp == 0) {
    // ===== TMA producer: compressed weight slices =====
    if (lane == 0) {
      int rs = 0; uint32_t rph = 0;
      for (int u = blockIdx.x; u < p.nunits; u += gridDim.x) {
        const SpUnit w = sp_unit(p, u);
        for (int ks = w.ks0; ks < w.ks1; ++ks) {
          mbar_wait(&bars->empty_raw[rs], rph ^ 1);
          uint8_t* sr = rring + rs * kSpRawStage;
          mbar_expect_tx(&bars->full_raw[rs], kSpRawStage);
          tma_load_2d(sr, &vmap, &bars->full_raw[rs], ks * (kSpK / 2), w.n0);
          tma_load_2d(sr + kSpValBytes, &mmap, &bars->full_raw[rs], ks * (kSpK / 16), w.n0);
          if (++rs == kSpRawStages) { rs = 0; rph ^= 1; }
        }
      }
    }
  } else if (warp == 2) {
    // ===== TMA producer: token tiles (the atom past C of a partial last slice is not loaded) =====
    if (lane == 0) {
      int xs = 0; uint32_t xph = 0;
      for (int u = blockIdx.x; u < p.nunits; u += gridDim.x) {
        const SpUnit w = sp_unit(p, u);
        for (int ks = w.ks0; ks < w.ks1; ++ks) {
          const int k0 = ks * kSpK, na = p.C - k0 > 64 ? 2 : 1;
          mbar_wait(&bars->empty_x[xs], xph ^ 1);
          uint8_t* sx = xring + xs * kSpXStage;
          mbar_expect_tx(&bars->full_x[xs], (uint32_t)(na * p.N * 128));
          for (int a = 0; a < na; ++a) tma_load_2d(sx + a * kSpXAtom, &xmap, &bars->full_x[xs], k0 + 64 * a, w.t0);
          if (++xs == kSpXStages) { xs = 0; xph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (one thread) =====
    if (lane == 0) {
      int ds = 0, xs = 0; uint32_t dph = 0, xph = 0;
      int it = 0;
      for (int u = blockIdx.x; u < p.nunits; u += gridDim.x, ++it) {
        const SpUnit w = sp_unit(p, u);
        const int ab = it & 1;
        mbar_wait(&bars->tmem_empty[ab], ((it >> 1) & 1) ^ 1);       // the drain has emptied this accumulator
        tc_fence_after();
        const uint32_t acc = tmem_base + ab * p.acc_cols;
        for (int ks = w.ks0; ks < w.ks1; ++ks) {
          const int na = p.C - ks * kSpK > 64 ? 2 : 1;
          mbar_wait(&bars->conv[ds], dph);
          mbar_wait(&bars->full_x[xs], xph);
          tc_fence_after();
          const uint32_t sd = smem_u32(dring + ds * kSpDenseStage), sx = smem_u32(xring + xs * kSpXStage);
          for (int a = 0; a < na; ++a) {
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
              tc_mma_f16(acc, sp_desc(sd + a * kSpAtom + kk * 32), sp_desc(sx + a * kSpXAtom + kk * 32), idesc,
                         (ks > w.ks0 || a > 0 || kk > 0) ? 1u : 0u);
          }
          tc_commit(&bars->empty_dense[ds]);
          tc_commit(&bars->empty_x[xs]);
          if (++ds == kSpDenseStages) { ds = 0; dph ^= 1; }
          if (++xs == kSpXStages) { xs = 0; xph ^= 1; }
        }
        tc_commit(&bars->tmem_full[ab]);
      }
    }
  } else if (warp < kSpDrWarp0) {
    // ===== converters: values + meta -> dense SW128 tile =====
    // thread -> 16-byte output chunk j (8 columns = 2 groups) of atom a, rows rb + 8 i: a half-warp reads one row's
    // 128 value bytes and a quarter-warp writes one 128-byte swizzled row of one atom (both conflict-free)
    const int ct = threadIdx.x - kSpCvtWarp0 * 32;
    const int j = ct & 7, a = (ct >> 3) & 1, rb = ct >> 4;
    int rs = 0, ds = 0; uint32_t rph = 0, dph = 0;
    for (int u = blockIdx.x; u < p.nunits; u += gridDim.x) {
      const SpUnit w = sp_unit(p, u);
      for (int ks = w.ks0; ks < w.ks1; ++ks) {
        mbar_wait(&bars->full_raw[rs], rph);
        mbar_wait(&bars->empty_dense[ds], dph ^ 1);
        const uint8_t* sv = rring + rs * kSpRawStage;
        const uint8_t* sm = sv + kSpValBytes;
        uint8_t* sd = dring + ds * kSpDenseStage + a * kSpAtom;
#pragma unroll 4
        for (int i = 0; i < kSpRows / 8; ++i) {
          const int r = rb + 8 * i;
          const uint2 v = *reinterpret_cast<const uint2*>(sv + r * 128 + a * 64 + j * 8);
          const uint32_t m = sm[r * 16 + a * 8 + j];
          const uint64_t g0 = sp_expand_group(v.x, m & 15u), g1 = sp_expand_group(v.y, m >> 4);
          *reinterpret_cast<uint4*>(sd + r * 128 + ((j ^ (r & 7)) << 4)) =
              make_uint4((uint32_t)g0, (uint32_t)(g0 >> 32), (uint32_t)g1, (uint32_t)(g1 >> 32));
        }
        mbar_arrive(&bars->empty_raw[rs]);
        fence_proxy_async_smem();
        mbar_arrive(&bars->conv[ds]);
        if (++rs == kSpRawStages) { rs = 0; rph ^= 1; }
        if (++ds == kSpDenseStages) { ds = 0; dph ^= 1; }
      }
    }
  } else {
    // ===== drain =====
    const int q = warp & 3;                 // TMEM lane quarter this warp may touch
    const int row = q * 32 + lane;
    const int dt = threadIdx.x - kSpDrWarp0 * 32;
    uint16_t* y = reinterpret_cast<uint16_t*>(p.y);
    const uint16_t* bias = reinterpret_cast<const uint16_t*>(p.bias);
    int it = 0;
    for (int u = blockIdx.x; u < p.nunits; u += gridDim.x, ++it) {
      const SpUnit w = sp_unit(p, u);
      const int ab = it & 1;
      const int r = w.n0 + row;
      const float b = (bias && r < p.R) ? sp_float<T>(bias[r]) : 0.f;
      float* part = p.S > 1 ? p.part + ((size_t)w.tile * p.S + w.s) * (size_t)p.N * kSpRows : nullptr;
      mbar_wait(&bars->tmem_full[ab], (it >> 1) & 1);
      tc_fence_after();
      for (int c0 = 0; c0 < p.N; c0 += 32) {
        uint32_t v[32];
        tc_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + ab * p.acc_cols + c0, v);
        tc_wait_ld();
        if (part) {
#pragma unroll
          for (int e = 0; e < 32; ++e)
            if (c0 + e < p.N) part[(size_t)(c0 + e) * kSpRows + row] = __uint_as_float(v[e]);
        } else if (r < p.R) {
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const int t = w.t0 + c0 + e;
            if (c0 + e < p.N && t < p.T) y[(int64_t)t * p.ldy + r] = sp_round<T>(__uint_as_float(v[e]) + b);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars->tmem_empty[ab]);
      if (part) {
        __threadfence();
        asm volatile("bar.sync 1, %0;" :: "n"(kSpDrThreads) : "memory");
        if (dt == 0) bars->last = atomicAdd(p.tickets + w.tile, 1u) == (unsigned)(p.S - 1);
        asm volatile("bar.sync 1, %0;" :: "n"(kSpDrThreads) : "memory");
        if (bars->last) {
          __threadfence();
          const float* base = p.part + (size_t)w.tile * p.S * p.N * kSpRows + row;
          const size_t split_stride = (size_t)p.N * kSpRows;
          const int ncols = p.T - w.t0 < p.N ? p.T - w.t0 : p.N;
          if (r < p.R) {
            // 4 columns x 8 splits of loads in flight per step (the partials are in another SM's L2 slice); each column
            // is still summed in split order
            for (int c0 = 0; c0 < ncols; c0 += 4) {
              float acc[4] = {0.f, 0.f, 0.f, 0.f};
              for (int s0 = 0; s0 < p.S; s0 += 8) {
                float v[4][8];
#pragma unroll
                for (int cc = 0; cc < 4; ++cc)
#pragma unroll
                  for (int ss = 0; ss < 8; ++ss) {       // clamped: every address is inside this tile's partials
                    const int sc = min(s0 + ss, p.S - 1), ccl = min(c0 + cc, ncols - 1);
                    v[cc][ss] = __ldcg(base + (size_t)sc * split_stride + (size_t)ccl * kSpRows);
                  }
#pragma unroll
                for (int cc = 0; cc < 4; ++cc)
#pragma unroll
                  for (int ss = 0; ss < 8; ++ss)
                    if (s0 + ss < p.S) acc[cc] = (s0 + ss == 0) ? v[cc][ss] : acc[cc] + v[cc][ss];
              }
#pragma unroll
              for (int cc = 0; cc < 4; ++cc)
                if (c0 + cc < ncols) y[(int64_t)(w.t0 + c0 + cc) * p.ldy + r] = sp_round<T>(acc[cc] + b);
            }
          }
          if (dt == 0) p.tickets[w.tile] = 0u;
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(2 * p.acc_cols) : "memory");
  }
}

// ---- K24 / K25: one thread per 16-column word (4 groups) --------------------------------------------------------------
__device__ __forceinline__ void sp_load16(const uint16_t* src, bool vec, uint16_t* e) {
  if (vec) {
    const uint4 a = ld_stream(src), b = ld_stream(src + 8);
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int i = 0; i < 8; ++i) { e[2 * i] = (uint16_t)w[i]; e[2 * i + 1] = (uint16_t)(w[i] >> 16); }
  } else {
#pragma unroll
    for (int i = 0; i < 16; ++i) e[i] = src[i];
  }
}

template <bool kVec>
__global__ void __launch_bounds__(256)
sparse24_compress_kernel(const uint16_t* __restrict__ W, int64_t ldw, int R, int wpr, uint16_t* __restrict__ vals,
                         int64_t ldv, uint16_t* __restrict__ meta, int64_t ldm, int* status) {
  const int64_t total = (int64_t)R * wpr;
  bool bad = false;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(idx / wpr), wd = (int)(idx - (int64_t)r * wpr);
    uint16_t e[16];
    sp_load16(W + r * ldw + 16 * wd, kVec, e);
    uint32_t out[4], mw = 0;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      uint32_t kept = 0;
#pragma unroll
      for (int i = 0; i < 4; ++i) kept |= (uint32_t)((e[4 * g + i] & 0x7fffu) != 0) << i;     // +-0 pruned, NaN kept
      bad |= __popc(kept) > 2;
      uint32_t sel = kept;
#pragma unroll
      for (int i = 0; i < 4; ++i)                                 // pad with the lowest zero positions
        if (__popc(sel) < 2 && !((sel >> i) & 1u)) sel |= 1u << i;
      const uint32_t i0 = __ffs(sel) - 1, i1 = 31 - __clz(sel);
      uint32_t v0 = 0, v1 = 0;                                    // padded slots store +0
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint32_t ev = ((kept >> i) & 1u) ? e[4 * g + i] : 0u;
        v0 = i == (int)i0 ? ev : v0;
        v1 = i == (int)i1 ? ev : v1;
      }
      out[g] = v0 | (v1 << 16);
      mw |= (i0 | (i1 << 2)) << (4 * g);
    }
    uint16_t* dv = vals + r * ldv + 8 * wd;
    if (kVec) {
      st_stream(dv, make_uint4(out[0], out[1], out[2], out[3]));
    } else {
#pragma unroll
      for (int g = 0; g < 4; ++g) { dv[2 * g] = (uint16_t)out[g]; dv[2 * g + 1] = (uint16_t)(out[g] >> 16); }
    }
    meta[r * ldm + wd] = (uint16_t)mw;
  }
  if (__syncthreads_or(bad) && threadIdx.x == 0) atomicOr(status, VLMC_NOT_2OF4);
}

// K27: the kept set read from a bool mask instead of W's non-zeros.  Exactly two kept per group, else VLMC_NOT_2OF4;
// the values keep W's bits at the kept positions (+-0, NaN and inf included).
__device__ __forceinline__ void sp_load16_mask(const uint8_t* src, bool vec, uint32_t* kept4) {
  uint8_t b[16];
  if (vec) {
    const uint4 a = ld_stream(src);
    const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int i = 0; i < 16; ++i) b[i] = (uint8_t)(w[i / 4] >> (8 * (i % 4)));
  } else {
#pragma unroll
    for (int i = 0; i < 16; ++i) b[i] = src[i];
  }
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    uint32_t k = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) k |= (uint32_t)(b[4 * g + i] != 0) << i;
    kept4[g] = k;
  }
}

template <bool kVec>
__global__ void __launch_bounds__(256)
sparse24_compress_masked_kernel(const uint16_t* __restrict__ W, int64_t ldw, const uint8_t* __restrict__ mask,
                                int64_t ldk, int R, int wpr, uint16_t* __restrict__ vals, int64_t ldv,
                                uint16_t* __restrict__ meta, int64_t ldm, int* status) {
  const int64_t total = (int64_t)R * wpr;
  bool bad = false;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(idx / wpr), wd = (int)(idx - (int64_t)r * wpr);
    uint16_t e[16];
    uint32_t kept[4];
    sp_load16(W + r * ldw + 16 * wd, kVec, e);
    sp_load16_mask(mask + r * ldk + 16 * wd, kVec, kept);
    uint32_t out[4], mw = 0;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      bad |= __popc(kept[g]) != 2;
      const uint32_t sel = kept[g] ? kept[g] : 1u;
      const uint32_t i0 = __ffs(sel) - 1, i1 = 31 - __clz(sel);
      uint32_t v0 = 0, v1 = 0;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        v0 = i == (int)i0 ? e[4 * g + i] : v0;
        v1 = i == (int)i1 ? e[4 * g + i] : v1;
      }
      out[g] = v0 | (v1 << 16);
      mw |= (i0 | (i1 << 2)) << (4 * g);
    }
    uint16_t* dv = vals + r * ldv + 8 * wd;
    if (kVec) {
      st_stream(dv, make_uint4(out[0], out[1], out[2], out[3]));
    } else {
#pragma unroll
      for (int g = 0; g < 4; ++g) { dv[2 * g] = (uint16_t)out[g]; dv[2 * g + 1] = (uint16_t)(out[g] >> 16); }
    }
    meta[r * ldm + wd] = (uint16_t)mw;
  }
  if (__syncthreads_or(bad) && threadIdx.x == 0) atomicOr(status, VLMC_NOT_2OF4);
}

template <bool kVec>
__global__ void __launch_bounds__(256)
sparse24_decompress_kernel(const uint16_t* __restrict__ vals, int64_t ldv, const uint16_t* __restrict__ meta, int64_t ldm,
                           int R, int wpr, uint16_t* __restrict__ W, int64_t ldw) {
  const int64_t total = (int64_t)R * wpr;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(idx / wpr), wd = (int)(idx - (int64_t)r * wpr);
    const uint16_t* sv = vals + r * ldv + 8 * wd;
    uint32_t pair[4];
    if (kVec) {
      const uint4 v = ld_stream(sv);
      pair[0] = v.x; pair[1] = v.y; pair[2] = v.z; pair[3] = v.w;
    } else {
#pragma unroll
      for (int g = 0; g < 4; ++g) pair[g] = (uint32_t)sv[2 * g] | ((uint32_t)sv[2 * g + 1] << 16);
    }
    const uint32_t mw = __ldg(meta + r * ldm + wd);
    uint64_t o[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) o[g] = sp_expand_group(pair[g], (mw >> (4 * g)) & 15u);
    uint16_t* dw = W + r * ldw + 16 * wd;
    if (kVec) {
      st_stream(dw, make_uint4((uint32_t)o[0], (uint32_t)(o[0] >> 32), (uint32_t)o[1], (uint32_t)(o[1] >> 32)));
      st_stream(dw + 8, make_uint4((uint32_t)o[2], (uint32_t)(o[2] >> 32), (uint32_t)o[3], (uint32_t)(o[3] >> 32)));
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) dw[i] = (uint16_t)(o[i >> 2] >> (16 * (i & 3)));
    }
  }
}

static int sp_grid(int64_t words) {
  const int64_t want = (words + 255) / 256, cap = (int64_t)kNumSMs * 8;
  return (int)(want < cap ? want : cap);
}

// tokens per tile, token tiles, k splits: the split count minimises (waves of units) x (slices per unit) over the SMs
struct SpPlan { int N, ntt, nrt, nsl, S; };
static SpPlan sp_plan(int64_t T, int R, int C) {
  SpPlan pl;
  const int64_t n16 = (T + 15) / 16 * 16;
  pl.N = (int)(n16 < kSpMaxN ? n16 : kSpMaxN);
  pl.ntt = (int)((T + pl.N - 1) / pl.N);
  pl.nrt = (R + kSpRows - 1) / kSpRows;
  pl.nsl = (C + kSpK - 1) / kSpK;
  pl.S = 1;
  const int64_t tiles = (int64_t)pl.ntt * pl.nrt;
  if (tiles <= kSpMaxTickets) {
    int64_t best = (tiles + kNumSMs - 1) / kNumSMs * pl.nsl;
    for (int s = 2; s <= pl.nsl && s <= kSpMaxSplit; ++s) {
      const int64_t cost = (tiles * s + kNumSMs - 1) / kNumSMs * ((pl.nsl + s - 1) / s);
      if (cost < best) { best = cost; pl.S = s; }
    }
  }
  return pl;
}

size_t sparse24_linear_workspace_bytes(int64_t T, int R, int C) {
  if (T < 1 || R < 1 || C < 16) return VLMC_WS_COUNTER_BYTES;
  const SpPlan pl = sp_plan(T, R, C);
  if (pl.S == 1) return VLMC_WS_COUNTER_BYTES;
  return VLMC_WS_COUNTER_BYTES + (size_t)pl.ntt * pl.nrt * pl.S * pl.N * kSpRows * sizeof(float);
}

static int sp_map(CUtensorMap* map, CUtensorMapDataType type, const void* base, uint64_t inner, uint64_t outer, int64_t ld,
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
static int sp_launch(const CUtensorMap& xmap, const CUtensorMap& vmap, const CUtensorMap& mmap, const SpParams& p,
                     uint32_t idesc, cudaStream_t st) {
  auto kern = sparse24_linear_kernel<T>;
  static bool attr_set = false;
  if (!attr_set) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSpSmem) != cudaSuccess)
      return check_launch();
    attr_set = true;
  }
  const int grid = p.nunits < kNumSMs ? p.nunits : kNumSMs;
  kern<<<grid, kSpThreads, kSpSmem, st>>>(xmap, vmap, mmap, p, idesc);
  return check_launch();
}

static bool sp_aligned16(const void* ptr) { return ((uintptr_t)ptr & 15) == 0; }

}  // namespace vlmc

extern "C" int vlmc_sparse24_compress(const void* W, int dtype, int R, int C, int64_t ldw, void* values, int64_t ldv,
                                      uint16_t* meta, int64_t ldm, int* status, void* stream) {
  using namespace vlmc;
  if (!W || !values || !meta || !status || R < 1 || C < 16 || C % 16 != 0 || ldw < C || ldv < C / 2 || ldm < C / 16)
    return VLMC_ERR_BAD_ARG;
  if (dtype != VLMC_F16 && dtype != VLMC_BF16) return dtype == VLMC_F32 ? VLMC_ERR_UNSUPPORTED : VLMC_ERR_BAD_ARG;
  if (!is_device_ptr(W) || !is_device_ptr(values) || !is_device_ptr(meta) || !is_device_ptr(status))
    return VLMC_ERR_NOT_DEVICE;
  cudaStream_t st = (cudaStream_t)stream;
  if (cudaMemsetAsync(status, 0, sizeof(int), st) != cudaSuccess) return check_launch();
  const int wpr = C / 16;
  const bool vec = sp_aligned16(W) && sp_aligned16(values) && ldw % 8 == 0 && ldv % 8 == 0;
  const int grid = sp_grid((int64_t)R * wpr);
  const uint16_t* w16 = static_cast<const uint16_t*>(W);
  uint16_t* v16 = static_cast<uint16_t*>(values);
  if (vec) sparse24_compress_kernel<true><<<grid, 256, 0, st>>>(w16, ldw, R, wpr, v16, ldv, meta, ldm, status);
  else sparse24_compress_kernel<false><<<grid, 256, 0, st>>>(w16, ldw, R, wpr, v16, ldv, meta, ldm, status);
  return check_launch();
}

extern "C" int vlmc_sparse24_compress_masked(const void* W, int dtype, int R, int C, int64_t ldw, const uint8_t* keep_mask,
                                             int64_t ldk, void* values, int64_t ldv, uint16_t* meta, int64_t ldm, int* status,
                                             void* stream) {
  using namespace vlmc;
  if (!W || !keep_mask || !values || !meta || !status || R < 1 || C < 16 || C % 16 != 0 || ldw < C || ldk < C ||
      ldv < C / 2 || ldm < C / 16)
    return VLMC_ERR_BAD_ARG;
  if (dtype != VLMC_F16 && dtype != VLMC_BF16) return dtype == VLMC_F32 ? VLMC_ERR_UNSUPPORTED : VLMC_ERR_BAD_ARG;
  if (!is_device_ptr(W) || !is_device_ptr(keep_mask) || !is_device_ptr(values) || !is_device_ptr(meta) ||
      !is_device_ptr(status))
    return VLMC_ERR_NOT_DEVICE;
  cudaStream_t st = (cudaStream_t)stream;
  if (cudaMemsetAsync(status, 0, sizeof(int), st) != cudaSuccess) return check_launch();
  const int wpr = C / 16;
  const bool vec = sp_aligned16(W) && sp_aligned16(values) && sp_aligned16(keep_mask) && ldw % 8 == 0 && ldv % 8 == 0 &&
                   ldk % 16 == 0;
  const int grid = sp_grid((int64_t)R * wpr);
  const uint16_t* w16 = static_cast<const uint16_t*>(W);
  uint16_t* v16 = static_cast<uint16_t*>(values);
  if (vec) sparse24_compress_masked_kernel<true><<<grid, 256, 0, st>>>(w16, ldw, keep_mask, ldk, R, wpr, v16, ldv, meta, ldm, status);
  else sparse24_compress_masked_kernel<false><<<grid, 256, 0, st>>>(w16, ldw, keep_mask, ldk, R, wpr, v16, ldv, meta, ldm, status);
  return check_launch();
}

extern "C" int vlmc_sparse24_decompress(const void* values, int dtype, int R, int C, int64_t ldv, const uint16_t* meta,
                                        int64_t ldm, void* W, int64_t ldw, void* stream) {
  using namespace vlmc;
  if (!W || !values || !meta || R < 1 || C < 16 || C % 16 != 0 || ldw < C || ldv < C / 2 || ldm < C / 16)
    return VLMC_ERR_BAD_ARG;
  if (dtype != VLMC_F16 && dtype != VLMC_BF16) return dtype == VLMC_F32 ? VLMC_ERR_UNSUPPORTED : VLMC_ERR_BAD_ARG;
  if (!is_device_ptr(W) || !is_device_ptr(values) || !is_device_ptr(meta)) return VLMC_ERR_NOT_DEVICE;
  cudaStream_t st = (cudaStream_t)stream;
  const int wpr = C / 16;
  const bool vec = sp_aligned16(W) && sp_aligned16(values) && ldw % 8 == 0 && ldv % 8 == 0;
  const int grid = sp_grid((int64_t)R * wpr);
  const uint16_t* v16 = static_cast<const uint16_t*>(values);
  uint16_t* w16 = static_cast<uint16_t*>(W);
  if (vec) sparse24_decompress_kernel<true><<<grid, 256, 0, st>>>(v16, ldv, meta, ldm, R, wpr, w16, ldw);
  else sparse24_decompress_kernel<false><<<grid, 256, 0, st>>>(v16, ldv, meta, ldm, R, wpr, w16, ldw);
  return check_launch();
}

extern "C" int vlmc_sparse24_linear_forward(const void* x, int dtype, int64_t T, int C, int64_t ldx, const void* values,
                                            int64_t ldv, const uint16_t* meta, int64_t ldm, int R, const void* bias, void* y,
                                            int64_t ldy, void* ws, size_t ws_bytes, void* stream) {
  using namespace vlmc;
  if (!x || !values || !meta || !y || !ws || T < 0 || R < 1 || C < 16 || C % 16 != 0 || ldx < C || ldv < C / 2 ||
      ldm < C / 16 || ldy < R)
    return VLMC_ERR_BAD_ARG;
  if (dtype != VLMC_F16 && dtype != VLMC_BF16) return dtype == VLMC_F32 ? VLMC_ERR_UNSUPPORTED : VLMC_ERR_BAD_ARG;
  if (T == 0) return VLMC_OK;
  if (T > 0x7fffffff) return VLMC_ERR_UNSUPPORTED;
  // TMA: 16-byte aligned bases and row pitches
  if (ldx % 8 != 0 || ldv % 8 != 0 || ldm % 8 != 0 || !sp_aligned16(x) || !sp_aligned16(values) || !sp_aligned16(meta))
    return VLMC_ERR_UNSUPPORTED;
  if (!is_device_ptr(x) || !is_device_ptr(values) || !is_device_ptr(meta) || !is_device_ptr(y) || !is_device_ptr(ws) ||
      (bias && !is_device_ptr(bias)))
    return VLMC_ERR_NOT_DEVICE;
  if (ws_bytes < sparse24_linear_workspace_bytes(T, R, C)) return VLMC_ERR_WORKSPACE;

  const SpPlan pl = sp_plan(T, R, C);
  const CUtensorMapDataType dt = dtype == VLMC_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  CUtensorMap xmap, vmap, mmap;
  int rc = sp_map(&xmap, dt, x, (uint64_t)C, (uint64_t)T, ldx, 64, (uint32_t)pl.N, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  rc = sp_map(&vmap, dt, values, (uint64_t)(C / 2), (uint64_t)R, ldv, kSpK / 2, kSpRows, CU_TENSOR_MAP_SWIZZLE_NONE);
  if (rc) return rc;
  rc = sp_map(&mmap, CU_TENSOR_MAP_DATA_TYPE_UINT16, meta, (uint64_t)(C / 16), (uint64_t)R, ldm, kSpK / 16, kSpRows,
              CU_TENSOR_MAP_SWIZZLE_NONE);
  if (rc) return rc;

  SpParams p;
  p.y = y; p.ldy = ldy; p.bias = bias;
  p.tickets = static_cast<unsigned int*>(ws);
  p.part = reinterpret_cast<float*>(static_cast<uint8_t*>(ws) + VLMC_WS_COUNTER_BYTES);
  p.T = (int)T; p.R = R; p.C = C; p.N = pl.N; p.nrt = pl.nrt; p.S = pl.S; p.nsl = pl.nsl;
  const int64_t nunits = (int64_t)pl.ntt * pl.nrt * pl.S;
  if (nunits > 0x7fffffff) return VLMC_ERR_UNSUPPORTED;
  p.nunits = (int)nunits;
  uint32_t cols = 32;
  while ((int)cols < pl.N) cols <<= 1;
  p.acc_cols = cols;
  // instruction descriptor (cute::UMMA::InstrDescriptor): fp32 accumulate, A (weights) and B (tokens) K-major, M = 128
  const uint32_t fmt = dtype == VLMC_F16 ? 0u : 1u;
  const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(pl.N >> 3) << 17) | ((uint32_t)(kSpRows >> 4) << 24);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == VLMC_F16) return sp_launch<__half>(xmap, vmap, mmap, p, idesc, st);
  return sp_launch<__nv_bfloat16>(xmap, vmap, mmap, p, idesc, st);
}
