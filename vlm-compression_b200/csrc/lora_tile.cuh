// The streaming tile loop K14 (masked merge, in place) and K15 (effective weight, out of place) share; sparse24.cuh holds
// its compressed-weight variant (K28, K30).
//
// A 128-thread CTA walks a contiguous span of units of kLtUnitRows rows x 1024 columns (16 bytes of W per thread and row).
// The rank x 1024 slice of lora_A it needs is staged in shared memory when the span enters a new column tile (once or twice per CTA) as float4 planes (conflict-free 16-byte reads), so a
// thread holds no A values in registers (the register form kept rank x 8 floats per thread: 94-128 registers, 4-5 CTAs
// of 128 threads per SM and one to four rows in flight - 0.40 / 0.63 of the HBM roofline).  Four rows are in flight per
// thread; per rank step one A vector is read from shared memory and applied to all four rows, which keeps the shared
// memory traffic at a quarter of a row-at-a-time loop.  Per output element the products are still added in ascending k
// with one fma each, exactly like the register form (bit-identical results).
#pragma once
#include "common.cuh"

namespace vlmc {

constexpr int kLtThreads = 128;
constexpr int kLtRows = 4;              // rows in flight per thread
constexpr int kLtUnitRows = 4;          // rows per work unit: a CTA takes a CONTIGUOUS span of units (column tile major, row
                                        // blocks fastest), so A is staged once per span, not per unit, and small matrices still
                                        // split into thousands of units (4096 x 4096: 4096 units for ~700 resident CTAs)
constexpr int kLtMaxRank = 16;

template <typename T> constexpr size_t lt_smem_bytes(int rank) {
  return (size_t)rank * Elem<T>::kVec * kLtThreads * sizeof(float);
}

// ---- the reference's roundings of the effective weight (lora.py:364-375), shared by K15 and K23 ----
template <typename T> __device__ __forceinline__ float round_dt(float v);
template <> __device__ __forceinline__ float round_dt<float>(float v) { return v; }
template <> __device__ __forceinline__ float round_dt<__half>(float v) { return __half2float(__float2half_rn(v)); }
template <> __device__ __forceinline__ float round_dt<__nv_bfloat16>(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }

template <typename T> __device__ __forceinline__ float2 round_dt2(float2 v);
template <> __device__ __forceinline__ float2 round_dt2<float>(float2 v) { return v; }
template <> __device__ __forceinline__ float2 round_dt2<__half>(float2 v) { return __half22float2(__floats2half2_rn(v.x, v.y)); }
template <> __device__ __forceinline__ float2 round_dt2<__nv_bfloat16>(float2 v) { return __bfloat1622float2(__floats2bfloat162_rn(v.x, v.y)); }

// f[V] (the weights, widened) <- the effective weight from the rank-r dot acc and the mask bytes mb:
//   sparse:  round(W + d) * mask      not sparse:  round(W * mask + d)      d = round(round(acc) * scaling)
// (B @ A).to(dtype) -> * scaling (rounded in dtype) -> W + . (rounded in dtype) -> * mask (exact).  The three roundings
// run on PAIRS (packed f32 -> 2 x 16-bit -> f32 conversions are full rate; the scalar F2F form is a quarter-rate
// instruction and made K15 conversion-bound: 6 per weight).
template <typename T, int V = Elem<T>::kVec>
__device__ __forceinline__ void lt_effective(float (&f)[V], const float (&acc)[V], const uint32_t (&mb)[2], float scaling,
                                             int sparse) {
#pragma unroll
  for (int e = 0; e < V; e += 2) {
    const bool k0 = (mb[e / 4] >> (8 * (e % 4))) & 0xffu, k1 = (mb[(e + 1) / 4] >> (8 * ((e + 1) % 4))) & 0xffu;
    float2 d = round_dt2<T>(make_float2(acc[e], acc[e + 1]));
    d = round_dt2<T>(make_float2(__fmul_rn(d.x, scaling), __fmul_rn(d.y, scaling)));
    float2 r;
    if (sparse) {
      r = round_dt2<T>(make_float2(__fadd_rn(f[e], d.x), __fadd_rn(f[e + 1], d.y)));
      f[e] = k0 ? r.x : 0.f;
      f[e + 1] = k1 ? r.y : 0.f;
    } else {
      r = round_dt2<T>(make_float2(__fadd_rn(k0 ? f[e] : 0.f, d.x), __fadd_rn(k1 ? f[e + 1] : 0.f, d.y)));
      f[e] = r.x;
      f[e + 1] = r.y;
    }
  }
}

// stage A[0:rank, col0 : col0 + 1024) -> sA[(kk * V/4 + q) * 128 + t] = A[kk][col0 + t * V + 4q .. +3]  (zero past C)
template <typename T>
__device__ __forceinline__ void lt_stage_a(float4* sA, const float* __restrict__ A, int rank, int C, int col0) {
  constexpr int V = Elem<T>::kVec;
  const int t = threadIdx.x;
  const int col = col0 + t * V;
  for (int kk = 0; kk < rank; ++kk)
#pragma unroll
    for (int q = 0; q < V / 4; ++q) {
      float4 av = make_float4(0.f, 0.f, 0.f, 0.f);
      if (col + 4 * q < C) av = __ldg(reinterpret_cast<const float4*>(A + (int64_t)kk * C + col + 4 * q));
      sA[(kk * (V / 4) + q) * kLtThreads + t] = av;
    }
}

// K14's combine (lora.py:384-387 + train.py:634-637): f[V] <- keep ? round(W + (BA * scaling)) : (remask ? 0 : W), the
// rounding to W's dtype left to the store.  (BA * scaling) * mask, then W += : two separately rounded fp32 ops, no FMA
// contraction.  Shared by the dense merge (K14) and the compressed one (K30).
template <typename T, int V = Elem<T>::kVec>
__device__ __forceinline__ void lt_merge(float (&f)[V], const float (&acc)[V], const uint32_t (&mb)[2], float scaling,
                                         int remask) {
#pragma unroll
  for (int e = 0; e < V; ++e) {
    const bool keep = (mb[e / 4] >> (8 * (e % 4))) & 0xffu;
    const float delta = __fmul_rn(acc[e], scaling);
    const float merged = __fadd_rn(f[e], delta);
    f[e] = keep ? merged : (remask ? 0.f : f[e]);
  }
}

// acc[r][.] = sum_k B[row0 + r][k] A[k][this thread's V columns] for the kLtRows rows from row0 (rows past row_end repeat
// the last row and are not stored).  The rank-r dot on packed fp32 FMAs (fma.rn.f32x2, sm_100): two IEEE fmas per
// instruction, per lane identical to fmaf - the loop is instruction-issue bound (8 fmas per weight at r = 8), not HBM
// bound, without them.  k ascending, so every caller gets the same bits for the same (B, A).
template <typename T>
__device__ __forceinline__ void lt_dot(float2 (&acc)[kLtRows][Elem<T>::kVec / 2], const float* __restrict__ B, int rank,
                                       int row0, int row_end, const float4* sA) {
  constexpr int V = Elem<T>::kVec;
  const int t = threadIdx.x;
#pragma unroll
  for (int r = 0; r < kLtRows; ++r)
#pragma unroll
    for (int e = 0; e < V / 2; ++e) acc[r][e] = make_float2(0.f, 0.f);
  const float* brow[kLtRows];
#pragma unroll
  for (int r = 0; r < kLtRows; ++r) brow[r] = B + (int64_t)(row0 + r < row_end ? row0 + r : row_end - 1) * rank;
#pragma unroll 4
  for (int kk = 0; kk < rank; ++kk) {
    float2 a[V / 2];
#pragma unroll
    for (int q = 0; q < V / 4; ++q) {
      const float4 av = sA[(kk * (V / 4) + q) * kLtThreads + t];
      a[2 * q] = make_float2(av.x, av.y);
      a[2 * q + 1] = make_float2(av.z, av.w);
    }
#pragma unroll
    for (int r = 0; r < kLtRows; ++r) {
      const float b = __ldg(brow[r] + kk);
      const float2 b2 = make_float2(b, b);
#pragma unroll
      for (int e = 0; e < V / 2; ++e) acc[r][e] = __ffma2_rn(b2, a[e], acc[r][e]);      // k ascending, like SGEMM
    }
  }
}

// rows [row_begin, row_end) of this thread's 16-byte column.  comb(f, acc, mb) rewrites f[V] from the weights f, the
// rank-r dot acc = sum_k B[row][k] A[k][col..] and the mask bytes mb, then the vector is stored to out.
template <typename T, class Combine>
__device__ __forceinline__ void lt_rows(const T* __restrict__ W, int64_t ldw, T* __restrict__ out, int64_t ldo, int col,
                                        int row_begin, int row_end, const float* __restrict__ B, int rank,
                                        const uint8_t* __restrict__ mask, int64_t ldm, const float4* sA, Combine comb) {
  constexpr int V = Elem<T>::kVec;
  for (int row0 = row_begin; row0 < row_end; row0 += kLtRows) {
    uint4 wv[kLtRows];
    uint2 mv[kLtRows];
#pragma unroll
    for (int r = 0; r < kLtRows; ++r) {
      if (row0 + r < row_end) {
        wv[r] = ld_stream(W + (int64_t)(row0 + r) * ldw + col);
        const uint8_t* mp = mask + (int64_t)(row0 + r) * ldm + col;
        if (V == 8) mv[r] = *reinterpret_cast<const uint2*>(mp);
        else mv[r] = make_uint2(*reinterpret_cast<const uint32_t*>(mp), 0u);
      }
    }
    float2 acc[kLtRows][V / 2];
    lt_dot<T>(acc, B, rank, row0, row_end, sA);
#pragma unroll
    for (int r = 0; r < kLtRows; ++r) {
      if (row0 + r >= row_end) break;
      float f[V], ac[V];
      Elem<T>::unpack(wv[r], f);
#pragma unroll
      for (int e = 0; e < V / 2; ++e) { ac[2 * e] = acc[r][e].x; ac[2 * e + 1] = acc[r][e].y; }
      const uint32_t mb[2] = {mv[r].x, mv[r].y};
      comb(f, ac, mb);
      st_stream(out + (int64_t)(row0 + r) * ldo + col, Elem<T>::pack(f));
    }
  }
}

}  // namespace vlmc
