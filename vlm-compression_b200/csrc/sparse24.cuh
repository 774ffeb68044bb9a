// Device helpers of the compressed 2:4 format (include/vlmc.h, "Compressed 2:4 weights"), shared by K24-K26
// (sparse24.cu) and the SparseLoRA kernels that read it (K28-K30).
#pragma once
#include "lora_tile.cuh"

namespace vlmc {

// one 4-column group: the value pair (first kept in the low half) and its 4-bit index nibble -> four 16-bit slots
__device__ __forceinline__ uint64_t sp_expand_group(uint32_t pair, uint32_t nib) {
  const uint32_t i0 = nib & 3u, i1 = (nib >> 2) & 3u;
  return ((uint64_t)(pair & 0xffffu) << (16 * i0)) | ((uint64_t)(pair >> 16) << (16 * i1));
}

// the inverse on four 16-bit slots: the pair stored at the nibble's two indices
__device__ __forceinline__ uint32_t sp_gather_group(uint64_t slots, uint32_t nib) {
  const uint32_t i0 = nib & 3u, i1 = (nib >> 2) & 3u;
  return (uint32_t)((slots >> (16 * i0)) & 0xffffu) | ((uint32_t)((slots >> (16 * i1)) & 0xffffu) << 16);
}

// the four mask bytes (1 = kept) of a group, in the layout the dense kernels read a bool mask in
__device__ __forceinline__ uint32_t sp_nibble_mask(uint32_t nib) {
  return (1u << (8 * (nib & 3u))) | (1u << (8 * ((nib >> 2) & 3u)));
}

// The kept set of a mask-driven compression (K27) is exactly the mask, so meta IS the mask: columns [col, col + V) of a
// row as mask bytes (V = 4 or 8, col % V == 0).  Group g of word j sits at bits [4g, 4g + 4): the shift is col % 16.
template <int V>
__device__ __forceinline__ void sp_meta_mask(const uint16_t* __restrict__ meta, int64_t ldm, int row, int col,
                                             uint32_t (&mb)[2]) {
  const uint32_t w = __ldg(meta + (int64_t)row * ldm + col / 16) >> (col & 15);
  mb[0] = sp_nibble_mask(w & 15u);
  mb[1] = V == 8 ? sp_nibble_mask((w >> 4) & 15u) : 0u;
}

// lt_rows (lora_tile.cuh) on a compressed weight: per row and 8 columns it loads 4 values (8 bytes) and 8 bits of meta,
// expands them into the dense 16-byte vector and the 8 mask bytes decompress() and the bool mask would give, and runs
// the same rank-r dot (lt_dot) and the same combine on them - so every result is bit-identical to the dense kernel's
// on (decompress(values, meta), mask from meta).  kInPlace: the combined vector goes back into the values at the
// meta's indices (K30); otherwise the dense vector is stored to out (K28).
template <typename T, bool kInPlace, class Combine>
__device__ __forceinline__ void lt_rows_sp24(uint16_t* values, int64_t ldv, const uint16_t* __restrict__ meta, int64_t ldm,
                                             T* __restrict__ out, int64_t ldo, int col, int row_begin, int row_end,
                                             const float* __restrict__ B, int rank, const float4* sA, Combine comb) {
  static_assert(Elem<T>::kVec == 8, "compressed 2:4 weights are 16-bit");
  constexpr int V = 8;
  for (int row0 = row_begin; row0 < row_end; row0 += kLtRows) {
    uint2 vv[kLtRows];
    uint32_t nb[kLtRows];
#pragma unroll
    for (int r = 0; r < kLtRows; ++r) {
      if (row0 + r < row_end) {
        const int64_t row = row0 + r;
        vv[r] = *reinterpret_cast<const uint2*>(values + row * ldv + col / 2);
        nb[r] = (uint32_t)(__ldg(meta + row * ldm + col / 16) >> (col & 15)) & 0xffu;
      }
    }
    float2 acc[kLtRows][V / 2];
    lt_dot<T>(acc, B, rank, row0, row_end, sA);
#pragma unroll
    for (int r = 0; r < kLtRows; ++r) {
      if (row0 + r >= row_end) break;
      const uint32_t n0 = nb[r] & 15u, n1 = nb[r] >> 4;
      const uint64_t g0 = sp_expand_group(vv[r].x, n0), g1 = sp_expand_group(vv[r].y, n1);
      float f[V], ac[V];
      Elem<T>::unpack(make_uint4((uint32_t)g0, (uint32_t)(g0 >> 32), (uint32_t)g1, (uint32_t)(g1 >> 32)), f);
#pragma unroll
      for (int e = 0; e < V / 2; ++e) { ac[2 * e] = acc[r][e].x; ac[2 * e + 1] = acc[r][e].y; }
      const uint32_t mb[2] = {sp_nibble_mask(n0), sp_nibble_mask(n1)};
      comb(f, ac, mb);
      const uint4 o = Elem<T>::pack(f);
      if (kInPlace) {
        *reinterpret_cast<uint2*>(values + (int64_t)(row0 + r) * ldv + col / 2) =
            make_uint2(sp_gather_group((uint64_t)o.x | ((uint64_t)o.y << 32), n0),
                       sp_gather_group((uint64_t)o.z | ((uint64_t)o.w << 32), n1));
      } else {
        st_stream(out + (int64_t)(row0 + r) * ldo + col, o);
      }
    }
  }
}

}  // namespace vlmc
