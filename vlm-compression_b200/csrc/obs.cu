// K11 + K12 + K13: the SparseGPT column-block OBS sweep.
//
// Replaces lavis/compression/pruners/sparsegpt_pruner.py:160-215 (fasterprune after the factorisation):
//   s = W^2 / diag(U)^2 ; importance_score = mean(s)                                           (:160-165)
//   for each 128-column block:                                                                  (:169)
//     unstructured: thresh = sort((W1^2/diag(U1)^2).flatten())[int(numel*p)] ; mask1 = tmp <= thresh  (:183-185) K11
//     n:m: every m-th column the n smallest of the group, on the already compensated W1         (:193-195)
//     128 sequential steps: q = masked w ; err = (w-q)/d ; W1[:, i:] -= err (x) U1[i, i:]        (:189-205) K12
//     W[:, i2:] -= Err1 @ U[i1:i2, i2:]                                                         (:210)     K13
// The reference issues ~8 launches per COLUMN (~90 k per down_proj) and one flatten-sort per block.  Here a block is
//   K11  obs_hist_kernel<0,1,2>  exact k-th smallest of the R x 128 block scores by an 11/11/10-bit radix select:
//                                per-CTA shared-memory histograms flushed to a global one, three stream-ordered
//                                passes, no sort and no host round trip.  (When rows are sharded over GPUs these
//                                three 8 KB histograms are the only data exchanged per block, SURVEY F6.)
//   K12  obs_sweep4_kernel       four weight rows per warp (8 lanes x 16 registers hold a row's 128 columns), the
//                                U1 tile in shared memory; the 128 sequential steps broadcast the pivot column by
//                                shuffle inside the lane group.  Writes the finished columns to the fp16/bf16
//                                weight, the fp32 working copy, Err1 and the keep mask.
//   K13  the lazy trailing update on the tensor cores: the 3xTF32 tcgen05 GEMM of gemm3x.cu (fp32-grade accuracy).
#include <stdlib.h>
#include <cooperative_groups.h>
#include "gemm3x.cuh"

namespace vlmc {

int launch_mean_finalize(const float* part, int n, double denom, float* out, cudaStream_t st);

constexpr int kOB = 128;            // column block (the reference's blocksize default, the only one the scripts use)
// Super-block schedule of the lazy update (:210).  The reference subtracts Err1 @ U[i1:i2, i2:] from ALL remaining
// columns after every 128-column block: a K = 128 GEMM that read-modify-writes the whole fp32 trailing matrix 86 times
// for down_proj (15.5 GB, the traffic that bounded K13 at 95 TFLOP/s logical).  Here kSB consecutive blocks form a
// super-block: after a block only the remaining columns of ITS super-block are updated (a small K = 128 GEMM), and the
// far columns receive the super-block's accumulated errors once, as ONE GEMM with K = kSB * 128 - a quarter of the
// passes over W32 and four times the arithmetic per byte.  Every output element still receives exactly the same
// products, summed in fp32 (3xTF32, 128-wide chunks added round-to-nearest); only the order of the chunk sums differs.
constexpr int kSBMax = 8;
constexpr int kErrLd = kSBMax * kOB;      // Err is [R, kErrLd]: block b of a super-block writes columns [slot * 128, slot * 128 + 128)
constexpr int kObsBins = 2048;
constexpr int kObsThreads = 256;
constexpr int kObsMaxM = 16;

typedef unsigned long long ull;

struct ObsHist { unsigned int h[3][kObsBins]; };

template <typename T> __device__ __forceinline__ T from_float(float v);
template <> __device__ __forceinline__ float from_float<float>(float v) { return v; }
template <> __device__ __forceinline__ __half from_float<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_float<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <typename T> __device__ __forceinline__ float to_float(T v);
template <> __device__ __forceinline__ float to_float<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_float<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float to_float<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

// W (dtype) -> fp32 working copy, dead input channels zeroed (sparsegpt_pruner.py:84-97)
template <typename T>
__global__ void obs_upcast_kernel(const T* __restrict__ W, int64_t ldw, float* __restrict__ W32, int R, int C,
                                  const uint8_t* __restrict__ dead) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const bool d = dead ? dead[c] != 0 : false;
  for (int r = blockIdx.y; r < R; r += gridDim.y)
    W32[(int64_t)r * C + c] = d ? 0.f : to_float<T>(W[(int64_t)r * ldw + c]);
}

// sum over the matrix of W^2 / diag(U)^2 (the reference's importance score numerator)
__global__ void obs_importance_kernel(const float* __restrict__ W32, int R, int C, const float* __restrict__ U,
                                      int64_t ldu, float* __restrict__ part) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  float s = 0.f;
  if (c < C) {
    const float d = U[(int64_t)c * ldu + c];
    const float d2 = __fmul_rn(d, d);
    for (int r = blockIdx.y; r < R; r += gridDim.y) {
      const float w = W32[(int64_t)r * C + c];
      s += __fdiv_rn(__fmul_rn(w, w), d2);
    }
  }
  __shared__ float red[8];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
    part[blockIdx.y * gridDim.x + blockIdx.x] = t;
  }
}

struct ObsParams {
  float* W32;          // [R, C] fp32 working copy
  void* Wout;          // weight tensor (dtype), receives the finished columns
  int64_t ldw;
  int R, C;
  const float* U;
  int64_t ldu;
  int i1, bs;          // column block [i1, i1 + bs)
  float* Err;          // [R, kErrLd], already offset to this block's slot
  uint8_t* keep;       // optional [R, ldm]
  int64_t ldm;
  unsigned int kth;    // unstructured: 1-indexed rank of the threshold value among the R*bs block scores
  int prune_n, prune_m;
  ObsHist* hist;       // this block's three histograms (zero on entry)
  const int* fail;     // optional device flag: non-zero = the factor U is invalid, leave W and the keep mask untouched
};

// score of one weight: w^2 / d^2 with the reference's roundings (:183); non-negative, so bit order = value order
__device__ __forceinline__ uint32_t obs_key(float w, float d2) {
  return __float_as_uint(__fdiv_rn(__fmul_rn(w, w), d2));
}

// bin holding the kk-th (1-indexed) entry of a global histogram and the count before it; every thread returns both
template <int NT>
__device__ void obs_find_bin(const unsigned int* __restrict__ gh, unsigned int kk, unsigned int* s_scan,
                             unsigned int& bin, unsigned int& before) {
  const int tid = threadIdx.x;
  constexpr int per = kObsBins / NT;
  unsigned int c[per];
  unsigned int local = 0;
#pragma unroll
  for (int j = 0; j < per; ++j) { c[j] = __ldcg(gh + tid * per + j); local += c[j]; }
  unsigned int incl = local;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
    if ((tid & 31) >= o) incl += t;
  }
  __syncthreads();
  if ((tid & 31) == 31) s_scan[tid >> 5] = incl;
  __syncthreads();
  unsigned int wbase = 0;
  for (int w = 0; w < (tid >> 5); ++w) wbase += s_scan[w];
  incl += wbase;
  const unsigned int excl = incl - local;
  __syncthreads();
  if (excl < kk && kk <= incl) {
    unsigned int run = excl;
#pragma unroll
    for (int j = 0; j < per; ++j) {
      if (kk <= run + c[j]) { s_scan[16] = tid * per + j; s_scan[17] = run; break; }
      run += c[j];
    }
  }
  __syncthreads();
  bin = s_scan[16];
  before = s_scan[17];
}

// K11 pass PASS: histogram of bits [21,32) / [10,21) / [0,10) of the block scores that match the bins chosen so far
template <int PASS>
__global__ void __launch_bounds__(kObsThreads)
obs_hist_kernel(const ObsParams p) {
  __shared__ unsigned int sh[kObsBins];
  __shared__ unsigned int s_scan[32];
  __shared__ float s_d2[kOB];
  const int tid = threadIdx.x;
  for (int b = tid; b < kObsBins; b += kObsThreads) sh[b] = 0;
  if (tid < kOB) {
    const float d = tid < p.bs ? p.U[(int64_t)(p.i1 + tid) * p.ldu + p.i1 + tid] : 1.f;
    s_d2[tid] = __fmul_rn(d, d);
  }
  unsigned int b1 = 0, b2 = 0, before = 0, kk = p.kth;
  if (PASS >= 1) { obs_find_bin<kObsThreads>(p.hist->h[0], kk, s_scan, b1, before); kk -= before; }
  if (PASS >= 2) { obs_find_bin<kObsThreads>(p.hist->h[1], kk, s_scan, b2, before); kk -= before; }
  __syncthreads();
  const int vec_per_row = p.bs >> 2;
  const int64_t nvec = (int64_t)p.R * vec_per_row;
  for (int64_t idx = (int64_t)blockIdx.x * kObsThreads + tid; idx < nvec; idx += (int64_t)gridDim.x * kObsThreads) {
    const int row = (int)(idx / vec_per_row), c4 = (int)(idx % vec_per_row) * 4;
    const float4 w = *reinterpret_cast<const float4*>(p.W32 + (int64_t)row * p.C + p.i1 + c4);
    const float ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const uint32_t key = obs_key(ww[e], s_d2[c4 + e]);
      if (PASS == 0) atomicAdd(&sh[key >> 21], 1u);
      else if (PASS == 1) { if ((key >> 21) == b1) atomicAdd(&sh[(key >> 10) & 0x7ffu], 1u); }
      else { if ((key >> 21) == b1 && ((key >> 10) & 0x7ffu) == b2) atomicAdd(&sh[key & 0x3ffu], 1u); }
    }
  }
  __syncthreads();
  for (int b = tid; b < kObsBins; b += kObsThreads)
    if (sh[b]) atomicAdd(&p.hist->h[PASS][b], sh[b]);
}

// K12 (+ the tail of K11), four rows per warp.  A warp per row is instruction-issue bound: ~60 instructions per
// column step of bookkeeping that is identical for every row (measured: 39.5 us per 4096-row block; this kernel: 27.5 us).  Here a row belongs to EIGHT lanes
// (lane l of the group holds the float4s at columns 32 t + 4 l, t = 0..3), so one warp carries four rows through the
// same 128 steps and the bookkeeping is shared: ~10 instructions per row and step.  The pivot column of every row
// comes from a shuffle inside its lane group; rows that keep the column run the update with err = 0, which leaves
// every value bit-identical (w - 0 * u == w).  Column
// slices that are finished for every row of the warp (t < t0) are skipped statically.  Same arithmetic, same
// roundings and the same order per row as the reference (:189-205).
constexpr int kSw4Threads = 256;
constexpr int kSw4RowsPerCta = (kSw4Threads / 32) * 4;

template <int M>   // 0: unstructured (threshold from the block histograms), else the m of n:m
__global__ void __launch_bounds__(kSw4Threads, 3)
obs_sweep4_kernel(const ObsParams p, int dtype, int vec_ok) {
  extern __shared__ __align__(16) float Us[];                  // [kOB][kOB] U1 tile, zero padded
  __shared__ unsigned int s_scan[32];
  __shared__ __align__(16) float s_d[kOB];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int bs = p.bs;
#pragma unroll 4
  for (int idx = tid; idx < kOB * kOB / 4; idx += kSw4Threads) {
    const int i = idx / (kOB / 4), j = (idx % (kOB / 4)) * 4;
    float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < bs && j < bs && j + 3 >= i) u = *reinterpret_cast<const float4*>(p.U + (int64_t)(p.i1 + i) * p.ldu + p.i1 + j);
    *reinterpret_cast<float4*>(Us + i * kOB + j) = u;
  }
  if (tid < kOB) s_d[tid] = tid < bs ? p.U[(int64_t)(p.i1 + tid) * p.ldu + p.i1 + tid] : 1.f;
  uint32_t v = 0;
  if (M == 0) {
    unsigned int b1, b2, b3, before, kk = p.kth;
    obs_find_bin<kSw4Threads>(p.hist->h[0], kk, s_scan, b1, before); kk -= before;
    obs_find_bin<kSw4Threads>(p.hist->h[1], kk, s_scan, b2, before); kk -= before;
    obs_find_bin<kSw4Threads>(p.hist->h[2], kk, s_scan, b3, before);
    v = (b1 << 21) | (b2 << 10) | b3;                          // the k-th smallest block score, exactly (:184)
  }
  __syncthreads();
  const int g = lane >> 3, l = lane & 7, gbase = lane & ~7;
  const int n = p.prune_n;
  const bool skip_out = p.fail != nullptr && *p.fail != 0;
  const float4* Us4 = reinterpret_cast<const float4*>(Us);

  for (int row0 = (blockIdx.x * (kSw4Threads / 32) + warp) * 4; row0 < p.R; row0 += gridDim.x * kSw4RowsPerCta) {
    const int row = row0 + g;
    const bool valid = row < p.R;
    float* w32 = p.W32 + (int64_t)row * p.C + p.i1 + 4 * l;
    float w[4][4];
    uint32_t mbits = 0;                                          // bit 4 t + e: column 32 t + 4 l + e of this row is pruned
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
      if (valid && 32 * t + 4 * l < bs) x = *reinterpret_cast<const float4*>(w32 + 32 * t);
      w[t][0] = x.x; w[t][1] = x.y; w[t][2] = x.z; w[t][3] = x.w;
      if (M == 0 && valid && 32 * t + 4 * l < bs) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float d = s_d[32 * t + 4 * l + e];
          if (obs_key(w[t][e], __fmul_rn(d, d)) <= v) mbits |= 1u << (4 * t + e);     // `<=` (:185)
        }
      }
    }
    float er[4][4];
#pragma unroll
    for (int t = 0; t < 4; ++t)
#pragma unroll
      for (int e = 0; e < 4; ++e) er[t][e] = 0.f;

#pragma unroll
    for (int t0 = 0; t0 < 4; ++t0) {
      if (32 * t0 < bs) {
#pragma unroll 1
        for (int li = 0; li < 8; ++li) {
          const int ib = 32 * t0 + 4 * li;
          if (ib >= bs) break;
          if (M >= 8 && (ib % (M >= 8 ? M : 8)) == 0) {
            // n:m over M >= 8 columns: lanes li .. li + M/4 - 1 of every group hold the group's columns in slot t0
            float kown[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int col = 32 * t0 + 4 * l + e;
              const float d = s_d[col];
              kown[e] = col < bs ? __fdiv_rn(__fmul_rn(w[t0][e], w[t0][e]), __fmul_rn(d, d)) : __int_as_float(0x7f800000);
            }
            float keys[M >= 8 ? M : 8];
#pragma unroll
            for (int a = 0; a < M; ++a) keys[a] = __shfl_sync(0xffffffffu, kown[a & 3], gbase + ((li + (a >> 2)) & 7));
            const int mypos = 4 * (l - li);                      // position of this lane's first column in the group
            if (mypos >= 0 && mypos < M) {
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                int rank = 0;
#pragma unroll
                for (int b = 0; b < M; ++b)
                  rank += (keys[b] < kown[e] || (keys[b] == kown[e] && b < mypos + e)) ? 1 : 0;
                if (rank < n) mbits |= 1u << (4 * t0 + e);
              }
            }
          }
          uint32_t pm = 0;
          if (M == 0 || M >= 8) pm = __shfl_sync(0xffffffffu, mbits, gbase + li);
          const float4 d4 = *reinterpret_cast<const float4*>(s_d + ib);     // diagonal of the four pivots of this lane slot
          const float dd[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int i = ib + e;
            if (M == 2 || M == 4) {
              if ((e % ((M == 2 || M == 4) ? M : 4)) == 0) {
                // n:m inside one float4: the owning lane ranks its own (already compensated) weights (:193-195)
                if (l == li) {
                  float keys[4];
#pragma unroll
                  for (int a = 0; a < M; ++a) {
                    const float d = s_d[i + a];
                    keys[a] = __fdiv_rn(__fmul_rn(w[t0][(e + a) & 3], w[t0][(e + a) & 3]), __fmul_rn(d, d));
                  }
#pragma unroll
                  for (int a = 0; a < M; ++a) {
                    int rank = 0;
#pragma unroll
                    for (int b = 0; b < M; ++b) rank += (keys[b] < keys[a] || (keys[b] == keys[a] && b < a)) ? 1 : 0;
                    if (rank < n) mbits |= 1u << (4 * t0 + ((e + a) & 3));
                  }
                }
                pm = __shfl_sync(0xffffffffu, mbits, gbase + li);
              }
            }
            const float wi = __shfl_sync(0xffffffffu, w[t0][e], gbase + li);
            const bool pruned = (pm >> (4 * t0 + e)) & 1u;
            // (w - 0) / d (:202); rows that keep the column get err = 0.  No branch: the quotient is computed by every
            // lane and selected, so the step is one straight dependency chain shuffle -> divide -> multiply -> subtract
            const float quot = __fdiv_rn(wi, dd[e]);
            const float err = pruned ? quot : 0.f;
            // product and subtraction rounded separately, like the reference's outer product + in-place sub (:204);
            // U1[i, j < i] is exactly 0, so finished columns are untouched
#pragma unroll
            for (int t = t0; t < 4; ++t) {
              const float4 u = Us4[i * (kOB / 4) + 8 * t + l];
              w[t][0] = __fsub_rn(w[t][0], __fmul_rn(err, u.x)); w[t][1] = __fsub_rn(w[t][1], __fmul_rn(err, u.y));
              w[t][2] = __fsub_rn(w[t][2], __fmul_rn(err, u.z)); w[t][3] = __fsub_rn(w[t][3], __fmul_rn(err, u.w));
            }
            if (l == li && pruned) { w[t0][e] = 0.f; er[t0][e] = err; }     // Q1[:, i] = 0, Err1[:, i] = err
          }
        }
      }
    }
    if (valid) {
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int col = 32 * t + 4 * l;
        *reinterpret_cast<float4*>(p.Err + (int64_t)row * kErrLd + col) = make_float4(er[t][0], er[t][1], er[t][2], er[t][3]);
        if (col < bs) {
          *reinterpret_cast<float4*>(w32 + 32 * t) = make_float4(w[t][0], w[t][1], w[t][2], w[t][3]);
          if (skip_out) continue;          // failed factorisation: only the scratch copies are written
          const int64_t off = (int64_t)row * p.ldw + p.i1 + col;
          if (dtype == VLMC_F32) {
            float* wo = reinterpret_cast<float*>(p.Wout) + off;
            if (vec_ok) *reinterpret_cast<float4*>(wo) = make_float4(w[t][0], w[t][1], w[t][2], w[t][3]);
            else { wo[0] = w[t][0]; wo[1] = w[t][1]; wo[2] = w[t][2]; wo[3] = w[t][3]; }
          } else if (dtype == VLMC_F16) {
            __half* wo = reinterpret_cast<__half*>(p.Wout) + off;
            const __half2 a = __floats2half2_rn(w[t][0], w[t][1]), b = __floats2half2_rn(w[t][2], w[t][3]);
            if (vec_ok) *reinterpret_cast<uint2*>(wo) = make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
            else { wo[0] = __low2half(a); wo[1] = __high2half(a); wo[2] = __low2half(b); wo[3] = __high2half(b); }
          } else {
            __nv_bfloat16* wo = reinterpret_cast<__nv_bfloat16*>(p.Wout) + off;
            const __nv_bfloat162 a = __floats2bfloat162_rn(w[t][0], w[t][1]), b = __floats2bfloat162_rn(w[t][2], w[t][3]);
            if (vec_ok) *reinterpret_cast<uint2*>(wo) = make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
            else { wo[0] = __low2bfloat16(a); wo[1] = __high2bfloat16(a); wo[2] = __low2bfloat16(b); wo[3] = __high2bfloat16(b); }
          }
          if (p.keep) {
            uint8_t* kp = p.keep + (int64_t)row * p.ldm + p.i1 + col;
            const uint32_t mb = (mbits >> (4 * t)) & 0xfu;
            const uint32_t bytes = ((mb & 1u) ? 0u : 1u) | ((mb & 2u) ? 0u : 0x100u) | ((mb & 4u) ? 0u : 0x10000u) | ((mb & 8u) ? 0u : 0x1000000u);
            if (vec_ok) *reinterpret_cast<uint32_t*>(kp) = bytes;
            else { kp[0] = bytes & 1u; kp[1] = (bytes >> 8) & 1u; kp[2] = (bytes >> 16) & 1u; kp[3] = (bytes >> 24) & 1u; }
          }
        }
      }
    }
  }
}

// K11 + K12 in ONE launch for the unstructured sweep (VERDICT r1 next #3): a cooperative grid in which every warp owns four
// rows for the whole block.  The block scores (16 per lane) are computed once and stay in registers through the three
// histogram passes of the exact radix select; between the passes the grid meets at a grid barrier (the CTAs' shared-memory
// histograms flushed to the block's global one, every CTA then finds the chosen bin itself), then the 128-step sweep runs on
// the same registers.  Replaces three obs_hist_kernel launches, their three passes over the fp32 working copy and the
// 3 x find_bin prologue of obs_sweep4_kernel; same arithmetic per element, same threshold, bit-identical results.
// Needs every CTA resident at once: launched with cudaLaunchCooperativeKernel, R <= 32 * (resident CTAs).
__global__ void __launch_bounds__(kSw4Threads, 3)
obs_block_fused_kernel(const ObsParams p, int dtype, int vec_ok) {
  namespace cg = cooperative_groups;
  cg::grid_group grid = cg::this_grid();
  extern __shared__ __align__(16) float Us[];                  // [kOB][kOB] U1 tile, zero padded, then the CTA histogram
  unsigned int* sh_hist = reinterpret_cast<unsigned int*>(Us + kOB * kOB);   // [kObsBins]
  __shared__ unsigned int s_scan[32];
  __shared__ __align__(16) float s_d[kOB];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int bs = p.bs;
#pragma unroll 4
  for (int idx = tid; idx < kOB * kOB / 4; idx += kSw4Threads) {
    const int i = idx / (kOB / 4), j = (idx % (kOB / 4)) * 4;
    float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < bs && j < bs && j + 3 >= i) u = *reinterpret_cast<const float4*>(p.U + (int64_t)(p.i1 + i) * p.ldu + p.i1 + j);
    *reinterpret_cast<float4*>(Us + i * kOB + j) = u;
  }
  if (tid < kOB) s_d[tid] = tid < bs ? p.U[(int64_t)(p.i1 + tid) * p.ldu + p.i1 + tid] : 1.f;
  for (int b = tid; b < kObsBins; b += kSw4Threads) sh_hist[b] = 0;
  __syncthreads();
  const int g = lane >> 3, l = lane & 7, gbase = lane & ~7;
  const bool skip_out = p.fail != nullptr && *p.fail != 0;
  const float4* Us4 = reinterpret_cast<const float4*>(Us);

  const int row = (blockIdx.x * (kSw4Threads / 32) + warp) * 4 + g;
  const bool valid = row < p.R;
  float* w32 = p.W32 + (int64_t)row * p.C + p.i1 + 4 * l;
  float w[4][4];
  uint32_t key[4][4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    const bool in = valid && 32 * t + 4 * l < bs;
    if (in) x = *reinterpret_cast<const float4*>(w32 + 32 * t);
    w[t][0] = x.x; w[t][1] = x.y; w[t][2] = x.z; w[t][3] = x.w;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float d = s_d[32 * t + 4 * l + e];
      key[t][e] = in ? obs_key(w[t][e], __fmul_rn(d, d)) : 0xffffffffu;      // 0xffffffff: not an element of the block
    }
  }
  // ---- exact k-th smallest block score: 11 / 11 / 10-bit radix select, three grid-wide rounds ----
  unsigned int b1 = 0, b2 = 0, before = 0, kk = p.kth;
#pragma unroll 1
  for (int pass = 0; pass < 3; ++pass) {
#pragma unroll
    for (int t = 0; t < 4; ++t)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const uint32_t k = key[t][e];
        if (k == 0xffffffffu) continue;                        // (a NaN score has other bits: obs_key never yields all ones)
        if (pass == 0) atomicAdd(&sh_hist[k >> 21], 1u);
        else if (pass == 1) { if ((k >> 21) == b1) atomicAdd(&sh_hist[(k >> 10) & 0x7ffu], 1u); }
        else { if ((k >> 21) == b1 && ((k >> 10) & 0x7ffu) == b2) atomicAdd(&sh_hist[k & 0x3ffu], 1u); }
      }
    __syncthreads();
    for (int b = tid; b < kObsBins; b += kSw4Threads) {
      const unsigned int c = sh_hist[b];
      if (c) { atomicAdd(&p.hist->h[pass][b], c); sh_hist[b] = 0; }
    }
    __threadfence();
    grid.sync();
    unsigned int bin;
    obs_find_bin<kSw4Threads>(p.hist->h[pass], kk, s_scan, bin, before);
    kk -= before;
    if (pass == 0) b1 = bin; else if (pass == 1) b2 = bin; else before = bin;      // `before` carries b3 out of the loop
    __syncthreads();
  }
  const uint32_t v = (b1 << 21) | (b2 << 10) | before;          // the k-th smallest block score, exactly (:184)
  uint32_t mbits = 0;                                            // bit 4 t + e: column 32 t + 4 l + e of this row is pruned
#pragma unroll
  for (int t = 0; t < 4; ++t)
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (key[t][e] != 0xffffffffu && key[t][e] <= v) mbits |= 1u << (4 * t + e);           // `<=` (:185)

  float er[4][4];
#pragma unroll
  for (int t = 0; t < 4; ++t)
#pragma unroll
    for (int e = 0; e < 4; ++e) er[t][e] = 0.f;
#pragma unroll
  for (int t0 = 0; t0 < 4; ++t0) {
    if (32 * t0 < bs) {
#pragma unroll 1
      for (int li = 0; li < 8; ++li) {
        const int ib = 32 * t0 + 4 * li;
        if (ib >= bs) break;
        const uint32_t pm = __shfl_sync(0xffffffffu, mbits, gbase + li);
        const float4 d4 = *reinterpret_cast<const float4*>(s_d + ib);
        const float dd[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int i = ib + e;
          const float wi = __shfl_sync(0xffffffffu, w[t0][e], gbase + li);
          const bool pruned = (pm >> (4 * t0 + e)) & 1u;
          const float quot = __fdiv_rn(wi, dd[e]);
          const float err = pruned ? quot : 0.f;
#pragma unroll
          for (int t = t0; t < 4; ++t) {
            const float4 u = Us4[i * (kOB / 4) + 8 * t + l];
            w[t][0] = __fsub_rn(w[t][0], __fmul_rn(err, u.x)); w[t][1] = __fsub_rn(w[t][1], __fmul_rn(err, u.y));
            w[t][2] = __fsub_rn(w[t][2], __fmul_rn(err, u.z)); w[t][3] = __fsub_rn(w[t][3], __fmul_rn(err, u.w));
          }
          if (l == li && pruned) { w[t0][e] = 0.f; er[t0][e] = err; }
        }
      }
    }
  }
  if (valid) {
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int col = 32 * t + 4 * l;
      *reinterpret_cast<float4*>(p.Err + (int64_t)row * kErrLd + col) = make_float4(er[t][0], er[t][1], er[t][2], er[t][3]);
      if (col < bs) {
        *reinterpret_cast<float4*>(w32 + 32 * t) = make_float4(w[t][0], w[t][1], w[t][2], w[t][3]);
        if (skip_out) continue;
        const int64_t off = (int64_t)row * p.ldw + p.i1 + col;
        if (dtype == VLMC_F32) {
          float* wo = reinterpret_cast<float*>(p.Wout) + off;
          if (vec_ok) *reinterpret_cast<float4*>(wo) = make_float4(w[t][0], w[t][1], w[t][2], w[t][3]);
          else { wo[0] = w[t][0]; wo[1] = w[t][1]; wo[2] = w[t][2]; wo[3] = w[t][3]; }
        } else if (dtype == VLMC_F16) {
          __half* wo = reinterpret_cast<__half*>(p.Wout) + off;
          const __half2 a = __floats2half2_rn(w[t][0], w[t][1]), b = __floats2half2_rn(w[t][2], w[t][3]);
          if (vec_ok) *reinterpret_cast<uint2*>(wo) = make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
          else { wo[0] = __low2half(a); wo[1] = __high2half(a); wo[2] = __low2half(b); wo[3] = __high2half(b); }
        } else {
          __nv_bfloat16* wo = reinterpret_cast<__nv_bfloat16*>(p.Wout) + off;
          const __nv_bfloat162 a = __floats2bfloat162_rn(w[t][0], w[t][1]), b = __floats2bfloat162_rn(w[t][2], w[t][3]);
          if (vec_ok) *reinterpret_cast<uint2*>(wo) = make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
          else { wo[0] = __low2bfloat16(a); wo[1] = __high2bfloat16(a); wo[2] = __low2bfloat16(b); wo[3] = __high2bfloat16(b); }
        }
        if (p.keep) {
          uint8_t* kp = p.keep + (int64_t)row * p.ldm + p.i1 + col;
          const uint32_t mb = (mbits >> (4 * t)) & 0xfu;
          const uint32_t bytes = ((mb & 1u) ? 0u : 1u) | ((mb & 2u) ? 0u : 0x100u) | ((mb & 4u) ? 0u : 0x10000u) | ((mb & 8u) ? 0u : 0x1000000u);
          if (vec_ok) *reinterpret_cast<uint32_t*>(kp) = bytes;
          else { kp[0] = bytes & 1u; kp[1] = (bytes >> 8) & 1u; kp[2] = (bytes >> 16) & 1u; kp[3] = (bytes >> 24) & 1u; }
        }
      }
    }
  }
}

// resident CTAs of the fused kernel on this device (0: cooperative launch not available)
static int obs_fused_capacity() {
  static int cap = -1;
  if (cap >= 0) return cap;
  const size_t smem = (size_t)kOB * kOB * sizeof(float) + kObsBins * sizeof(unsigned int);
  int dev = 0, coop = 0, per_sm = 0;
  cap = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return cap; }
  if (cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev) != cudaSuccess || !coop) { cudaGetLastError(); return cap; }
  if (cudaFuncSetAttribute(obs_block_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) { cudaGetLastError(); return cap; }
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, obs_block_fused_kernel, kSw4Threads, smem) != cudaSuccess) { cudaGetLastError(); return cap; }
  cap = per_sm * kNumSMs;
  return cap;
}

// VLMC_OBS_FUSED=0 keeps the three histogram launches + obs_sweep4_kernel (A/B runs, tests)
static bool obs_fused_enabled(int R) {
  const char* e = getenv("VLMC_OBS_FUSED");
  if (e && e[0] == '0') return false;
  const int ctas = (R + kSw4RowsPerCta - 1) / kSw4RowsPerCta;
  return ctas <= obs_fused_capacity();
}

static int launch_fused(const ObsParams& p, int dtype, int vec_ok, cudaStream_t st) {
  const size_t smem = (size_t)kOB * kOB * sizeof(float) + kObsBins * sizeof(unsigned int);
  const int grid = (p.R + kSw4RowsPerCta - 1) / kSw4RowsPerCta;
  ObsParams pp = p;
  void* args[] = {&pp, &dtype, &vec_ok};
  if (cudaLaunchCooperativeKernel((const void*)obs_block_fused_kernel, dim3(grid), dim3(kSw4Threads), args, smem, st) != cudaSuccess)
    return check_launch();
  return check_launch();
}

template <int M>
static int launch_sweep4(const ObsParams& p, int dtype, int vec_ok, cudaStream_t st) {
  auto kern = obs_sweep4_kernel<M>;
  const size_t smem = (size_t)kOB * kOB * sizeof(float);
  static bool attr_set = false;
  if (!attr_set) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return check_launch();
    attr_set = true;
  }
  int grid = (p.R + kSw4RowsPerCta - 1) / kSw4RowsPerCta;
  if (grid > kNumSMs * 3) grid = kNumSMs * 3;
  kern<<<grid, kSw4Threads, smem, st>>>(p, dtype, vec_ok);
  return check_launch();
}

size_t obs_workspace_bytes(int R, int C) {
  const int nblk = (C + kOB - 1) / kOB;
  return VLMC_WS_COUNTER_BYTES + align_up((size_t)R * C * sizeof(float), 256) + align_up(2 * (size_t)R * kErrLd * sizeof(float), 256) +
         align_up((size_t)nblk * sizeof(ObsHist), 256) + align_up((size_t)kNumSMs * 64 * sizeof(float), 256);
}

}  // namespace vlmc

namespace vlmc {

struct ObsLayout { float* W32; float* Err; ObsHist* hist; float* part; };

// blocks per super-block: VLMC_OBS_SUPERBLOCK (1, 2, 4 or 8; default 4; 1 = the reference's block-by-block schedule)
static int obs_superblock() {
  const char* e = getenv("VLMC_OBS_SUPERBLOCK");
  if (e) {
    const int v = atoi(e);
    if (v == 1 || v == 2 || v == 4 || v == 8) return v;
  }
  return 4;
}
static ObsLayout obs_carve(void* ws, int R, int C) {
  const int nblk = (C + kOB - 1) / kOB;
  char* base = reinterpret_cast<char*>(ws) + VLMC_WS_COUNTER_BYTES;
  ObsLayout l;
  l.W32 = reinterpret_cast<float*>(base);
  base += align_up((size_t)R * C * sizeof(float), 256);
  l.Err = reinterpret_cast<float*>(base);
  base += align_up(2 * (size_t)R * kErrLd * sizeof(float), 256);     // two buffers: super-blocks alternate (look-ahead)
  l.hist = reinterpret_cast<ObsHist*>(base);
  base += align_up((size_t)nblk * sizeof(ObsHist), 256);
  l.part = reinterpret_cast<float*>(base);
  return l;
}

static int obs_checks(void* W, int dtype, int R, int C, int64_t ldw, const float* U, int64_t ldu, double sparsity,
                      int prune_n, int prune_m, int blocksize, const uint8_t* keep_mask, int64_t ldm, void* ws,
                      size_t ws_bytes) {
  if (!W || !U || !ws || R < 1 || C < 1 || ldw < C || ldu < C) return VLMC_ERR_BAD_ARG;
  if (dtype != VLMC_F32 && dtype != VLMC_F16 && dtype != VLMC_BF16) return VLMC_ERR_BAD_ARG;
  if (blocksize != kOB) return VLMC_ERR_UNSUPPORTED;
  if (prune_n < 0 || (prune_n > 0 && (prune_m <= prune_n || prune_m > kObsMaxM || kOB % prune_m != 0))) return VLMC_ERR_BAD_ARG;
  if (prune_n == 0 && !(sparsity >= 0.0 && sparsity < 1.0)) return VLMC_ERR_BAD_ARG;
  if ((C & 3) || (ldu & 3) || ((uintptr_t)U & 15)) return VLMC_ERR_UNSUPPORTED;
  if (keep_mask && ldm < C) return VLMC_ERR_BAD_ARG;
  if ((uint64_t)R * kOB >= 0xffffffffull) return VLMC_ERR_UNSUPPORTED;
  if (!is_device_ptr(W) || !is_device_ptr(U) || !is_device_ptr(ws)) return VLMC_ERR_NOT_DEVICE;
  if (ws_bytes < obs_workspace_bytes(R, C)) return VLMC_ERR_WORKSPACE;
  return VLMC_OK;
}

static ObsParams obs_block_params(const ObsLayout& l, void* W, int R, int C, int64_t ldw, const float* U, int64_t ldu,
                                  int blk, int64_t rows_total, double sparsity, int prune_n, int prune_m,
                                  uint8_t* keep_mask, int64_t ldm, unsigned int* hist) {
  ObsParams p;
  p.W32 = l.W32; p.Wout = W; p.ldw = ldw; p.R = R; p.C = C; p.U = U; p.ldu = ldu;
  p.i1 = blk * kOB;
  p.bs = (C - p.i1 < kOB) ? (C - p.i1) : kOB;
  {
    const int sb = obs_superblock();
    p.Err = l.Err + (size_t)((blk / sb) & 1) * (size_t)R * kErrLd + (size_t)(blk % sb) * kOB;
  }
  p.keep = keep_mask; p.ldm = ldm;
  // int(numel * sparsity) is the 0-indexed rank of the threshold (:184); numel counts the rows of ALL shards
  p.kth = (unsigned int)((ull)((double)((ull)rows_total * (ull)p.bs) * sparsity)) + 1u;
  p.prune_n = prune_n; p.prune_m = prune_m;
  p.hist = hist ? reinterpret_cast<ObsHist*>(hist) + blk : l.hist + blk;
  p.fail = nullptr;
  return p;
}

}  // namespace vlmc

extern "C" int vlmc_obs_begin(void* W, int dtype, int R, int C, int64_t ldw, const float* U, int64_t ldu,
                              const uint8_t* dead, float* importance_sum, void* ws, size_t ws_bytes, void* stream) {
  using namespace vlmc;
  int rc = obs_checks(W, dtype, R, C, ldw, U, ldu, 0.0, 0, 0, kOB, nullptr, 0, ws, ws_bytes);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  ObsLayout l = obs_carve(ws, R, C);
  const int nblk = (C + kOB - 1) / kOB;
  if (cudaMemsetAsync(l.hist, 0, (size_t)nblk * sizeof(ObsHist), st) != cudaSuccess) return check_launch();
  dim3 grid((C + 255) / 256, R < 64 ? R : 64);
  VLMC_DISPATCH_DTYPE(dtype, (obs_upcast_kernel<scalar_t><<<grid, 256, 0, st>>>(
                                 reinterpret_cast<const scalar_t*>(W), ldw, l.W32, R, C, dead)));
  if (importance_sum) {
    obs_importance_kernel<<<grid, 256, 0, st>>>(l.W32, R, C, U, ldu, l.part);
    rc = launch_mean_finalize(l.part, grid.x * grid.y, 1.0, importance_sum, st);   // sum; the caller divides by numel
    if (rc) return rc;
  }
  return check_launch();
}

extern "C" int vlmc_obs_block_hist(int R, int C, const float* U, int64_t ldu, int blk, int pass, int64_t rows_total,
                                   double sparsity, unsigned int* hist, void* ws, size_t ws_bytes, void* stream) {
  using namespace vlmc;
  if (!U || !ws || R < 1 || C < 1 || blk < 0 || blk * kOB >= C || pass < 0 || pass > 2 || rows_total < R)
    return VLMC_ERR_BAD_ARG;
  if (ws_bytes < obs_workspace_bytes(R, C)) return VLMC_ERR_WORKSPACE;
  if ((uint64_t)rows_total * kOB >= 0xffffffffull) return VLMC_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  ObsLayout l = obs_carve(ws, R, C);
  ObsParams p = obs_block_params(l, nullptr, R, C, C, U, ldu, blk, rows_total, sparsity, 0, 0, nullptr, 0, hist);
  const int64_t nvec = (int64_t)R * (p.bs >> 2);
  int hgrid = (int)((nvec + kObsThreads * 4 - 1) / (kObsThreads * 4));
  if (hgrid > kNumSMs * 4) hgrid = kNumSMs * 4;
  if (hgrid < 1) hgrid = 1;
  if (pass == 0) obs_hist_kernel<0><<<hgrid, kObsThreads, 0, st>>>(p);
  else if (pass == 1) obs_hist_kernel<1><<<hgrid, kObsThreads, 0, st>>>(p);
  else obs_hist_kernel<2><<<hgrid, kObsThreads, 0, st>>>(p);
  return check_launch();
}

namespace vlmc {
static int obs_block_finish_impl(void* W, int dtype, int R, int C, int64_t ldw, const float* U, int64_t ldu, int blk,
                                 int64_t rows_total, double sparsity, int prune_n, int prune_m, uint8_t* keep_mask,
                                 int64_t ldm, unsigned int* hist, void* ws, size_t ws_bytes, void* stream, const int* fail,
                                 ChainSide* side = nullptr, bool* pending_far = nullptr, bool fused = false) {
  int rc = obs_checks(W, dtype, R, C, ldw, U, ldu, sparsity, prune_n, prune_m, kOB, keep_mask, ldm, ws, ws_bytes);
  if (rc) return rc;
  if (blk < 0 || blk * kOB >= C || rows_total < R) return VLMC_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  ObsLayout l = obs_carve(ws, R, C);
  ObsParams p = obs_block_params(l, W, R, C, ldw, U, ldu, blk, rows_total, sparsity, prune_n, prune_m, keep_mask, ldm, hist);
  p.fail = fail;
  // 8-byte weight stores / 4-byte mask stores need aligned rows; otherwise the kernel stores element by element
  const int esz = elem_size(dtype);
  const int vec_ok = ((ldw * esz) % (4 * esz) == 0) && (((uintptr_t)W) % (4 * esz) == 0) &&
                     (!keep_mask || ((ldm % 4 == 0) && (((uintptr_t)keep_mask) % 4 == 0)));
  switch (prune_n == 0 ? 0 : prune_m) {
    case 0: rc = fused ? launch_fused(p, dtype, vec_ok, st) : launch_sweep4<0>(p, dtype, vec_ok, st); break;
    case 2: rc = launch_sweep4<2>(p, dtype, vec_ok, st); break;
    case 4: rc = launch_sweep4<4>(p, dtype, vec_ok, st); break;
    case 8: rc = launch_sweep4<8>(p, dtype, vec_ok, st); break;
    case 16: rc = launch_sweep4<16>(p, dtype, vec_ok, st); break;
    default: return VLMC_ERR_UNSUPPORTED;
  }
  if (rc) return rc;
  const int i2 = p.i1 + p.bs;
  if (i2 < C) {
    // K13: W[:, i2:] -= Err1 @ U[i1:i2, i2:], on the super-block schedule (see kSBMax)
    const int sb = obs_superblock();
    const int slot = blk % sb;
    const int sb_i1 = (blk - slot) * kOB;                       // first column of the super-block
    const int sb_i2 = sb_i1 + sb * kOB < C ? sb_i1 + sb * kOB : C;   // one past its last column
    if (i2 < sb_i2) {      // near: the rest of this super-block gets this block's errors now
      rc = gemm3x(false, R, sb_i2 - i2, kOB, -1.f, p.Err, kErrLd, U + (int64_t)p.i1 * ldu + i2, ldu, 1.f, l.W32 + i2, C, 0, 0, st);
      if (rc) return rc;
    } else if (sb_i2 < C) {  // far: the super-block is complete, everything behind it gets all of its errors at once
      // kc = K: one in-TMEM accumulation over the whole super-block (256-wide tiles, no per-chunk register sums); the
      // round-toward-zero drift of K / 8 * 3 accumulations stays below 1.2e-5 of the update term at K = 512
      const char* ce = getenv("VLMC_OBS_FAR_CHUNKED");
      const int K = i2 - sb_i1;
      const int kc = (ce && ce[0] == '1') ? 0 : K;
      const float* ErrSB = l.Err + (size_t)((blk / sb) & 1) * (size_t)R * kErrLd;
      const float* Ufar = U + (int64_t)sb_i1 * ldu + sb_i2;
      const int behind = C - sb_i2;
      const int next_cols = sb * kOB < behind ? sb * kOB : behind;      // the next super-block's columns
      if (!side || behind - next_cols < kOB) {
        // the previous super-block's far_rest may still be writing these columns on the side stream
        if (pending_far && *pending_far) {
          if (cudaStreamWaitEvent(st, side->updated, 0) != cudaSuccess) return check_launch();
          *pending_far = false;
        }
        rc = gemm3x(false, R, behind, K, -1.f, ErrSB, kErrLd, Ufar, ldu, 1.f, l.W32 + sb_i2, C, 0, kc, st);
        if (rc) return rc;
      } else {
        // Look-ahead: only the NEXT super-block's columns are needed before its sweeps can start; the rest of the far
        // update runs on a side stream under them.  far_rest(s - 1) wrote the columns far_near(s) updates, hence the wait;
        // far_rest(s) reads this super-block's Err buffer, which is not rewritten before super-block s + 2, i.e. after the
        // wait at the end of super-block s + 1.
        if (*pending_far) {
          if (cudaStreamWaitEvent(st, side->updated, 0) != cudaSuccess) return check_launch();
          *pending_far = false;
        }
        if (cudaEventRecord(side->solved, st) != cudaSuccess) return check_launch();
        rc = gemm3x(false, R, next_cols, K, -1.f, ErrSB, kErrLd, Ufar, ldu, 1.f, l.W32 + sb_i2, C, 0, kc, st);
        if (rc) return rc;
        if (cudaStreamWaitEvent(side->stream, side->solved, 0) != cudaSuccess) return check_launch();
        rc = gemm3x(false, R, behind - next_cols, K, -1.f, ErrSB, kErrLd, Ufar + next_cols, ldu, 1.f,
                    l.W32 + sb_i2 + next_cols, C, 0, kc, side->stream, 0, false, kNumSMs - 20);
        if (rc) return rc;
        if (cudaEventRecord(side->updated, side->stream) != cudaSuccess) return check_launch();
        *pending_far = true;
      }
    }
  }
  return check_launch();
}
}  // namespace vlmc

extern "C" int vlmc_obs_block_finish(void* W, int dtype, int R, int C, int64_t ldw, const float* U, int64_t ldu, int blk,
                                     int64_t rows_total, double sparsity, int prune_n, int prune_m, uint8_t* keep_mask,
                                     int64_t ldm, unsigned int* hist, void* ws, size_t ws_bytes, void* stream) {
  return vlmc::obs_block_finish_impl(W, dtype, R, C, ldw, U, ldu, blk, rows_total, sparsity, prune_n, prune_m, keep_mask, ldm,
                                     hist, ws, ws_bytes, stream, nullptr);
}

namespace vlmc {
static int obs_sweep_impl(void* W, int dtype, int R, int C, int64_t ldw, const float* U, int64_t ldu,
                          const uint8_t* dead, double sparsity, int prune_n, int prune_m, int blocksize,
                          uint8_t* keep_mask, int64_t ldm, float* importance_score,
                          void* ws, size_t ws_bytes, void* stream, const int* fail) {
  int rc = obs_checks(W, dtype, R, C, ldw, U, ldu, sparsity, prune_n, prune_m, blocksize, keep_mask, ldm, ws, ws_bytes);
  if (rc) return rc;
  rc = vlmc_obs_begin(W, dtype, R, C, ldw, U, ldu, dead, importance_score, ws, ws_bytes, stream);
  if (rc) return rc;
  if (importance_score) {   // vlmc_obs_begin left the sum: mean = sum / numel (:163-165)
    rc = launch_mean_finalize(importance_score, 1, (double)R * (double)C, importance_score, (cudaStream_t)stream);
    if (rc) return rc;
  }
  const int nblk = (C + kOB - 1) / kOB;
  cudaStream_t st = (cudaStream_t)stream;
  // the far updates run ahead on a side stream for a chain that has the GPU to itself (same switch as the Cholesky's
  // look-ahead: callers that enqueue several chains concurrently turn it off)
  ChainSide* side = (chain_lookahead_enabled() && nblk > 2 * obs_superblock()) ? chain_side_for(st, 1) : nullptr;
  bool pending_far = false;
  // Histogram passes + sweep of a block in one cooperative launch - for a chain that has the GPU to itself (the same switch
  // as the look-ahead: vlmc.schedule turns it off while it enqueues several chains).  A cooperative grid starts only when ALL
  // its CTAs fit at once, so next to other chains' kernels it waits for a drained GPU: measured on B200, 4096^2 sweep alone
  // 2.50 -> 2.18 ms, 4096 x 11008 8.02 -> 7.84 ms, the 7 sweeps of a block on concurrent streams 17.4 -> 17.9 ms.
  const bool fused = prune_n == 0 && chain_lookahead_enabled() && obs_fused_enabled(R);
  for (int blk = 0; blk < nblk; ++blk) {
    if (prune_n == 0 && !fused)
      for (int pass = 0; pass < 3; ++pass) {
        rc = vlmc_obs_block_hist(R, C, U, ldu, blk, pass, R, sparsity, nullptr, ws, ws_bytes, stream);
        if (rc) return rc;
      }
    rc = obs_block_finish_impl(W, dtype, R, C, ldw, U, ldu, blk, R, sparsity, prune_n, prune_m, keep_mask, ldm,
                               nullptr, ws, ws_bytes, stream, fail, side, &pending_far, fused);
    if (rc) return rc;
  }
  if (pending_far && cudaStreamWaitEvent(st, side->updated, 0) != cudaSuccess) return check_launch();
  return VLMC_OK;
}
}  // namespace vlmc

extern "C" int vlmc_obs_sweep(void* W, int dtype, int R, int C, int64_t ldw, const float* U, int64_t ldu,
                              const uint8_t* dead, double sparsity, int prune_n, int prune_m, int blocksize,
                              uint8_t* keep_mask, int64_t ldm, float* importance_score,
                              void* ws, size_t ws_bytes, void* stream) {
  return vlmc::obs_sweep_impl(W, dtype, R, C, ldw, U, ldu, dead, sparsity, prune_n, prune_m, blocksize, keep_mask, ldm,
                              importance_score, ws, ws_bytes, stream, nullptr);
}

extern "C" int vlmc_obs_sweep_guarded(void* W, int dtype, int R, int C, int64_t ldw, const float* U, int64_t ldu,
                                      const uint8_t* dead, double sparsity, int prune_n, int prune_m, int blocksize,
                                      uint8_t* keep_mask, int64_t ldm, float* importance_score, const int* fail_flag,
                                      void* ws, size_t ws_bytes, void* stream) {
  if (fail_flag && !vlmc::is_device_ptr(fail_flag)) return VLMC_ERR_NOT_DEVICE;
  return vlmc::obs_sweep_impl(W, dtype, R, C, ldw, U, ldu, dead, sparsity, prune_n, prune_m, blocksize, keep_mask, ldm,
                              importance_score, ws, ws_bytes, stream, fail_flag);
}
