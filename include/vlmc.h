/*
 * vlmc.h - C ABI of the B200 (sm_100a) calibration-and-masking kernels.
 *
 * This is the drop-in boundary for the one hot path of Shwai-He/VLM-Compression:
 * the per-linear-layer statistics / mask-selection / OBS-sweep / masked-merge code in
 *   lavis/compression/pruners/{wanda,sparsegpt,dsnot}_pruner.py and
 *   lavis/peft/src/peft/tuners/lora.py.
 * The reference has no FFI of its own (it is pure torch), so every entry point below
 * names the torch call sites (file:line) it replaces.  INTEGRATION.md shows the ctypes
 * stub a maintainer adds on the reference side.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (torch allocates, we never do);
 *     nothing is retained after the call returns
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); calls are
 *     asynchronous unless stated otherwise
 *   - matrices are row-major with an explicit leading dimension in ELEMENTS
 *   - `ws` is caller-provided scratch of at least vlmc_workspace_bytes() bytes.  The first
 *     VLMC_WS_COUNTER_BYTES bytes hold inter-CTA tickets: they must be ZERO before the
 *     first use of a workspace and every call leaves them zero again.  One workspace must
 *     not be shared by calls running concurrently on different streams.
 *   - return value: 0 ok; <0 argument / launch error; >0 numerical status
 *   - there is NO CPU path: host pointers are rejected with VLMC_ERR_NOT_DEVICE
 */
#ifndef VLMC_H_
#define VLMC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VLMC_ABI_VERSION 1

enum vlmc_dtype { VLMC_F32 = 0, VLMC_F16 = 1, VLMC_BF16 = 2 };

enum vlmc_status {
  VLMC_OK = 0,
  VLMC_ERR_BAD_ARG = -1,      /* null pointer, non-positive size, bad enum            */
  VLMC_ERR_UNSUPPORTED = -2,  /* shape / alignment outside what the kernels are built for */
  VLMC_ERR_NOT_DEVICE = -3,   /* a pointer is not CUDA device memory                  */
  VLMC_ERR_WORKSPACE = -4,    /* ws too small                                         */
  VLMC_ERR_CUDA = -5,         /* launch failed; see vlmc_last_cuda_error()            */
  /* numerical status BITS of the factorisation's device status word (0 = clean) */
  VLMC_NOT_POSDEF = 1,        /* Cholesky met a non-positive / NaN pivot (caller damps, retries)           */
  VLMC_NONFINITE = 2,         /* the input matrix holds +-inf or NaN (caller clamps like :101-109, retries) */
  VLMC_HUGE_FACTOR = 4,       /* an entry of U exceeds 1e15: diag(H^-1) may overflow fp32, the caller runs the
                                 reference's second stage (:131-157) explicitly                           */
  VLMC_NOT_2OF4 = 8           /* vlmc_sparse24_compress: a group of 4 columns holds more than two non-zeros */
};

#define VLMC_WS_COUNTER_BYTES 4096

enum vlmc_op {
  VLMC_OP_SQNORM = 0,       /* (T, C, 0)       */
  VLMC_OP_DSNOT_STATS = 1,  /* (nseg*S, C, nseg) */
  VLMC_OP_WANDA_SELECT = 2, /* (R, C, 0)       */
  VLMC_OP_LORA_MERGE = 3,   /* (R, C, r)       */
  VLMC_OP_HESSIAN = 4,      /* (T, C, 0)       */
  VLMC_OP_CHOL = 5,         /* (C, 0, 0)       */
  VLMC_OP_OBS = 6,          /* (R, C, blocksize) */
  VLMC_OP_DSNOT_REFINE = 7, /* (R, C, max_cycle_time) */
  VLMC_OP_SPARSE24_LINEAR = 8 /* (T, R, C)       */
};

int vlmc_version(void);
const char* vlmc_status_string(int status);
/* cudaError_t of the most recent failing launch on this thread (0 if none). */
int vlmc_last_cuda_error(void);
size_t vlmc_workspace_bytes(int op, int64_t d0, int64_t d1, int64_t d2);

/*
 * K1  Wanda calibration statistic.  Replaces WrappedGPT.add_batch, wanda_pruner.py:66-81:
 *   scaler_row[c] <- scaler_row[c] * n_before/(n_before+b) + (sum_t x[t,c]^2) / (n_before+b)
 * x: [T, C] row-major activations of one add_batch call (the reference's inp.reshape(-1, C)),
 * T = b * seq_len.  fp16 / bf16 / fp32 inputs are up-cast to fp32 like wanda_pruner.py:80.
 * One streaming pass over x, fp32 per-thread partials, fp64 cross-CTA combine (deterministic).
 */
int vlmc_sqnorm_accum(const void* x, int dtype, int64_t T, int C, int64_t ldx,
                      float* scaler_row, double n_before, double b,
                      void* ws, size_t ws_bytes, void* stream);

/*
 * K1 for several linears in ONE launch (the 7 accumulations of a transformer block, or a rank's share of them when the
 * calibration tokens are sharded over GPUs): same arithmetic and the same deterministic combine as vlmc_sqnorm_accum per
 * item, one ramp-up and one drain.  count <= 16, one dtype per launch; ws of vlmc_sqnorm_accum_batch_workspace_bytes.
 */
typedef struct vlmc_stats_item {
  const void* x; int64_t T; int C; int64_t ldx;
  float* scaler_row; double n_before; double b;
} vlmc_stats_item;
size_t vlmc_sqnorm_accum_batch_workspace_bytes(const vlmc_stats_item* items, int count, int dtype);
int vlmc_sqnorm_accum_batch(const vlmc_stats_item* items, int count, int dtype, void* ws, size_t ws_bytes, void* stream);

/*
 * K2  DSnoT calibration statistics.  Replaces WrappedGPT.add_batch, dsnot_pruner.py:79-101.
 * x is treated as `nseg` consecutive add_batch calls of S rows each, every one with leading
 * batch dimension b_per_seg (nseg = 1 reproduces a single reference call exactly):
 *   scaler_row, sum_row : running means over samples of sum_t x^2 and sum_t x   (:96-101)
 *   mean, var           : token-weighted running means of the per-call mean and
 *                         per-call BIASED variance                                (:89-93)
 * ntok_before is the wrapper's ntokens before the call.
 */
int vlmc_dsnot_stats(const void* x, int dtype, int64_t nseg, int64_t S, int C, int64_t ldx,
                     float* scaler_row, float* sum_row, float* mean, float* var,
                     double n_before, double b_per_seg, double ntok_before,
                     void* ws, size_t ws_bytes, void* stream);

/*
 * K2 for several linears in ONE launch (the 7 wrappers of a transformer block): the same plan, partial sums and results as
 * vlmc_dsnot_stats per item.  The grid is ordered so that linears fed the same activations (q / k / v, gate / up) work on the
 * same call at the same time: the repeated reads hit in L2.  count <= 16, one dtype per launch.
 */
typedef struct vlmc_dsnot_stats_item {
  const void* x; int64_t nseg; int64_t S; int C; int64_t ldx;
  float* scaler_row; float* sum_row; float* mean; float* var;
  double n_before; double b_per_seg; double ntok_before;
} vlmc_dsnot_stats_item;
size_t vlmc_dsnot_stats_batch_workspace_bytes(const vlmc_dsnot_stats_item* items, int count, int dtype);
int vlmc_dsnot_stats_batch(const vlmc_dsnot_stats_item* items, int count, int dtype, void* ws, size_t ws_bytes, void* stream);

/*
 * K4+K5  Wanda score + per-row unstructured selection.  Replaces wanda_pruner.py:318-341
 * (LLM path): S = |W| * sqrt(scaler_row) in fp32; in every row the k smallest scores are
 * pruned, ties going to the LOWER column (torch.sort(stable=True), :332).  k = int(C * p)
 * is computed by the caller (:336).
 *   keep_mask [R, ldm] bytes: 1 = kept, 0 = pruned (= module.mask, :339)
 *   zero_w != 0 writes 0 into pruned weights in place (:341); 0 leaves W untouched (lora_model)
 *   score_mean (device float, may be NULL): mean(S) (= weight.importance_score, :320)
 */
int vlmc_wanda_rowselect(void* W, int dtype, int R, int C, int64_t ldw,
                         const float* scaler_row, int k, int zero_w,
                         uint8_t* keep_mask, int64_t ldm, float* score_mean,
                         void* ws, size_t ws_bytes, void* stream);

/*
 * K4+K6  Wanda score + n:m selection.  Replaces the C/m-iteration python loop at
 * wanda_pruner.py:323-329 (and its ViT copy :671-677): in every group of m consecutive
 * columns the n smallest scores are pruned; ties go to the lower column.
 * m in {2,4,8,16}, 0 < n < m, C % m == 0.
 */
int vlmc_wanda_nm(void* W, int dtype, int R, int C, int64_t ldw,
                  const float* scaler_row, int n, int m, int zero_w,
                  uint8_t* keep_mask, int64_t ldm, float* score_mean,
                  void* ws, size_t ws_bytes, void* stream);

/*
 * K4+K6 for ALL linears of one transformer block in one launch (the per-block loop at
 * wanda_pruner.py:313-347 calls the selection once per linear; the matrices are 34-90 MB, so launched one by one
 * the kernels are short enough for ramp-up and drain to cost a third of their time).  `items` is a HOST array of
 * `count` (<= 16) descriptors, read during the call; every pointer inside is a device pointer.  Same results as
 * `count` calls of vlmc_wanda_nm (score_mean up to fp32 summation order).  score_mean may be NULL per item.
 */
typedef struct vlmc_select_item {
  void* W; int64_t ldw; int R; int C;
  const float* scaler_row;      /* [C] fp32, 16-byte aligned */
  uint8_t* keep_mask; int64_t ldm;
  float* score_mean;            /* 1 float or NULL */
} vlmc_select_item;
size_t vlmc_wanda_nm_batch_workspace_bytes(const vlmc_select_item* items, int count, int dtype, int m);
int vlmc_wanda_nm_batch(const vlmc_select_item* items, int count, int dtype, int n, int m, int zero_w,
                        void* ws, size_t ws_bytes, void* stream);

/*
 * K4+K5 for up to 16 linears in one call (wanda_pruner.py:332-341 runs per linear; a block's linears are independent):
 * items of equal C share ONE launch whose CTAs walk the concatenated rows (a Vicuna block: 2 launches instead of 7, 25-30
 * rows per CTA instead of 5).  k[i] (HOST array) = rows' prune count of item i.  Same masks, weights and score means as
 * vlmc_wanda_rowselect per item, bit for bit.  `items` and `k` are read during the call.
 */
size_t vlmc_wanda_rowselect_batch_workspace_bytes(const vlmc_select_item* items, int count);
int vlmc_wanda_rowselect_batch(const vlmc_select_item* items, const int* k, int count, int dtype, int zero_w,
                               void* ws, size_t ws_bytes, void* stream);

/*
 * K4+K7  Wanda score + whole-matrix threshold (ViT path).  Replaces wanda_pruner.py:682-683:
 *   thres = sort(S.flatten())[k_global];  prune S < thres   (strict: ties are kept)
 * k_global = int(R * C * p) computed by the caller.
 */
int vlmc_wanda_threshold(void* W, int dtype, int R, int C, int64_t ldw,
                         const float* scaler_row, int64_t k_global, int zero_w,
                         uint8_t* keep_mask, int64_t ldm, float* score_mean,
                         void* ws, size_t ws_bytes, void* stream);

/*
 * Multi-GPU mask exchange (new: the reference prunes independent replicas, SURVEY F2).  When the output rows of a linear
 * are split across GPUs (SURVEY 8e) each rank computes module.mask (wanda_pruner.py:339) for its rows only; the weights
 * are replicated, so ranks exchange the masks as BITS (1 bit per weight) and zero their own replica (:341) locally.
 *   vlmc_mask_pack          keep_mask [R, ldm] bytes (0/1) -> bits [R, ldb] bytes; bit e of byte j = column 8j + e
 *   vlmc_mask_apply_packed  bits -> keep_mask bytes (may be NULL) and, if zero_w, W[r,c] = 0 where the bit is 0.
 *                           The bits of row r are at bits + (r / rows_per_seg) * seg_stride + (r % rows_per_seg) * ldb:
 *                           an all-gathered buffer laid out [rank][this linear's row shard] is consumed in ONE call
 *                           (rows_per_seg = R / world, seg_stride = bytes per rank); rows_per_seg <= 0: one segment.
 * C must be a multiple of 16.
 */
int vlmc_mask_pack(const uint8_t* keep_mask, int R, int C, int64_t ldm, uint8_t* bits, int64_t ldb, void* stream);
int vlmc_mask_apply_packed(void* W, int dtype, int R, int C, int64_t ldw, const uint8_t* bits, int64_t ldb,
                           int rows_per_seg, int64_t seg_stride, uint8_t* keep_mask, int64_t ldm, int zero_w,
                           void* stream);

/* The same for up to 16 matrices per launch (`items` is a HOST array read during the call): the masks of all linears of a
 * block are packed before, and expanded after, ONE all-gather.  Same results as the per-matrix calls. */
typedef struct vlmc_pack_item { const uint8_t* keep_mask; int R; int C; int64_t ldm; uint8_t* bits; int64_t ldb; } vlmc_pack_item;
typedef struct vlmc_apply_item {
  void* W; int R; int C; int64_t ldw; const uint8_t* bits; int64_t ldb; int rows_per_seg; int64_t seg_stride;
  uint8_t* keep_mask; int64_t ldm;
} vlmc_apply_item;
int vlmc_mask_pack_batch(const vlmc_pack_item* items, int count, void* stream);
int vlmc_mask_apply_packed_batch(const vlmc_apply_item* items, int count, int dtype, int zero_w, void* stream);

/*
 * K14  SparseLoRA masked merge.  Replaces Linear.merge() (sparse branch), lora.py:384-387,
 * fused with the re-mask of train.py:634-637:
 *   W[r,c] <- keep_mask[r,c] ? round_to_W_dtype( float(W[r,c]) + scaling * sum_k B[r,k]*A[k,c] ) : 0
 * A = lora_A.weight [rank, C], B = lora_B.weight [R, rank], both fp32 row-major contiguous.
 * remask = 0 keeps W[r,c] unchanged where keep_mask is 0 (merge() alone).
 * The arithmetic: sum_k B A is one fmaf per k, k ascending from +0; then W + (sum * scaling) as two separately rounded
 * fp32 operations (no contraction), rounded once to W's dtype.  A masked entry is +0 (remask) or W's value as it was,
 * whatever the LoRA product holds there (see the masked-position rule below K16).
 */
int vlmc_sparselora_merge(void* W, int dtype, int R, int C, int64_t ldw,
                          const float* A, const float* B, int rank, float scaling,
                          const uint8_t* keep_mask, int64_t ldm, int remask,
                          void* stream);

/*
 * K14 for up to 16 LoRA linears in one launch (train.py:626-637 merges module by module).  `items` is a HOST array
 * read during the call.  rank <= 16; same results as vlmc_sparselora_merge per item.
 */
typedef struct vlmc_merge_item {
  void* W; int64_t ldw; int R; int C;
  const float* A; const float* B; int rank; float scaling;
  const uint8_t* keep_mask; int64_t ldm;
} vlmc_merge_item;
int vlmc_sparselora_merge_batch(const vlmc_merge_item* items, int count, int dtype, int remask, void* stream);

/*
 * K15  SparseLoRA masked training forward, the weight part.  Replaces the weight expression of Linear.forward
 * (r > 0, not merged), lora.py:364-375, that the reference re-materialises every step:
 *   sparse != 0:  out = ((W + ((B @ A).to(dtype) * scaling)) * mask)        (:364-369)
 *   sparse == 0:  out = ( W * mask + ((B @ A).to(dtype) * scaling))         (:370-375)
 * with the reference's roundings (product cast to W's dtype, scaled in that dtype, added in that dtype); the product is
 * K14's (one fmaf per k, k ascending from +0).  A masked W counts as +0: with sparse != 0 masked entries of out are +0
 * whatever W or the product hold there (the masked-position rule below K16).  W is not modified; out [R, C] has W's dtype.  y = F.linear(x, out, bias) stays a
 * library GEMM.
 */
int vlmc_sparselora_effective_weight(const void* W, int dtype, int R, int C, int64_t ldw, const float* A,
                                     const float* B, int rank, float scaling, const uint8_t* keep_mask,
                                     int64_t ldm, int sparse, void* out, int64_t ldo, void* stream);

/*
 * K23  SparseLoRA masked training forward as one kernel (lora.py:359-382, F.linear(x, <the K15 weight expression>, bias)):
 *   y[T, R] = x[T, C] . W_eff[R, C]^T (+ bias[R]),  W_eff as vlmc_sparselora_effective_weight defines it (same roundings,
 * bit-identical operand), built on chip per 128 x 64 weight slice and fed to tcgen05 - no effective weight reaches HBM.
 * x, W, bias, y share `dtype` (VLMC_F16 or VLMC_BF16; VLMC_F32 returns VLMC_ERR_UNSUPPORTED - the caller keeps K15 + a
 * library GEMM there); fp32 accumulation, y rounded once to dtype (after the bias).  bias may be NULL.  rank <= 16;
 * C, R, ldx, ldw, ldy multiples of 8, ldm a multiple of 16, 16-byte aligned bases (TMA).
 */
int vlmc_sparselora_linear_forward(const void* x, int dtype, int64_t T, int C, int64_t ldx, const void* W, int R,
                                   int64_t ldw, const float* A, const float* B, int rank, float scaling,
                                   const uint8_t* keep_mask, int64_t ldm, int sparse, const void* bias, void* y,
                                   int64_t ldy, void* stream);

/*
 * K16  LoRA gradients of that forward.  G [R, C] (W's dtype) is the gradient w.r.t. the effective weight
 * (dy^T x, a library GEMM).  The reference's autograd masks G (sparse only), scales it in W's dtype, casts to fp32 and
 * runs two rank-r GEMMs; here  E = float(round_dtype(G * mask * scaling)),  dB [R, rank] = E A^T,
 * dA [rank, C] = B^T E  in one call (fp32 accumulation, fixed order).  rank <= 16.
 *
 * The masked-position rule of K14, K15 and K16, and through them of K23, K28, K29 and K30: a masked W counts as +0,
 * so masked entries of the sparse effective weight (and of K14's result with remask) are +0 and those of the dense one
 * are +0 + d; with sparse != 0 a masked entry of G contributes nothing (E = 0 there).  This holds whatever W, the LoRA
 * product or G hold at that position.  The reference's expressions differ in two ways the values alone do not show:
 * (W + d) * mask and W * mask give -0 where the masked factor is negative and NaN where it is +-inf, and G * mask turns
 * an inf or NaN of G into NaN.
 * K28 and K29 read only the stored kept values, so they cannot know W at a masked position; +0 / nothing is the rule
 * the whole family can share.  F.linear cannot tell it apart from the reference's, except through 0 * inf in x.
 * At kept positions inf and NaN propagate as in IEEE arithmetic; NaN payloads are not preserved.
 */
size_t vlmc_sparselora_lora_grads_workspace_bytes(int R, int C, int rank);
int vlmc_sparselora_lora_grads(const void* G, int dtype, int R, int C, int64_t ldg, const uint8_t* keep_mask,
                               int64_t ldm, int sparse, const float* A, const float* B, int rank, float scaling,
                               float* dA, float* dB, void* ws, size_t ws_bytes, void* stream);

/*
 * Compressed 2:4 weights (K24-K26, K31).  A weight W [R, C] (fp16 / bf16, C % 16 == 0) whose every group of 4 consecutive
 * columns holds at most two non-zeros - what Wanda / SparseGPT / DSnoT leave with prune_n = 2, prune_m = 4 - is stored as
 *   values [R, C/2]   W's dtype.  Group g (columns 4g..4g+3) keeps its two values at [2g, 2g+1], in ascending column order.
 *   meta   [R, C/16]  uint16.  Word j covers columns [16j, 16j+16); group g of the word uses bits [4g, 4g+4): the low
 *                     2 bits hold the index (0-3) of the first kept element, the high 2 bits the index of the second,
 *                     first < second.
 * 0.5625x the bytes of the dense weight.  This is the logical order of NVIDIA's 2:4 metadata, not the interleaved order
 * the sparse tensor-core instructions read.  The rules that make the format exact and deterministic:
 *   - an element is kept when w != 0: NaN is kept, +0 and -0 are pruned;
 *   - a group with fewer than two kept elements is padded with its lowest-index pruned positions, whose stored value is
 *     +0 (so every group names two distinct indices);
 *   - a group with more than two non-zeros is rejected: the status word gets VLMC_NOT_2OF4, W is not modified and
 *     values / meta are unspecified;
 *   - decompression writes +0 at pruned positions.  A round trip is exact at every non-zero; the only thing not kept is
 *     the sign of pruned zeros (a pruner that multiplies by the mask leaves -0 where the weight was negative).
 *
 * K24  vlmc_sparse24_compress    W -> values, meta.  *status (device int) is cleared, then set to VLMC_NOT_2OF4 if any
 *                                group is rejected (the call itself returns 0: it does not synchronise).
 * K25  vlmc_sparse24_decompress  values, meta -> W [R, ldw] (the pruned positions of W are written, +0).
 * K26  vlmc_sparse24_linear_forward  y[T, R] = x[T, C] . W^T (+ bias[R]) read from the compressed weight: each 128 x 128
 *                                weight slice is expanded on chip into the dense tensor-core operand (bit-identical to
 *                                K25's output) and multiplied with tcgen05 (kind::f16, fp32 accumulation).  x, values,
 *                                bias and y share `dtype`; bias may be NULL; y is rounded once, after the bias.  Small T
 *                                is split over K: fp32 partials in ws, summed in split order by the tile's last CTA, so
 *                                equal inputs give equal bits.  ws of vlmc_workspace_bytes(VLMC_OP_SPARSE24_LINEAR, T, R,
 *                                C).  TMA: ldx, ldv, ldm multiples of 8 elements, x / values / meta 16-byte aligned.
 */
int vlmc_sparse24_compress(const void* W, int dtype, int R, int C, int64_t ldw, void* values, int64_t ldv,
                           uint16_t* meta, int64_t ldm, int* status, void* stream);
int vlmc_sparse24_decompress(const void* values, int dtype, int R, int C, int64_t ldv, const uint16_t* meta,
                             int64_t ldm, void* W, int64_t ldw, void* stream);
int vlmc_sparse24_linear_forward(const void* x, int dtype, int64_t T, int C, int64_t ldx, const void* values,
                                 int64_t ldv, const uint16_t* meta, int64_t ldm, int R, const void* bias, void* y,
                                 int64_t ldy, void* ws, size_t ws_bytes, void* stream);

/*
 * K31  vlmc_sparse24_linear_sp_forward  y[T, R] = x[T, C] . W^T (+ bias[R]) on the sparse tensor cores
 *      (tcgen05.mma.sp, kind::f16, fp32 accumulation in TMEM), reading values and meta exactly as stored: the weight is
 *      the sparse operand (M = weight rows), the tokens the dense one.  Each 32-bit TMEM metadata column the instruction
 *      reads is two consecutive meta words of a row, the lower-column word in the low half - the stored order, no
 *      reordered copy.  No workspace and no split over K: one CTA owns an output tile and walks K in order, so equal
 *      inputs give equal bits.  x, values, bias and y share `dtype` (fp16 / bf16); bias may be NULL; y is rounded once,
 *      after the bias.  C % 32 == 0, R >= 1, any T >= 0; TMA: ldx, ldv, ldm multiples of 8 elements, x / values / meta
 *      16-byte aligned.  Anything else returns an error and launches nothing.
 *      Semantics: only the two positions meta names in each group of four take part in the product.  For inputs without
 *      inf or NaN, y equals x . decompress(values, meta)^T up to fp32 summation order.  An inf or NaN in x at a position
 *      meta does not name leaves y finite, where the expand path (0 * inf) gives NaN.  Padded positions are named and
 *      store +0, so there the product is the dense one (0 * inf = NaN).  A meta code whose two indices are both 0 is
 *      not a 2:4 pattern (the format never writes one); the kernel reads it as indices {0, 1}.
 */
int vlmc_sparse24_linear_sp_forward(const void* x, int dtype, int64_t T, int C, int64_t ldx, const void* values,
                                    int64_t ldv, const uint16_t* meta, int64_t ldm, int R, const void* bias, void* y,
                                    int64_t ldy, void* stream);

/*
 * SparseLoRA on compressed 2:4 weights (K27-K30).  A SparseLoRA layer pruned with lora_model=True keeps its pruned
 * weights unzeroed and a bool mask beside them, so the kept set cannot come from W's non-zeros.  The mask-driven rule:
 *   - the kept set IS keep_mask: every group of 4 columns must keep exactly two elements (what Wanda / SparseGPT / DSnoT
 *     leave with prune_n = 2, prune_m = 4).  Any other count sets VLMC_NOT_2OF4; W is never written;
 *   - values hold W's bits at the kept positions (+-0, NaN and inf included); there is no padding, so the kept set
 *     decoded from meta is exactly the mask.
 * The stored format is the one above, so K25, K26 and the compressed checkpoints read the result unchanged.
 *
 * K27  vlmc_sparse24_compress_masked  (W, keep_mask) -> (values, meta).  *status as for K24.  Any pitch and element
 *                                     alignment of W and keep_mask.
 * K28  vlmc_sparse24_lora_effective_weight  the weight of the masked training forward (lora.py:364-375) from the
 *                                     compressed pair: out [R, C] (values' dtype, pitch ldo) bit-identical to
 *                                     vlmc_sparselora_effective_weight on (decompress(values, meta), mask = meta).
 * K29  vlmc_sparse24_lora_grads       vlmc_sparselora_lora_grads with the mask read from meta: same results bit for bit,
 *                                     same workspace (vlmc_sparselora_lora_grads_workspace_bytes).
 * K30  vlmc_sparse24_lora_merge       Linear.merge() (sparse branch, lora.py:384-394) with the re-mask of
 *                                     train.py:634-637, in place on values: every stored slot becomes
 *                                     round(float(v) + scaling * sum_k B A) with K14's arithmetic, so decompress() of
 *                                     the result equals vlmc_sparselora_merge(remask = 1) on the dense pair.  Only the
 *                                     sparse branch exists: the dense-delta merge leaves a weight that is not 2:4.
 * fp16 / bf16, C % 16 == 0, rank <= 16; A = lora_A [rank, C], B = lora_B [R, rank] fp32 row-major, A 16-byte aligned.
 * K28 / K30: values 8-byte aligned with ldv % 4 == 0; K28's out 16-byte aligned with ldo % 8 == 0.  K29: G 16-byte aligned,
 * ldg % 8 == 0.  None allocates or retains anything.
 */
int vlmc_sparse24_compress_masked(const void* W, int dtype, int R, int C, int64_t ldw, const uint8_t* keep_mask,
                                  int64_t ldk, void* values, int64_t ldv, uint16_t* meta, int64_t ldm, int* status,
                                  void* stream);
int vlmc_sparse24_lora_effective_weight(const void* values, int dtype, int R, int C, int64_t ldv, const uint16_t* meta,
                                        int64_t ldm, const float* A, const float* B, int rank, float scaling, int sparse,
                                        void* out, int64_t ldo, void* stream);
int vlmc_sparse24_lora_grads(const void* G, int dtype, int R, int C, int64_t ldg, const uint16_t* meta, int64_t ldm,
                             int sparse, const float* A, const float* B, int rank, float scaling, float* dA, float* dB,
                             void* ws, size_t ws_bytes, void* stream);
int vlmc_sparse24_lora_merge(void* values, int dtype, int R, int C, int64_t ldv, const uint16_t* meta, int64_t ldm,
                             const float* A, const float* B, int rank, float scaling, void* stream);

/*
 * K17  Non-zero element counts of up to 64 tensors of one dtype per call ("Remaining Proportion",
 * evaluate_old.py:331-334: sum((param != 0).float().sum() for param in model.parameters())).  `items` is a HOST array
 * read during the call; out[i] (device, uint64) receives the count of items[i].  x != 0 as torch evaluates it (-0.0 is
 * zero, NaN is not).  Tensors must be contiguous; any element alignment.
 */
typedef struct vlmc_tensor_item { const void* ptr; int64_t numel; } vlmc_tensor_item;
int vlmc_count_nonzero_batch(const vlmc_tensor_item* items, int count, int dtype, unsigned long long* out, void* stream);

/*
 * K18-K22  Global sparsity allocation on fp32 importance scores (SURVEY 8f-4).  Replaces the CPU torch.topk / cat /
 * compare passes of LayerSparsity.get_mask / get_layerwise_mask / global_iterative_pruning and the score build of
 * compute_importance_scores (layer_single_base_pruner.py:149-190, :192-238, :422-475) and of
 * BLIPT5GlobalPruner.get_mask / get_layerwise_mask (global_pruner.py:108-148).
 *
 * `items` is a HOST array of any length, read during the call (the library walks it 64 tensors per launch).  Tensors are
 * contiguous, scores fp32 (4-byte aligned is enough).  `segment` groups tensors that share one rank / threshold:
 * all 0 for the whole-model select, one segment per tensor for the layer-wise variants.
 *
 *   vlmc_scores_kth      kth_out[s] = the k[s]-th smallest score (1-based) of segment s, exact, in torch.topk's order
 *                        (NaN greatest, -0.0 == +0.0): topk(all, k, largest=False)[0][-1] (:168-169); the j-th LARGEST of
 *                        :157-158 is rank numel - j + 1.  k: DEVICE int64 [nseg], 1 <= k[s] <= numel of the segment.
 *                        Three counting passes (11/11/10 key bits) over the scores, no host synchronisation.
 *   vlmc_scores_protect  scores[v >= thr[segment]] = FLT_MAX in place (:160)
 *   vlmc_scores_mask     out = (v > thr[segment]) as 1.0f / 0.0f (:174, out may be NULL) and, when aux is given,
 *                        aux *= that mask in aux's dtype (:223-225 `v.data *= masks[k]`: pruned weights become +-0)
 *   vlmc_scores_sum      out[i] (device double [count]) = sum of items[i].scores, fixed summation order
 *                        (group_scores += importance_measure[l].sum(), :296)
 *   vlmc_importance_accum     scores += float(aux)^2 (mode 0, "obd", :456) or |float(aux)| (mode 1, :458); aux = gradient
 *   vlmc_importance_finalize  out = float(aux)^2 * (scores / nb) (mode 0, :468), |float(aux)| * |scores / nb| (mode 1, :470)
 *                        or |scores / nb| (mode 2, :473); aux = parameter (unused for mode 2); every product and the
 *                        division rounded separately like the reference's tensor expression
 */
typedef struct vlmc_score_item {
  float* scores;     /* fp32 scores / accumulator */
  int64_t numel;
  int segment;
  int aux_dtype;     /* vlmc_dtype of aux */
  void* aux;         /* parameter or gradient tensor of numel elements, or NULL */
  float* out;        /* fp32 output of numel elements, or NULL */
} vlmc_score_item;
size_t vlmc_scores_workspace_bytes(const vlmc_score_item* items, int count, int nseg);
int vlmc_scores_kth(const vlmc_score_item* items, int count, int nseg, const int64_t* k, float* kth_out,
                    void* ws, size_t ws_bytes, void* stream);
int vlmc_scores_protect(const vlmc_score_item* items, int count, int nseg, const float* thr, void* stream);
int vlmc_scores_mask(const vlmc_score_item* items, int count, int nseg, const float* thr, void* stream);
int vlmc_scores_sum(const vlmc_score_item* items, int count, double* out, void* ws, size_t ws_bytes, void* stream);
int vlmc_importance_accum(const vlmc_score_item* items, int count, int mode, void* stream);
int vlmc_importance_finalize(const vlmc_score_item* items, int count, int mode, double num_batches, void* stream);

/*
 * K3  SparseGPT Hessian accumulation.  Replaces SparseGPT.add_batch, sparsegpt_pruner.py:68-79:
 *   H <- H * n_before/(n_before+b) + (2/(n_before+b)) * X^T X
 * x: [T, C] row-major fp16 / bf16 / fp32 (one add_batch call, T = b * seq_len); H: [C, C] fp32, full and symmetric.
 * TMA-fed tcgen05.mma (kind::f16, fp32 accumulate in TMEM), SYRK over the upper triangle with the mirror
 * written by the epilogue.  kc = tokens accumulated inside the tensor core before the partial sum is
 * added, round-to-nearest, into fp32 registers (0 = default 512; multiples of 64).  slab_tokens = tokens per
 * launch (0 = default: 65536 for C >= 8192, else unlimited): all tiles of one slab run before the next so operand re-reads stay in L2.
 * fp32 activations (EVA-ViT qkv / fc1 inputs under autocast) are not exact tensor-core operands: they run as a 3xTF32
 * split GEMM (tcgen05 kind::tf32, hi/lo split on chip, full square instead of SYRK; kc capped at 256, default 128).
 */
int vlmc_hessian_accum(const void* x, int dtype, int64_t T, int C, int64_t ldx,
                       float* H, int64_t ldh, double n_before, double b, int kc, int64_t slab_tokens,
                       void* stream);

/*
 * K10 prologue.  Replaces sparsegpt_pruner.py:95-96 and :111: channels whose diag(H) is 0 get H[c,c] = 1
 * (dead_out[c] = 1, may be NULL; the caller zeroes those weight columns, :97) and
 * *damp_out = percdamp * mean(diag(H)).  vlmc_hessian_add_damp adds *damp to the diagonal (the retry step, :126-128).
 */
int vlmc_hessian_prepare(float* H, int C, int64_t ldh, float percdamp, float* damp_out, uint8_t* dead_out,
                         void* stream);
int vlmc_hessian_add_damp(float* H, int C, int64_t ldh, const float* damp, void* stream);

/*
 * K10  U = upper Cholesky factor of H^-1 (H^-1 = U^T U).  Replaces the cholesky -> cholesky_inverse ->
 * cholesky(upper=True) chain of sparsegpt_pruner.py:114-157 with one blocked Cholesky of the flipped matrix and
 * one triangular inverse (same U mathematically, 2/3 C^3 flops).  H is not modified.  *status (device int) is set
 * to 0, or to a combination of the status bits: VLMC_NOT_POSDEF when a pivot is non-positive / NaN (the caller then damps
 * and retries exactly like the reference's while-loop), VLMC_NONFINITE when H holds +-inf / NaN (the caller clamps like
 * :101-109 first), VLMC_HUGE_FACTOR when the factor is so large that the reference's second stage may differ.  The function itself returns 0 in both cases (it does not synchronise).
 */
int vlmc_chol_inv_upper(const float* H, int C, int64_t ldh, float* U, int64_t ldu, int* status,
                        void* ws, size_t ws_bytes, void* stream);

/*
 * The reference's factorisation in its own three-step order, for the Hessians on which the fused vlmc_chol_inv_upper and
 * the chain cholesky -> cholesky_inverse -> [+-inf clamp] -> cholesky(upper=True) with its second damp-and-retry loop
 * (sparsegpt_pruner.py:131-157) can differ: status bit VLMC_HUGE_FACTOR, or on request (SparseGPT.exact_reference_order).
 *   vlmc_gram_upper              Hinv = U^T U (full symmetric matrix) for an upper factor U: the value of
 *                                torch.cholesky_inverse(cholesky(H)) when U = vlmc_chol_inv_upper(H)         (:131)
 *   vlmc_chol_upper              U = cholesky(A, upper=True) of a symmetric matrix A (A is not modified); *status gets
 *                                VLMC_NOT_POSDEF / VLMC_NONFINITE like vlmc_chol_inv_upper; ws of VLMC_OP_CHOL size   (:146)
 *   vlmc_matrix_nonfinite_count  out3 = {#+inf, #-inf, #NaN} of A (device uint64[3])                          (:101,:106,:133,:138)
 *   vlmc_matrix_replace_inf      A[A == +inf] = value (negative = 0) or A[A == -inf] = value (negative != 0)  (:103-104,:108-109)
 *   vlmc_diag_abs_mean           *out = scale * mean(|diag(A)|)                                              (:143)
 * The quantile the clamp needs is two order statistics of the whole matrix: vlmc_scores_kth.
 */
int vlmc_gram_upper(const float* U, int C, int64_t ldu, float* Hinv, int64_t ldh, void* stream);
int vlmc_chol_upper(const float* A, int C, int64_t lda, float* U, int64_t ldu, int* status,
                    void* ws, size_t ws_bytes, void* stream);
int vlmc_matrix_nonfinite_count(const float* A, int rows, int cols, int64_t lda, unsigned long long* out3, void* stream);
int vlmc_matrix_replace_inf(float* A, int rows, int cols, int64_t lda, float value, int negative, void* stream);
int vlmc_diag_abs_mean(const float* A, int C, int64_t lda, float scale, float* out, void* stream);
/*
 * Schedule of the blocked Cholesky inside vlmc_chol_inv_upper.  With the look-ahead (default) the trailing update of a panel
 * is split between the caller's stream and a library-owned side stream (forked from and joined to the caller's stream
 * with events, so the call stays stream-ordered) and the next diagonal factor runs under it: 21.2 -> 18.2 ms at
 * C = 11008 for a chain that has the GPU to itself.  Callers that run SEVERAL chains concurrently on their own streams
 * turn it off (the extra streams only add contention there: 63-65 ms -> 72-74 ms for the 7 chains of a Vicuna block).
 * mode: 1 on, 0 off, -1 follow the environment variable VLMC_CHOL_LOOKAHEAD (unset = on).  Returns the previous mode
 * (2 = was following the environment).  Host-side switch, read when a call is enqueued; equal factors either way.
 */
int vlmc_chol_set_lookahead(int mode);

/*
 * K13 / K10 building block: fp32-accurate GEMM on the tensor cores (3xTF32 split, tcgen05 + TMEM + TMA).
 * Replaces the fp32 torch.matmul of sparsegpt_pruner.py:210 (W[:, i2:] -= Err1 @ Hinv[i1:i2, i2:]) and the GEMMs inside
 * cuSOLVER's potrf / potri behind :114-157.
 *   C[M,N] = beta * C + alpha * A[M,K] * op(B)      A row-major [M,K]; b_nk != 0: B row-major [N,K] (C = A B^T),
 *                                                   else B row-major [K,N]
 *   tri != 0: only tiles touching the lower triangle are computed (symmetric rank-k update of a lower triangle)
 *   kc: K elements accumulated inside the tensor core between round-to-nearest flushes (0 = 128; multiples of 32)
 *   beta == 0: C is not read (NaN in C does not propagate)
 * K, N, lda, ldb, ldc multiples of 4; pointers 16-byte aligned; ldc >= N.  Anything else returns an error and launches
 * nothing.
 * Non-finite operands: every element a is split into hi = tf32(a) (round to nearest, ties away from zero) and
 * lo = a - hi.  For a = +-inf, lo = inf - inf is NaN, so every output whose dot product meets an inf or NaN of A or B is
 * NaN, whatever the other factor (also 0).  Finite values that round past the largest TF32 number (|a| >= 2^128 - 2^116,
 * e.g. FLT_MAX) split into hi = +-inf and lo = -+inf and behave the same way.  All other outputs are unaffected.
 */
int vlmc_gemm_tf32x3(int b_nk, int M, int N, int K, float alpha, const float* A, int64_t lda,
                     const float* B, int64_t ldb, float beta, float* C, int64_t ldc, int tri, int kc,
                     void* stream);

/*
 * K11-K13  The column-block OBS sweep.  Replaces sparsegpt_pruner.py:160-215: per 128-column block the
 * unstructured mask (score <= k-th smallest block score, k = int(R*128*sparsity)) or the n:m mask, the 128
 * sequential error-propagation steps, and the lazy trailing update W[:, i2:] -= Err1 @ U[i1:i2, i2:].
 * W (fp16 / bf16 / fp32, [R, C]) is overwritten with the compensated sparse weights (math in fp32, one rounding).
 * dead: optional [C] bytes from vlmc_hessian_prepare (those input channels are zeroed first, :97).
 * keep_mask (optional) receives 1 = kept / 0 = pruned; importance_score (optional) = mean(W^2 / diag(U)^2), :163-165.
 * Shapes: blocksize must be 128 and C a multiple of 4 (VLMC_ERR_UNSUPPORTED otherwise, as for ldu % 4 != 0 or U not
 * 16-byte aligned).  The last block may be partial (bs = C mod 128 columns); its threshold rank is int(R * bs * sparsity)
 * (0-indexed, the double product truncated as Python's int() does) among its R * bs scores.  n:m needs 0 < n < m, m
 * dividing 128 and m <= 16 (so m is 2, 4, 8 or 16); unstructured needs 0 <= sparsity < 1; both VLMC_ERR_BAD_ARG
 * otherwise, as is ldm < C.  Arguments are checked before anything is launched.
 * Every step but the trailing update rounds as the reference's fp32 code: where Err1 @ U[i1:i2, i2:] is exactly zero
 * (a block-diagonal U, or C <= 128) weights, mask and thresholds equal it bit for bit.  Pruned weights are +0.
 */
int vlmc_obs_sweep(void* W, int dtype, int R, int C, int64_t ldw, const float* U, int64_t ldu,
                   const uint8_t* dead, double sparsity, int prune_n, int prune_m, int blocksize,
                   uint8_t* keep_mask, int64_t ldm, float* importance_score,
                   void* ws, size_t ws_bytes, void* stream);

/*
 * vlmc_obs_sweep that can be enqueued BEFORE the host has looked at the factorisation's status word: fail_flag is that
 * device word (vlmc_chol_inv_upper's `status`); when it is non-zero at run time the sweep leaves W and keep_mask
 * untouched (only scratch is written), so the caller can damp, re-factorise and sweep again (sparsegpt_pruner.py:114-128
 * semantics) without a host round trip on the success path.  fail_flag == NULL: identical to vlmc_obs_sweep.
 * importance_score is computed (by vlmc_obs_begin) before the flag is read, so it is written even when the flag is set:
 * mean(W^2 / diag(U)^2) of the untouched W and the rejected U.  Nothing the failed call leaves in ws is read by the next.
 */
int vlmc_obs_sweep_guarded(void* W, int dtype, int R, int C, int64_t ldw, const float* U, int64_t ldu,
                           const uint8_t* dead, double sparsity, int prune_n, int prune_m, int blocksize,
                           uint8_t* keep_mask, int64_t ldm, float* importance_score, const int* fail_flag,
                           void* ws, size_t ws_bytes, void* stream);

/*
 * K11-K13 in steps, for runs that shard the OUTPUT ROWS of one linear across GPUs (rows are independent given U, except
 * for the unstructured block threshold, which is a k-th value over all rows x 128 columns, SURVEY F6).  Each rank holds
 * R of the rows_total rows.  `hist` is caller memory, [ceil(C/128)][3][2048] uint32, zero before vlmc_obs_begin
 * (NULL = a private buffer inside ws, single device).  Per block b the sequence is
 *     for pass in 0,1,2:  vlmc_obs_block_hist(b, pass)   then SUM-all-reduce hist[b][pass] over the row shards
 *     vlmc_obs_block_finish(b)                            (threshold from the three histograms, sweep, trailing update)
 * and the three 8 KB histograms are the only data exchanged.  n:m needs no histogram and no exchange.
 * vlmc_obs_begin: fp32 working copy of W (dead channels zeroed) and, if importance_sum != NULL, the SUM of
 * W^2 / diag(U)^2 over this rank's rows (device float; the caller reduces and divides by the element count).
 */
int vlmc_obs_begin(void* W, int dtype, int R, int C, int64_t ldw, const float* U, int64_t ldu,
                   const uint8_t* dead, float* importance_sum, void* ws, size_t ws_bytes, void* stream);
int vlmc_obs_block_hist(int R, int C, const float* U, int64_t ldu, int blk, int pass, int64_t rows_total,
                        double sparsity, unsigned int* hist, void* ws, size_t ws_bytes, void* stream);
int vlmc_obs_block_finish(void* W, int dtype, int R, int C, int64_t ldw, const float* U, int64_t ldu, int blk,
                          int64_t rows_total, double sparsity, int prune_n, int prune_m, uint8_t* keep_mask,
                          int64_t ldm, unsigned int* hist, void* ws, size_t ws_bytes, void* stream);

/*
 * K8+K9  DSnoT mask refinement.  Replaces the per-linear body of the DSnoT pruners, dsnot_pruner.py:359-755 (T5 / LLM)
 * and :1092-1485 (ViT): DSnoT_metric = W * sum_metric_row, the Wanda (or magnitude) initial mask, the three stable row
 * orderings + return_reorder_indice (:555-612, :1881-1925) and the prune / regrow cycle loop (:650-751; n:m :407-552).
 * Two passes, because the reference's `while any(update_mask)` couples all rows through the number of executed cycles:
 *   _walk   per row: initial selection, ordered candidate prefixes, the cycle loop; records every cycle's
 *           (pruned column, regrown column) in ws and atomically maxes *ncycles (device int, zeroed by the call).
 *           When rows are sharded across GPUs the caller all-reduces (MAX) *ncycles between the two passes.
 *   _apply  per row: initial mask + the recorded writes of the first *ncycles cycles -> keep_mask (1 = kept) and,
 *           if zero_w, zeroed weights (:753-755).  Same ws as _walk.
 * vlmc_dsnot_refine runs both back to back (one device).
 *   k                  unstructured prune count per row = round(C * sparsity) (python round, :562); ignored for n:m
 *   prune_n, prune_m   0,0 = unstructured; otherwise n of every m consecutive columns, m <= 8
 *   pow_of_var, max_cycle_time (<= 128), update_threshold, without_same_sign: the reference's knobs (:1629-1636)
 *   initial_magnitude  0: initial_method "wanda" (:370-374); 1: "magnitude" (:375-376)
 *   argmin_rule        tie-break of topk(1, largest=False) at :517 when a whole group is +inf: 0 lowest column,
 *                      1 what torch's CPU kernel returns (std::nth_element order) - matches the CPU reference
 *   ref_fixup          1: as shipped, the block at :734-740 writes every swap back (SURVEY F4); 0: upstream DSnoT
 * Unsupported (the reference indexes out of bounds there, SURVEY F12): C < max_cycle_time, C - k < max_cycle_time.
 */
int vlmc_dsnot_refine_walk(const void* W, int dtype, int R, int C, int64_t ldw, const float* scaler_row,
                           const float* sum_metric_row, const float* var, int k, int prune_n, int prune_m,
                           float pow_of_var, int max_cycle_time, float update_threshold, int without_same_sign,
                           int initial_magnitude, int argmin_rule, int* ncycles, void* ws, size_t ws_bytes,
                           void* stream);
int vlmc_dsnot_refine_apply(void* W, int dtype, int R, int C, int64_t ldw, const float* scaler_row,
                            int prune_n, int prune_m, int initial_magnitude, int max_cycle_time,
                            const int* ncycles, int ref_fixup, int zero_w, uint8_t* keep_mask, int64_t ldm,
                            void* ws, size_t ws_bytes, void* stream);
int vlmc_dsnot_refine(void* W, int dtype, int R, int C, int64_t ldw, const float* scaler_row,
                      const float* sum_metric_row, const float* var, int k, int prune_n, int prune_m,
                      float pow_of_var, int max_cycle_time, float update_threshold, int without_same_sign,
                      int initial_magnitude, int argmin_rule, int ref_fixup, int zero_w, uint8_t* keep_mask,
                      int64_t ldm, int* ncycles, void* ws, size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VLMC_H_ */
