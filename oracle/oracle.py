"""TEST INFRASTRUCTURE ONLY - CPU (numpy) restatement of the reference's calibration-and-masking path.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this module, and only as the checker (or the timed CPU baseline), never as part of the product
path: vlmc/ must not import it.

Parity status: PINNED.  The reference ships no tests or golden vectors for this path (SURVEY.md
section 4), but its modules load unmodified in the build container (oracle/ref_loader.py), so every
function below is checked against the reference itself: tests/golden/make_golden.py runs the
reference on seeded inputs and commits the outputs as fixtures (tests/golden/*.npz);
tests/test_oracle_vs_golden.py replays them through this file, and tests/test_oracle_vs_reference.py
does the same live whenever /root/reference is present.  The one golden vector the reference itself
holds, the return_reorder_indice docstring example (dsnot_pruner.py:1882-1893), is checked too.

All arrays are numpy.  Half / bfloat16 tensors are passed as float32 arrays holding the exactly
up-cast values plus a dtype tag ("f16" | "bf16" | "f32") where an output must be rounded back.
"""
import numpy as np

F32 = np.float32


# ---------------------------------------------------------------------------------------------
# dtype helpers (numpy has no bfloat16)
# ---------------------------------------------------------------------------------------------
def round_to_dtype(x32, tag):
    """Round float32 values to `tag` precision (round-to-nearest-even), returned as float32."""
    x32 = np.asarray(x32, dtype=F32)
    if tag == "f32":
        return x32
    if tag == "f16":
        return x32.astype(np.float16).astype(F32)
    if tag == "bf16":
        u = x32.view(np.uint32).astype(np.uint64)
        rounded = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
        out = rounded.astype(np.uint32).view(F32)
        return np.where(np.isnan(x32), x32, out)
    raise ValueError(tag)


# ---------------------------------------------------------------------------------------------
# a1 / K1  Wanda statistic                      wanda_pruner.py:66-81
# ---------------------------------------------------------------------------------------------
def wanda_add_batch(scaler_row, nsamples, x, b):
    """One WrappedGPT.add_batch call.  x: [T, C] float32 (inp.reshape(-1, C) up-cast, :74,:80).

    scaler_row *= n/(n+b); n += b; scaler_row += ||x[:, c]||_2^2 / n      (:77-81)
    The reference takes torch.norm(...)**2 (sqrt then square); the restatement sums squares in
    float64 and rounds once -- the two differ by <= ~2 ulp (SURVEY App. A), far inside 1e-5.
    """
    x = np.asarray(x)
    sq = (x.astype(np.float64) ** 2).sum(axis=0)
    out = scaler_row.astype(F32) * F32(nsamples / (nsamples + b))
    nsamples += b
    out = out + (sq.astype(F32) / F32(nsamples))
    return out.astype(F32), nsamples


# ---------------------------------------------------------------------------------------------
# a2 / K2  DSnoT statistics                     dsnot_pruner.py:79-101
# ---------------------------------------------------------------------------------------------
def dsnot_add_batch(state, x, b):
    """state: dict(scaler_row, sum_metric_row, mean, var, nsamples, ntokens); x: [T, C] float32.

    mean/var are token-weighted running means of the per-call mean and BIASED variance (:89-93);
    scaler_row / sum_metric_row are running means over samples of sum x^2 and sum x (:96-101).
    """
    x64 = np.asarray(x).astype(np.float64)
    T = x64.shape[0]
    mean_inp = x64.mean(axis=0)
    var_inp = x64.var(axis=0)  # biased (unbiased=False, :90)
    nt = state["ntokens"]
    if nt == 0:
        var, mean = var_inp, mean_inp
    else:
        var = (state["var"].astype(np.float64) * nt + var_inp * T) / (nt + T)
        mean = (state["mean"].astype(np.float64) * nt + mean_inp * T) / (nt + T)
    n = state["nsamples"]
    ratio = F32(n / (n + b))
    scaler = state["scaler_row"].astype(F32) * ratio
    summ = state["sum_metric_row"].astype(F32) * ratio
    n += b
    scaler = scaler + (x64 ** 2).sum(axis=0).astype(F32) / F32(n)
    summ = summ + x64.sum(axis=0).astype(F32) / F32(n)
    return dict(scaler_row=scaler.astype(F32), sum_metric_row=summ.astype(F32), mean=mean.astype(F32),
                var=var.astype(F32), nsamples=n, ntokens=nt + T)


# ---------------------------------------------------------------------------------------------
# a4 / K4-K6  Wanda score + selection            wanda_pruner.py:316-341
# ---------------------------------------------------------------------------------------------
def wanda_scores(W32, scaler_row):
    """|W| * sqrt(scaler_row) in float32: one IEEE sqrt, one IEEE multiply (:318)."""
    return (np.abs(W32.astype(F32)) * np.sqrt(scaler_row.astype(F32))[None, :]).astype(F32)


def score_mean(S):
    return float(S.astype(np.float64).mean())  # weight.importance_score (:320)


def wanda_rowselect(W32, scaler_row, k):
    """Unstructured LLM path: per row the k = int(C*p) smallest scores are pruned, stable order (:332-337).

    Returns (keep_mask bool [R,C], pruned W float32, importance_score).
    """
    S = wanda_scores(W32, scaler_row)
    order = np.argsort(S, axis=1, kind="stable")  # torch.sort(stable=True): ties -> lower column, NaN last
    prune = np.zeros(S.shape, dtype=bool)
    np.put_along_axis(prune, order[:, :k], True, axis=1)
    Wp = np.where(prune, F32(0), W32.astype(F32))
    return ~prune, Wp, score_mean(S)


def nm_select_scores(S, n, m):
    """Per group of m consecutive columns mark the n smallest; ties -> lower column.

    The reference uses torch.topk(largest=False) (:329) whose tie-break is implementation-defined
    (SURVEY F8); the build fixes 'lowest column wins', which equals the reference on tie-free groups.
    """
    R, C = S.shape
    G = S.reshape(R, C // m, m)
    order = np.argsort(G, axis=2, kind="stable")
    prune = np.zeros(G.shape, dtype=bool)
    np.put_along_axis(prune, order[:, :, :n], True, axis=2)
    return prune.reshape(R, C)


def wanda_nm(W32, scaler_row, n, m):
    S = wanda_scores(W32, scaler_row)
    prune = nm_select_scores(S, n, m)
    Wp = np.where(prune, F32(0), W32.astype(F32))
    return ~prune, Wp, score_mean(S)


# ---------------------------------------------------------------------------------------------
# a5 / K7  ViT whole-matrix threshold            wanda_pruner.py:682-683
# ---------------------------------------------------------------------------------------------
def wanda_threshold(W32, scaler_row, k_global):
    """thres = sort(S.flatten())[k_global]; prune S < thres (strict, ties kept)."""
    S = wanda_scores(W32, scaler_row)
    thres = np.partition(S.ravel(), k_global)[k_global]
    prune = S < thres
    Wp = np.where(prune, F32(0), W32.astype(F32))
    return ~prune, Wp, score_mean(S)


# ---------------------------------------------------------------------------------------------
# a8 / K14  SparseLoRA merge + re-mask           lora.py:384-387, train.py:634-637
# ---------------------------------------------------------------------------------------------
def _fma32(b, a, c):
    """fmaf(b, a, c) on float32 arrays, correctly rounded.  The product of two float32 values is exact in float64;
    TwoSum gives the float64 sum and its exact error, and the sum is rounded to odd (nudged to the odd neighbour when
    inexact), which makes the final rounding to float32 a single correct one.  float32(float64(b * a) + c) is not: the
    float64 sum can land exactly on a float32 midpoint (b = 1 - 2^-12 + 2^-24, a = 2^-24 (1 + 2^-12), c = 1 gives 1.0,
    not 1 + 2^-23)."""
    p = np.asarray(b, np.float64) * np.asarray(a, np.float64)
    c = np.asarray(c, np.float64)
    with np.errstate(invalid="ignore"):
        s = p + c
        bb = s - p
        err = (p - (s - bb)) + (c - bb)
        even = (s.view(np.int64) & 1) == 0
        s = np.where(np.isfinite(s) & (err != 0) & even, np.nextafter(s, np.where(err > 0, np.inf, -np.inf)), s)
    return s.astype(F32)


def sparselora_merge(W32, w_tag, A, B, scaling, keep_mask, remask=True):
    """W <- round_w( W + (B@A * scaling) * mask ), then W[~mask] = 0.

    fp32 math as torch does it: the rank-r product accumulates k ascending with fused multiply-adds
    (each correctly rounded, _fma32), `* scaling` and the final add are separately rounded float32 ops,
    one rounding to W's dtype.
    """
    R, C = W32.shape
    acc = np.zeros((R, C), dtype=F32)
    for kk in range(A.shape[0]):
        acc = _fma32(B[:, kk][:, None], A[kk][None, :], acc)
    delta = (acc * F32(scaling)).astype(F32)
    merged = round_to_dtype((W32.astype(F32) + delta).astype(F32), w_tag)
    out = np.where(keep_mask, merged, F32(0) if remask else W32.astype(F32))
    return out.astype(F32)


# ---------------------------------------------------------------------------------------------
# f-2 / K15, K16  SparseLoRA masked training forward and its LoRA gradients      lora.py:359-382
# ---------------------------------------------------------------------------------------------
def _lora_product(A, B):
    """B @ A in float32, k ascending with one correctly rounded fused multiply-add per step (_fma32)."""
    acc = np.zeros((B.shape[0], A.shape[1]), dtype=F32)
    for kk in range(A.shape[0]):
        acc = _fma32(B[:, kk][:, None], A[kk][None, :], acc)
    return acc


def sparselora_effective_weight(W32, w_tag, A, B, scaling, keep_mask, sparse=True):
    """The weight Linear.forward hands to F.linear (lora.py:364-375), with torch's roundings in W's dtype:
    (B @ A).to(dtype), * scaling, W + ., * mask   (sparse)   or   W * mask + .   (not sparse)."""
    d = round_to_dtype(_lora_product(A, B), w_tag)
    d = round_to_dtype((d * F32(scaling)).astype(F32), w_tag)
    W32 = W32.astype(F32)
    if sparse:
        return np.where(keep_mask, round_to_dtype((W32 + d).astype(F32), w_tag), F32(0)).astype(F32)
    return round_to_dtype((np.where(keep_mask, W32, F32(0)) + d).astype(F32), w_tag)


def sparselora_linear_forward(x32, W32, w_tag, A, B, scaling, keep_mask, sparse=True, bias32=None):
    """Linear.forward with r > 0, not merged (lora.py:359-382): F.linear(x, <the effective weight above>, bias) in W's
    dtype - float64 accumulation of the exact products (the truth a kernel with fp32 accumulation is compared with), bias
    added before the ONE rounding to the dtype.  K23 (vlmc_sparselora_linear_forward) computes exactly this."""
    weff = sparselora_effective_weight(W32, w_tag, A, B, scaling, keep_mask, sparse).astype(np.float64)
    y = np.asarray(x32, dtype=np.float64) @ weff.T
    if bias32 is not None:
        y = y + np.asarray(bias32, dtype=np.float64)
    return round_to_dtype(y.astype(F32), w_tag)


def sparselora_lora_grads(G32, w_tag, A, B, scaling, keep_mask, sparse=True):
    """Autograd of that expression w.r.t. lora_A / lora_B given G = dL/dW_eff (in W's dtype): mask (sparse only), scale
    in W's dtype, cast to float32, dB = E A^T, dA = B^T E.  Returned in float64-accumulated float32 (the truth the
    kernels are compared with at 1e-5)."""
    E = np.where(keep_mask, G32, F32(0)) if sparse else G32
    E = round_to_dtype((E.astype(F32) * F32(scaling)).astype(F32), w_tag).astype(np.float64)
    dB = (E @ A.astype(np.float64).T).astype(F32)
    dA = (B.astype(np.float64).T @ E).astype(F32)
    return dA, dB


# ---------------------------------------------------------------------------------------------
# a3 / K3  SparseGPT Hessian                     sparsegpt_pruner.py:68-79
# ---------------------------------------------------------------------------------------------
def sparsegpt_add_batch(H, nsamples, x, b):
    """H *= n/(n+b); n += b; x = sqrt(2/n) * x.float(); H += x^T x   (fp32, like the reference's SGEMM)."""
    H = H.astype(F32) * F32(nsamples / (nsamples + b))
    nsamples += b
    xs = (F32(np.sqrt(2.0 / nsamples)) * np.asarray(x, dtype=F32)).astype(F32)
    H = H + xs.T @ xs
    return H.astype(F32), nsamples


def hessian_truth(xs, n_total):
    """float64 ground truth (2/N) sum_t x x^T over a list of [T, C] calls."""
    C = xs[0].shape[1]
    H = np.zeros((C, C), dtype=np.float64)
    for x in xs:
        x64 = np.asarray(x, dtype=np.float64)
        H += x64.T @ x64
    return H * (2.0 / n_total)


# ---------------------------------------------------------------------------------------------
# a7 / K10-K13  SparseGPT.fasterprune             sparsegpt_pruner.py:81-215
# ---------------------------------------------------------------------------------------------
def _chol_retry(H, damp, upper):
    """cholesky with the reference's conditional damping: add `damp` to the diagonal only after a failure or
    NaNs, cumulatively (:114-128, :143-157).  Returns (factor, number of damping steps)."""
    from scipy.linalg import lapack
    steps = 0
    while True:
        c, info = lapack.spotrf(H, lower=0 if upper else 1, clean=1)
        if info == 0 and not np.isnan(c).any():
            return c.astype(F32), steps
        H = H.copy()
        H[np.diag_indices_from(H)] += F32(damp)
        steps += 1
        if steps > 200:
            raise RuntimeError("damping did not make the matrix positive definite")


def torch_quantile(a, q):
    """torch.quantile(a, q) for a float32 array, interpolation "linear", over ALL entries (infinite ones included), with
    ATen's own arithmetic (aten/src/ATen/native/Sorting.cpp quantile_compute): rank = float32(q) * float32(n - 1),
    values gathered at floor / ceil of the rank from the sorted data, combined by at::lerp in float32."""
    v = np.sort(np.asarray(a, dtype=F32).ravel())
    if np.isnan(v).any():
        return F32(np.nan)
    rank = F32(q) * F32(v.size - 1)
    lo, hi = int(np.floor(rank)), int(np.ceil(rank))
    w = F32(rank - F32(lo))
    x, y = v[lo], v[hi]
    with np.errstate(all="ignore"):
        return F32(x + w * (y - x)) if w < F32(0.5) else F32(y - (y - x) * (F32(1) - w))


def clamp_infinite(M):
    """:101-109 / :133-141: +inf -> quantile(M, 0.999), then -inf -> quantile(M, 0.001) of the updated matrix.  In place."""
    pos = np.isposinf(M)
    if pos.any():
        M[pos] = torch_quantile(M, 0.999)
    neg = np.isneginf(M)
    if neg.any():
        M[neg] = torch_quantile(M, 0.001)
    return M


def sparsegpt_second_stage(Hinv, percdamp=0.01):
    """:133-157 on a given H^-1: clamp, damp2 = percdamp * mean|diag|, cholesky(upper=True) with damp-and-retry.
    Returns (U, damping steps)."""
    Hinv = clamp_infinite(np.array(Hinv, dtype=F32))
    damp2 = F32(percdamp) * np.mean(np.abs(np.diag(Hinv)), dtype=F32)   # :143
    U, steps2 = _chol_retry(Hinv, damp2, upper=True)                    # :146-157
    return np.triu(U).astype(F32), steps2


def sparsegpt_inverse_factor(H, percdamp=0.01):
    """U = cholesky(cholesky_inverse(cholesky(H)), upper=True) in float32 LAPACK, with the dead-channel rule, both +-inf
    clamps and both conditional damping loops (:95-157).  Returns (U, dead mask, damping steps of the first factorisation)."""
    from scipy.linalg import lapack
    H = np.array(H, dtype=F32)
    dead = np.diag(H) == 0                                   # :95
    H[dead, dead] = 1                                        # :96
    clamp_infinite(H)                                        # :101-109
    damp = F32(percdamp) * np.mean(np.diag(H), dtype=F32)    # :111
    L, steps = _chol_retry(H, damp, upper=False)             # :114-128
    with np.errstate(all="ignore"):
        Hinv, info = lapack.spotri(L, lower=1)               # :131  cholesky_inverse
    Hinv = np.tril(Hinv) + np.tril(Hinv, -1).T
    U, _ = sparsegpt_second_stage(Hinv, percdamp)            # :133-157
    return U, dead, steps


def sparsegpt_fasterprune(W32, w_tag, H, sparsity, prune_n=0, prune_m=0, blocksize=128, percdamp=0.01, U=None,
                          dead=None, kth_fn=None):
    """The column-block OBS sweep (:160-215) in float32.  Returns (pruned W rounded to w_tag, importance score, U).
    kth_fn(tmp, k) -> threshold replaces the local k-th value when W32 is only a row shard (multi-rank tests)."""
    if U is None:
        U, dead, _ = sparsegpt_inverse_factor(H, percdamp)
    W = np.array(W32, dtype=F32)
    if dead is not None:
        W[:, dead] = 0                                       # :97
    R, C = W.shape
    dU = np.diag(U).astype(F32)
    score = float(((W ** 2) / (dU[None, :] ** 2)).astype(np.float64).mean())      # :160-165
    for i1 in range(0, C, blocksize):
        i2 = min(i1 + blocksize, C)
        count = i2 - i1
        W1 = W[:, i1:i2].copy()
        Q1 = np.zeros_like(W1)
        Err1 = np.zeros_like(W1)
        U1 = U[i1:i2, i1:i2]
        d1 = np.diag(U1).astype(F32)
        if prune_n == 0:
            tmp = ((W1 * W1) / ((d1 * d1)[None, :])).astype(F32)
            kk = int(tmp.size * sparsity)
            thresh = np.partition(tmp.ravel(), kk)[kk] if kth_fn is None else kth_fn(tmp, kk)          # :184
            mask1 = tmp <= thresh                                                                    # :185
        else:
            mask1 = np.zeros(W1.shape, dtype=bool)
        for i in range(count):
            w = W1[:, i]
            d = U1[i, i]
            if prune_n != 0 and i % prune_m == 0:
                grp = ((W1[:, i:i + prune_m] ** 2) / ((d1[i:i + prune_m] ** 2)[None, :])).astype(F32)   # :194
                order = np.argsort(grp, axis=1, kind="stable")[:, :prune_n]       # ties -> lower column (SURVEY F8)
                np.put_along_axis(mask1[:, i:i + prune_m], order, True, axis=1)
            q = np.where(mask1[:, i], F32(0), w).astype(F32)
            Q1[:, i] = q
            err = ((w - q) / d).astype(F32)
            W1[:, i:] = (W1[:, i:] - (err[:, None] * U1[i, i:][None, :]).astype(F32)).astype(F32)   # :204
            Err1[:, i] = err
        W[:, i1:i2] = Q1
        if i2 < C:
            W[:, i2:] = (W[:, i2:] - Err1 @ U[i1:i2, i2:]).astype(F32)             # :210
    return round_to_dtype(W, w_tag), score, U


# ---------------------------------------------------------------------------------------------
# return_reorder_indice                          dsnot_pruner.py:1881-1925
# ---------------------------------------------------------------------------------------------
def return_reorder_indice(t):
    """Positions of the negative entries in order, then positions of the positive entries reversed;
    slots left over (zeros in the input) are filled with index 0, like the reference's inf->0 trick."""
    t = np.asarray(t)
    R, C = t.shape
    out = np.zeros((R, C), dtype=np.int64)
    for r in range(R):
        neg = np.nonzero(t[r] < 0)[0]
        pos = np.nonzero(t[r] > 0)[0]
        row = np.zeros(C, dtype=np.int64)
        row[:neg.size] += neg
        # positive_value is sorted ascending with inf padding, then flipped: positives end up right-aligned
        # in DEscending index order; inf -> 0
        if pos.size:
            row[C - pos.size:] += pos[::-1]
        out[r] = row
    return out


# ---------------------------------------------------------------------------------------------
# a6 / K8-K9  DSnoT refine                        dsnot_pruner.py:359-755 (ViT copy :1092-1485)
# ---------------------------------------------------------------------------------------------
def _rowsum_f32(a):
    """torch.sum(x, dim=1, keepdim=True) on float32: accumulated wide, rounded once (the kernels do the same)."""
    return a.astype(np.float64).sum(axis=1, keepdims=True).astype(F32)


def _take(a, idx):
    return np.take_along_axis(a, idx, axis=1)


def torch_cpu_argmin(vals):
    """Index torch.topk(vals, 1, largest=False) returns on CPU for a short row (dsnot_pruner.py:517).

    For n < 64 ATen calls std::nth_element(begin, begin, end) on (value, index) pairs (TopKImpl.h); with tied
    minima the winner is whatever libstdc++'s introselect leaves in front, so that algorithm is restated here
    (median-of-3 pivot to front, unguarded Hoare partition, insertion sort below 4 elements).  NaN sorts last.
    """
    q = [(float(v), i) for i, v in enumerate(vals)]

    def lt(x, y):
        return (y[0] != y[0] and x[0] == x[0]) or x[0] < y[0]

    first, last, nth = 0, len(q), 0
    depth = 2 * (len(q).bit_length() - 1)
    while last - first > 3:
        if depth == 0:      # heap-select fallback: unreachable for the group widths used here (m <= 32)
            best = first
            for i in range(first + 1, last):
                if lt(q[i], q[best]):
                    best = i
            q[first], q[best] = q[best], q[first]
            return q[first][1]
        depth -= 1
        mid = first + (last - first) // 2
        a, b, c = first + 1, mid, last - 1
        if lt(q[a], q[b]):
            pick = b if lt(q[b], q[c]) else (c if lt(q[a], q[c]) else a)
        else:
            pick = a if lt(q[a], q[c]) else (c if lt(q[b], q[c]) else b)
        q[first], q[pick] = q[pick], q[first]
        lo, hi = first + 1, last
        while True:
            while lt(q[lo], q[first]):
                lo += 1
            hi -= 1
            while lt(q[first], q[hi]):
                hi -= 1
            if not lo < hi:
                break
            q[lo], q[hi] = q[hi], q[lo]
            lo += 1
        if lo <= nth:
            first = lo
        else:
            last = lo
    for i in range(first + 1, last):       # insertion sort of the last <= 3 candidates
        j = i
        while j > first and lt(q[j], q[j - 1]):
            q[j], q[j - 1] = q[j - 1], q[j]
            j -= 1
    return q[nth][1]


def _group_argmin(block, rule):
    """Row-wise argmin of [R, m]; rule 'lowest' = lowest index among tied minima, 'torch_cpu' = torch_cpu_argmin."""
    am = np.argmin(block, axis=1)
    if rule == "lowest":
        return am
    mn = block[np.arange(block.shape[0]), am]
    tied = (block == mn[:, None]).sum(axis=1) > 1
    for r in np.nonzero(tied)[0]:
        am[r] = torch_cpu_argmin(block[r])
    return am


def dsnot_refine(W32, scaler_row, sum_metric_row, var, sparsity_num=0, prune_n=0, prune_m=0, pow_of_var=1.0,
                 max_cycle_time=100, update_threshold=0.1, without_same_sign=True, initial_method="wanda",
                 ref_fixup=True, argmin_rule="torch_cpu", force_cycles=None):
    """One linear's DSnoT mask.  Returns (keep_mask bool [R, C], cycles executed).

    sparsity_num = round(C * p) is computed by the caller (:562; python round, not int - SURVEY F5).
    ref_fixup=True reproduces the shipped reference including the block at :734-740 that writes the swap back
    (SURVEY F4); False gives the upstream DSnoT behaviour (that block excised).  The n:m branch has no such block.
    force_cycles: run exactly that many cycles instead of `while any(update_mask)` - what a row shard does once the
    executed-cycle count of the whole matrix is known (multi-rank tests).
    Tie-breaks (SURVEY F8): the unstable per-group sort at :423 is taken as lowest-column-first; the topk at :517
    meets structural ties (groups whose members were all set to +inf) and follows argmin_rule.
    """
    W = np.asarray(W32, dtype=F32)
    R, C = W.shape
    D = (W * sum_metric_row.astype(F32)[None, :]).astype(F32)                       # :368 DSnoT_metric
    wanda = (np.abs(W) * np.sqrt(scaler_row.astype(F32))[None, :]).astype(F32)
    initial = wanda.copy() if initial_method == "wanda" else np.abs(W).astype(F32)  # :370-376
    mask = np.zeros((R, C), dtype=bool)                                             # True = pruned (:405)
    thr = F32(update_threshold)
    rows = np.arange(R)[:, None]
    varp = None
    if pow_of_var:
        varp = var.astype(F32).reshape(1, -1) if pow_of_var == 1 else \
            np.power(var.astype(F32).reshape(1, -1), F32(pow_of_var)).astype(F32)
    max_cycle_time = int(max_cycle_time)

    def sign(x):
        return np.sign(x).astype(F32)

    if prune_n != 0:
        m, n = prune_m, prune_n
        G = initial.reshape(R, C // m, m)
        order = np.argsort(G, axis=2, kind="stable") + (np.arange(C // m) * m)[None, :, None]   # :420-424
        prune_idx = order[:, :, :n].reshape(R, -1)
        res_idx = order[:, :, n:].reshape(R, -1)
        np.put_along_axis(mask, prune_idx, True, axis=1)                            # :438
        reg = D.copy()
        np.put_along_axis(reg, res_idx, F32(0), axis=1)                             # :442
        err = _rowsum_f32(reg)                                                      # :444
        sign0 = sign(err)
        if varp is not None:
            with np.errstate(divide="ignore", invalid="ignore"):
                reg = (reg / varp).astype(F32)                                      # :447-451
        reg_order = np.argsort(reg, axis=1, kind="stable")                          # :453 (NaN last, like torch)
        ptr = np.zeros((R, 2), dtype=np.int64)
        ptr[:, 1] = C - 1
        step = np.array([1, -1], dtype=np.int64)
        np.put_along_axis(initial, prune_idx, F32(np.inf), axis=1)                  # :469
        upd = np.ones((R, 1), dtype=bool)
        cycles = 0
        while (upd.any() if force_cycles is None else cycles < force_cycles) and cycles < max_cycle_time:   # :476-479
            cycles += 1
            which = (err > 0).astype(np.int64)                                      # :483
            p = _take(ptr, which)
            rg = _take(reg_order, p)
            rm = _take(D, rg)
            start = rg - rg % m                                                     # :502
            blk = start + np.arange(m)[None, :]
            pr = start + _group_argmin(_take(initial, blk), argmin_rule)[:, None]    # :513-521 topk(1, smallest)
            pm = _take(D, pr)
            after = ((err + pm).astype(F32) - rm).astype(F32)                       # :525
            upd = upd & (sign0 == sign(after)) & (np.abs(err) > thr)                # :527
            np.put_along_axis(initial, pr, F32(np.inf), axis=1)                     # :529 (max + 1 == inf)
            np.put_along_axis(mask, pr, upd, axis=1)                                # :531
            np.put_along_axis(mask, rg, ~upd, axis=1)                               # :532
            err = (err + np.where(upd, pm, F32(0))).astype(F32)                     # :534
            err = (err - np.where(upd, rm, F32(0))).astype(F32)                     # :539
            np.put_along_axis(ptr, which, p + step[which], axis=1)                  # :545
        return ~mask, cycles

    k = int(sparsity_num)
    order0 = np.argsort(initial, axis=1, kind="stable")                             # :555
    prune_idx, res_idx = order0[:, :k], order0[:, k:]
    np.put_along_axis(mask, prune_idx, True, axis=1)                                # :581
    wm = wanda.copy()
    np.put_along_axis(wm, prune_idx, F32(np.inf), axis=1)                           # :586
    wres = np.argsort(wm, axis=1, kind="stable")[:, :C - k]                         # :587-591
    reorder = return_reorder_indice(_take(D, wres))                                 # :592
    prune_block = _take(wres, reorder)                                              # :595
    reg = D.copy()
    np.put_along_axis(reg, res_idx, F32(0), axis=1)                                 # :600
    err = _rowsum_f32(reg)                                                          # :601
    sign0 = sign(err)
    if varp is not None:
        with np.errstate(divide="ignore", invalid="ignore"):
            reg = (reg / varp).astype(F32)                                          # :604-608
    reg_order = np.argsort(reg, axis=1, kind="stable")                              # :610
    ptr_r = np.zeros((R, 2), dtype=np.int64)
    ptr_r[:, 1] = C - 1
    ptr_p = np.zeros((R, 2), dtype=np.int64)
    ptr_p[:, 1] = prune_block.shape[1] - 1
    step = np.array([1, -1], dtype=np.int64)
    upd = np.ones((R, 1), dtype=bool)
    cycles = 0
    while (upd.any() if force_cycles is None else cycles < force_cycles) and cycles < max_cycle_time:   # :650
        cycles += 1
        wr = (err > 0).astype(np.int64)                                             # :654
        p = _take(ptr_r, wr)
        rg = _take(reg_order, p)                                                    # raises IndexError like torch (F12)
        rm = _take(D, rg)
        np.put_along_axis(ptr_r, wr, p + step[wr], axis=1)                          # :673
        wp = (err < 0).astype(np.int64)                                             # :683
        q = _take(ptr_p, wp)
        if (q < 0).any() or (q >= prune_block.shape[1]).any():
            raise IndexError("prune pointer out of range (reference fails the same way, SURVEY F12)")
        pr = _take(prune_block, q)
        pm = _take(D, pr)
        np.put_along_axis(ptr_p, wp, q + step[wp], axis=1)                          # :703
        after = ((err + pm).astype(F32) - rm).astype(F32)                           # :713
        if without_same_sign:
            upd = upd & (np.abs(err) > thr)                                         # :717-720
        else:
            upd = upd & (np.abs(err) > thr) & (sign0 == sign(after))                # :722-729
        np.put_along_axis(mask, pr, upd, axis=1)                                    # :731
        np.put_along_axis(mask, rg, ~upd, axis=1)                                   # :732
        if ref_fixup:                                                               # :734-740
            sub_p, sub_r = _take(mask, pr), _take(mask, rg)
            np.put_along_axis(mask, pr, sub_p & ~upd, axis=1)
            np.put_along_axis(mask, rg, upd | (sub_r & ~upd), axis=1)
        err = (err + np.where(upd, pm, F32(0))).astype(F32)                         # :742
        err = (err - np.where(upd, rm, F32(0))).astype(F32)                         # :747
    return ~mask, cycles


# ---------------------------------------------------------------------------------------------
# SURVEY 8f-4: global sparsity allocation (layer_single_base_pruner.py:149-190, :241-420; the
# same get_mask / get_layerwise_mask at global_pruner.py:108-148)
# ---------------------------------------------------------------------------------------------
def kth_smallest(values, k):
    """torch.topk(values, k, largest=False)[0][-1]: the k-th smallest (1-based), NaN sorted last."""
    v = np.asarray(values, dtype=F32).ravel()
    if k < 1:
        raise IndexError("index -1 is out of bounds for dimension 0 with size 0")   # threshold[-1] of an empty topk
    return np.sort(v)[k - 1]                                                        # np.sort puts NaN last as well


def global_get_mask(scores, p, max_sparsity_per_layer):
    """LayerSparsity.get_mask (:149-176).  `scores`: dict name -> float32 array, MODIFIED IN PLACE like the
    reference (:160 writes finfo.max over the protected entries).  Returns (masks, threshold)."""
    fmax = np.finfo(F32).max
    for k, v in scores.items():
        num_to_set = int(v.size * (1 - max_sparsity_per_layer))                     # :153
        if num_to_set > 0:
            thr = np.sort(v.ravel())[v.size - num_to_set]                           # :157-158 j-th largest
            v[v >= thr] = fmax                                                      # :160
    all_scores = np.concatenate([v.ravel() for v in scores.values()])               # :165
    thr = kth_smallest(all_scores, int(p * all_scores.size))                        # :168-170
    return {k: (v > thr).astype(F32) for k, v in scores.items()}, thr               # :173-174


def layerwise_get_mask(scores, p):
    """LayerSparsity.get_layerwise_mask (:178-190): one threshold per tensor."""
    masks = {}
    for k, v in scores.items():
        thr = kth_smallest(v, int(p * v.size))
        masks[k] = (v > thr).astype(F32)
    return masks


def importance_scores_first_order(params, grads_per_batch, mode="obd"):
    """compute_importance_scores (:422-475) for one parameter: fp32 running sum of grad^2 (obd) or |grad|, divided by the
    number of batches, times w^2 - every step rounded to fp32 as the tensor expression does.  ("aobd" and "gradient"
    take the "obd" branch / the last branch of the reference's `in` tests, :466-473.)"""
    w = np.asarray(params, dtype=F32)
    acc = np.zeros_like(w)
    for g in grads_per_batch:
        g = np.asarray(g, dtype=F32)
        acc = (acc + (g * g if mode == "obd" else np.abs(g))).astype(F32)
    acc = (acc / F32(len(grads_per_batch))).astype(F32)
    if "obd" in mode:
        return ((w * w).astype(F32) * acc).astype(F32)
    return np.abs(acc)


def group_sparsity_allocation(total_to_keep, group_scores, group_num_params, max_sparsity_per_layer=0.8):
    """compute_the_sparsity_per_group (:304-378), with torch's dtypes restated: `scores` float32, parameter counts int64,
    the kept-parameter vector int64 until the first `+ parameters_to_add` turns it float32 (:318).  The shipped
    "remove the extra parameters" branch ADDS them (:358, `+=`); that is kept.  Returns the list of group sparsities.
    One thing numpy cannot restate: the ORDER of torch.sum over the float32 group scores (:313) is internal to ATen; a
    last-place difference in that sum can move a parameter or two between groups (tests/test_oracle_vs_reference.py
    measures it: exact on > 90 % of random cases, within 2.5 parameters per group otherwise).  The product's host loop
    (vlmc/compression/pruners/layer_sparsity.py) runs the same tensor ops as the reference and is exact on all of them."""
    scores = np.asarray(group_scores, dtype=F32).copy()
    num = np.asarray(group_num_params, dtype=np.int64)
    floor_keep = np.ceil(num.astype(F32) * F32(1 - max_sparsity_per_layer)).astype(np.int32)     # :309
    keep = floor_keep.astype(np.int64)
    while keep.sum() < total_to_keep:                                               # :311
        total_ratio = scores.sum(dtype=F32)
        rest = F32(total_to_keep - keep.sum())                                      # 0-dim tensor -> float32 operand
        with np.errstate(divide="ignore", invalid="ignore"):
            to_add = np.ceil((scores / total_ratio).astype(F32) * rest).astype(F32)  # :316
        keep = (keep.astype(F32) + to_add).astype(F32)                              # :318
        scores[keep >= num.astype(F32)] = 0                                         # :320
        keep = np.minimum(keep, num.astype(F32))                                    # :322
        if to_add.sum(dtype=F32) == 0:                                              # :326-342
            need = F32(total_to_keep) - keep.sum(dtype=F32)
            while need > 0:
                idx = np.nonzero(scores > 0)[0]
                if idx.size == 0:
                    raise RuntimeError("allocation cannot place the remaining parameters (the reference loops forever)")
                for i in idx:
                    can = min(need, F32(num[i]) - keep[i])
                    keep[i] += can
                    need -= can
                    if need == 0:
                        break
        if keep.sum(dtype=F32) > total_to_keep:                                     # :344-364
            need = keep.sum(dtype=F32) - F32(total_to_keep)
            while need > 0:
                progressed = False
                for i in np.argsort(-keep, kind="stable"):
                    extra = (F32(num[i]) * F32(1 - max_sparsity_per_layer)).astype(np.int32)
                    can = min(need, keep[i] - F32(extra))
                    keep[i] += can                                                  # shipped: += (not -=)
                    need -= can
                    progressed = progressed or can > 0
                    if need == 0:
                        break
                if not progressed:
                    raise RuntimeError("allocation cannot remove the extra parameters (the reference loops forever)")
    ratio = keep.astype(F32) / num.astype(F32)                                      # int64 / int64 is a float32 division too
    return [float(x) for x in np.clip(F32(1) - ratio, 0, 1).astype(F32)]           # :370-371
