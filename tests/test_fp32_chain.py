"""The fp32 chain of SparseGPT: the 3xTF32 GEMM (gemm3x.cu, vlmc_gemm_tf32x3) and the factor primitives built on it.

CPU: the TF32 rounding helper on hand-checked values, and the coverage of the GEMM case list.
GPU:
  - gemm_tf32x3 against float64 at ragged shapes, every kernel instance the public entry point selects (b_nk, chunked or
    not, 128- or 256-wide tiles), with a bar shown to catch a single TF32 pass and a dropped cross term; chunking, tri,
    beta = 0, row pitches, determinism, non-finite operands, rejections and power-of-two scale invariance;
  - every SparseGPT chain entry point called on row-strided views (NaN in padding that is only read, a sentinel in
    padding that is written): the same bits as the contiguous call;
  - chol_inv_upper / chol_upper at small and ragged C, gram_upper and diag_abs_mean against float64.
"""
import random

import numpy as np
import pytest
import torch

# Max error of gemm3x relative to the envelope |alpha| |A| |op(B)| + |beta| |C0|, element by element.  Measured on an
# NVIDIA B200 (1000 W power limit): at most 2.05e-6 over the shape sweep, 2.15e-6 for gram_upper, 1.77e-6 for the
# all-positive K = 16384 product with the default kc (1.75e-4 with kc = K).  On the sweep's `rounded_up` inputs a single
# TF32 pass is at least 3.6e-4 off and the split without one cross term at least 1.6e-4: 30x the bar or more.
BAR = 5e-6
REL = 1e-5                     # the fp32-grade bar of the factorisation against float64 (tests/test_gpu_parity.py)

MS = [1, 127, 128, 129, 1000]
NS = [4, 124, 128, 132, 256, 260, 1000]
KS = [4, 28, 32, 36, 128, 132, 1000, 4100]
KCS = [0, 32, 100, 256]
ALPHA_BETA = [(1.0, 0.0), (-1.0, 1.0), (0.37, -2.0), (2.0 / 5.0, 3.0 / 5.0)]   # last: the Hessian's 2/n, n_before/n


def tile_n(N, K, kc):
    """Output tile width the public entry point picks (gemm3x.cu): 256 only for a non-chunked K and N > 128."""
    kc = 128 if kc <= 0 else (kc + 31) // 32 * 32
    return 256 if K <= kc and N > 128 else 128


def _case_keys(case):
    M, N, K, kc, b_nk, ab = case
    tn = tile_n(N, K, kc)
    return {("M", M, b_nk, tn), ("N", N, b_nk, tn), ("K", K, b_nk, tn), ("kc", kc, b_nk, tn), ("ab", ab, b_nk, tn)}


def gemm_cases(total=100):
    """About `total` (M, N, K, kc, b_nk, alpha_beta index) cases in which every value of every list meets both b_nk and
    both tile widths wherever the entry point can select that tile width (N <= 128 and K > kc always give 128): a greedy
    cover that prefers cheap shapes, filled up with seeded random cases."""
    cands = [(M, N, K, kc, b, ab) for M in MS for N in NS for K in KS for kc in KCS for b in (0, 1)
             for ab in range(len(ALPHA_BETA))]
    need = set().union(*(_case_keys(c) for c in cands))
    chosen = []
    while need:
        best = max(cands, key=lambda c: (len(_case_keys(c) & need), -c[0] * c[1] * c[2], c))
        chosen.append(best)
        need -= _case_keys(best)
    rng = random.Random(20261022)
    rest = [c for c in cands if c not in chosen]
    chosen += rng.sample(rest, total - len(chosen))
    return chosen


GEMM_CASES = gemm_cases()


def tf32(x):
    """TF32 value of fp32 `x` as the split computes it (cvt.rna.tf32.f32: round to nearest, ties away from zero, on the
    fp32 bits), returned as fp32.  Finite values that round past the largest TF32 number become +-inf."""
    b = x.contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    r = ((b + 0x1000) & ~0x1FFF) & 0xFFFFFFFF
    r = torch.where(r >= 2 ** 31, r - 2 ** 32, r)
    return r.to(torch.int32).view(torch.float32).view(x.shape)


# ------------------------------------------------------------------------------------------- CPU
def test_tf32_rounding_hand_checked():
    def f(bits):
        return torch.tensor(bits, dtype=torch.int64).to(torch.int32).view(torch.float32)

    def as_bits(t):
        return [v & 0xFFFFFFFF for v in t.view(torch.int32).tolist()]

    src = [0x3F800000,   # 1.0: exact
           0x3F801000,   # 1 + 2^-11: the tie between 1 and 1 + 2^-10 goes away from zero (nearest-even would give 1)
           0x3F800FFF,   # just below the tie: down
           0x3F802000,   # 1 + 2^-10: exact
           0xBF801000,   # -(1 + 2^-11): away from zero, the sign is untouched
           0x3F803000,   # 1 + 3 * 2^-11: tie, up
           0x40400000,   # 3.0
           0x00000000, 0x80000000,   # +0, -0
           0x00000001,   # smallest subnormal: to +0
           0x00001000,   # subnormal tie: up to 0x2000
           0x7F7FFFFF,   # FLT_MAX: past the largest TF32 number, +inf
           0x7F800000, 0xFF800000]   # +-inf
    want = [0x3F800000, 0x3F802000, 0x3F800000, 0x3F802000, 0xBF802000, 0x3F804000, 0x40400000, 0x00000000, 0x80000000,
            0x00000000, 0x00002000, 0x7F800000, 0x7F800000, 0xFF800000]
    assert as_bits(tf32(f(src))) == want
    assert tf32(torch.tensor([1.0 + 2.0 ** -11], dtype=torch.float32)).item() == 1.0 + 2.0 ** -10
    # the split: hi + lo == x exactly for normal x, |lo| <= 2^-11 |hi|
    g = torch.Generator().manual_seed(3)
    x = torch.randn(4096, generator=g) * torch.exp2(torch.randint(-60, 60, (4096,), generator=g).float())
    hi = tf32(x)
    lo = x - hi
    assert torch.equal(hi + lo, x)
    assert bool((lo.abs() <= hi.abs() * 2.0 ** -11).all())
    assert bool(((hi.view(torch.int32) & 0x1FFF) == 0).all())


def test_gemm_case_list_covers_every_value():
    cases = GEMM_CASES
    assert 90 <= len(cases) <= 110 and len(set(cases)) == len(cases)
    have = set().union(*(_case_keys(c) for c in cases))
    for name, values in (("M", MS), ("N", NS), ("K", KS), ("kc", KCS), ("ab", range(len(ALPHA_BETA)))):
        for v in values:
            for b in (0, 1):
                assert (name, v, b, 128) in have, (name, v, b)
                # a 256-wide tile needs N > 128 and K <= kc; every value that allows it meets it with both b_nk
                feasible = any(tile_n(N, K, kc) == 256 for N in NS for K in KS for kc in KCS
                               if {"M": True, "N": N == v, "K": K == v, "kc": kc == v, "ab": True}[name])
                assert ((name, v, b, 256) in have) == feasible, (name, v, b)
    assert {tile_n(c[1], c[2], c[3]) for c in cases} == {128, 256}


# ------------------------------------------------------------------------------------------- GPU helpers
@pytest.fixture(scope="module")
def native(built_lib):
    from vlmc import native as n
    n.load()
    assert torch.cuda.is_available()
    return n


def mixed(shape, seed, lo=-6, hi=6):
    """fp32 with random signs and magnitudes spread over 2^lo .. 2^(hi+1), never near zero (no subnormal anywhere in
    the split or the products, also after scaling by 2^+-48)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    sign = torch.randint(0, 2, shape, generator=g, device="cuda").float() * 2 - 1
    mag = torch.exp2(torch.empty(shape, device="cuda").uniform_(lo, hi, generator=g))
    return sign * mag * (1 + torch.rand(shape, generator=g, device="cuda"))


def rounded_up(shape, seed, sign_dim):
    """Mixed magnitudes like `mixed`, one random sign per row (sign_dim = 0) or per column (1), and the low 13 mantissa
    bits of every element at or above the TF32 tie, so tf32() always rounds the magnitude up.  In a product with such a
    B (signs per row of [N, K], per column of [K, N]) every term of a dot product has the same sign and the same kind of
    rounding error: a single TF32 pass or a dropped cross term is off by about 2^-12 of the envelope on EVERY output,
    whatever K, instead of a sum of random errors that can cancel when the output has only a few elements."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    mag = torch.exp2(torch.empty(shape, device="cuda").uniform_(-6, 6, generator=g))
    mag = mag * (1 + torch.rand(shape, generator=g, device="cuda"))
    low = torch.randint(0x1000, 0x2000, shape, generator=g, device="cuda", dtype=torch.int32)
    mag = ((mag.view(torch.int32) & ~0x1FFF) | low).view(torch.float32)
    sshape = (shape[0], 1) if sign_dim == 0 else (1, shape[1])
    return mag * (torch.randint(0, 2, sshape, generator=g, device="cuda").float() * 2 - 1)


def ref64(A, B, C0, alpha, beta, b_nk):
    """(beta C0 + alpha A op(B), |alpha| |A| |op(B)| + |beta| |C0|) in float64, alpha and beta as the kernel sees them."""
    a, b = float(np.float32(alpha)), float(np.float32(beta))
    A64, B64 = A.double(), B.double()
    opB = B64.T if b_nk else B64
    ref = a * (A64 @ opB) + (b * C0.double() if b != 0 else 0)
    env = abs(a) * (A64.abs() @ opB.abs()) + (abs(b) * C0.double().abs() if b != 0 else 0)
    return ref, env


def env_err(got, ref, env):
    return float(((got.double() - ref).abs() / env).max())


def bits(t):
    return t.contiguous().view({4: torch.int32, 2: torch.int16, 1: torch.uint8}[t.element_size()])


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(bits(a), bits(b))


def embed(x, extra, fill):
    """x copied into a view of a larger buffer: row pitch = x's width + `extra`, one row of padding above and two below,
    16 bytes of padding before each row (so the view stays 16-byte aligned when the pitch is).  Every other element of
    the buffer holds `fill`.  Returns (buffer, view, mask of the padding)."""
    rows, cols = x.shape
    off = 16 // x.element_size()
    assert extra >= off
    buf = torch.full((rows + 3, cols + extra), fill, dtype=x.dtype, device=x.device)
    view = buf[1:1 + rows, off:off + cols]
    view.copy_(x)
    pad = torch.ones(buf.shape, dtype=torch.bool, device=x.device)
    pad[1:1 + rows, off:off + cols] = False
    return buf, view, pad


def pad_kept(buf, pad, fill):
    want = torch.full_like(buf, fill)
    return torch.equal(bits(buf)[pad], bits(want)[pad])


def gemm(native, A, B, C0, alpha, beta, b_nk, **kw):
    C = C0.clone()
    native.gemm_tf32x3(A, B, C, alpha=alpha, beta=beta, b_nk=b_nk, **kw)
    return C


def operands(M, N, K, b_nk, seed):
    return mixed((M, K), seed), mixed((N, K) if b_nk else (K, N), seed + 1), mixed((M, N), seed + 2)


# ------------------------------------------------------------------------------------------- gemm_tf32x3 vs float64
def _case_id(c):
    M, N, K, kc, b, ab = c
    return f"M{M}-N{N}-K{K}-kc{kc}-{'nk' if b else 'kn'}-ab{ab}-tn{tile_n(N, K, kc)}"


PHASE_CASES = [(2048, 2048, 300, 0, b, 1) for b in (0, 1)]   # 256 tiles > 148 SMs, 3 kc chunks per tile


@pytest.mark.gpu
@pytest.mark.parametrize("case", GEMM_CASES + PHASE_CASES, ids=_case_id)
def test_gemm_vs_fp64_and_the_bar_discriminates(native, case):
    """Max error relative to the envelope below BAR, on random signs (`mixed`) and on same-sign dot products whose
    TF32 rounding errors add up (`rounded_up`).  On the second inputs a single TF32 pass (tf32(A) tf32(B)) and the split
    without the lo(A) hi(B) term, emulated in float64, are both at least 10x above BAR."""
    M, N, K, kc, b_nk, ab = case
    alpha, beta = ALPHA_BETA[ab]
    seed = M * 7 + N * 13 + K * 17 + kc + b_nk
    A, B, C0 = operands(M, N, K, b_nk, seed)
    err_signed = env_err(gemm(native, A, B, C0, alpha, beta, b_nk, kc=kc), *ref64(A, B, C0, alpha, beta, b_nk))
    A = rounded_up((M, K), seed + 3, 0)
    B = rounded_up((N, K) if b_nk else (K, N), seed + 4, 0 if b_nk else 1)
    C = gemm(native, A, B, C0, alpha, beta, b_nk, kc=kc)
    ref, env = ref64(A, B, C0, alpha, beta, b_nk)
    err = env_err(C, ref, env)
    Ah, Bh = tf32(A), tf32(B)
    one, _ = ref64(Ah, Bh, C0, alpha, beta, b_nk)
    Bh64, Bl64 = Bh.double(), B.double() - Bh.double()
    a, b = float(np.float32(alpha)), float(np.float32(beta))
    opBh, opBl = (Bh64.T, Bl64.T) if b_nk else (Bh64, Bl64)
    drop = a * (Ah.double() @ opBh + Ah.double() @ opBl) + (b * C0.double() if b != 0 else 0)
    e_one, e_drop = env_err(one, ref, env), env_err(drop, ref, env)
    print(f"\ngemm3x {_case_id(case)}: err {err_signed:.3e} / {err:.3e}  bar {BAR:.1e}  "
          f"single-pass {e_one:.3e}  dropped-cross {e_drop:.3e}")
    assert err_signed < BAR and err < BAR
    assert e_one >= 10 * BAR and e_drop >= 10 * BAR


@pytest.mark.gpu
def test_gemm_long_k_chunking_bounds_the_drift(native):
    """K = 16384, all-positive operands (the tensor core's round-toward-zero accumulation drifts the most): the default kc
    meets the bar, one in-TMEM accumulation over all of K (kc = K) is measurably worse."""
    M, N, K = 256, 256, 16384
    g = torch.Generator(device="cuda").manual_seed(11)
    A = 1 + torch.rand(M, K, generator=g, device="cuda")
    B = 1 + torch.rand(K, N, generator=g, device="cuda")
    C0 = torch.zeros(M, N, device="cuda")
    ref, env = ref64(A, B, C0, 1.0, 0.0, False)
    errs = {kc: env_err(gemm(native, A, B, C0, 1.0, 0.0, False, kc=kc), ref, env) for kc in (0, 1024, K)}
    print("gemm3x K=16384 all-positive, err vs kc:", {k: f"{v:.3e}" for k, v in errs.items()}, f"bar {BAR:.1e}")
    assert errs[0] < BAR
    assert errs[K] > 4 * errs[0]


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,K,b_nk", [(1000, 600, 128, 0), (1000, 600, 128, 1), (300, 1000, 36, 1),
                                        (600, 1000, 300, 0), (600, 1000, 300, 1), (1000, 260, 1000, 0)])
def test_gemm_tri_computes_the_lower_tiles_only(native, M, N, K, b_nk):
    """tri = 1: every entry i >= j (indeed every entry of a computed tile) has the bits of the tri = 0 call; the tiles the
    kernel skips (column start past the tile's last row) keep C0's bits."""
    A, B, C0 = operands(M, N, K, b_nk, 5 + M + N + K)
    full = gemm(native, A, B, C0, -1.0, 1.0, b_nk)
    tri = gemm(native, A, B, C0, -1.0, 1.0, b_nk, tri=True)
    tn = tile_n(N, K, 0)
    i = torch.arange(M, device="cuda")[:, None]
    j = torch.arange(N, device="cuda")[None, :]
    skipped = (j // tn) * tn > (i // 128) * 128 + 127
    assert bool(skipped.any()) and not bool(skipped[i >= j].any())
    assert torch.equal(bits(tri)[~skipped], bits(full)[~skipped])
    assert torch.equal(bits(tri)[skipped], bits(C0)[skipped])


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,K,b_nk", [(200, 260, 36, 0), (200, 260, 36, 1), (129, 132, 1000, 0), (129, 100, 1000, 1)])
def test_gemm_beta_zero_does_not_read_c(native, M, N, K, b_nk):
    A, B, _ = operands(M, N, K, b_nk, 21)
    nan = torch.full((M, N), float("nan"), device="cuda")
    zero = torch.zeros(M, N, device="cuda")
    got = gemm(native, A, B, nan, 0.37, 0.0, b_nk)
    assert bool(torch.isfinite(got).all())
    assert same_bits(got, gemm(native, A, B, zero, 0.37, 0.0, b_nk))
    ref, env = ref64(A, B, zero, 0.37, 0.0, b_nk)
    assert env_err(got, ref, env) < BAR
    assert bool(gemm(native, A, B, nan, 0.37, 1.0, b_nk).isnan().all())


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,K,b_nk,kc", [(200, 260, 36, 0, 0), (200, 260, 36, 1, 0), (129, 132, 1000, 0, 0),
                                           (129, 132, 1000, 1, 256), (1000, 1000, 132, 0, 0), (127, 4, 4100, 1, 0)])
def test_gemm_row_pitches(native, M, N, K, b_nk, kc):
    """A, B, C as views inside larger buffers (pitch != width, 16-byte aligned offset).  NaN in A's and B's padding (a
    tensor map built on the pitch instead of the width would read it whenever K or N is not a multiple of 32), a
    sentinel in C's: the bits of the contiguous call, the sentinel untouched."""
    A, B, C0 = operands(M, N, K, b_nk, 31 + K)
    want = gemm(native, A, B, C0, -1.0, 1.0, b_nk, kc=kc)
    Abuf, Av, Apad = embed(A, 12, float("nan"))
    Bbuf, Bv, Bpad = embed(B, 20, float("nan"))
    Cbuf, Cv, Cpad = embed(C0, 8, -1234.5)
    native.gemm_tf32x3(Av, Bv, Cv, alpha=-1.0, beta=1.0, b_nk=b_nk, kc=kc)
    assert Av.stride(0) != K and Cv.stride(0) != N and Cv.data_ptr() % 16 == 0
    assert same_bits(Cv, want)
    assert pad_kept(Cbuf, Cpad, -1234.5)
    assert pad_kept(Abuf, Apad, float("nan")) and pad_kept(Bbuf, Bpad, float("nan"))


@pytest.mark.gpu
def test_gemm_deterministic_across_calls_and_streams(native):
    for (M, N, K, b_nk) in [(2048, 2048, 300, 0), (1000, 1000, 128, 1), (129, 260, 4100, 1)]:
        A, B, C0 = operands(M, N, K, b_nk, 41)
        c1 = gemm(native, A, B, C0, -1.0, 1.0, b_nk)
        c2 = gemm(native, A, B, C0, -1.0, 1.0, b_nk)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            c3 = gemm(native, A, B, C0, -1.0, 1.0, b_nk)
        s.synchronize()
        assert same_bits(c1, c2) and same_bits(c1, c3)


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,K,b_nk", [(200, 260, 36, 0), (129, 132, 1000, 1)])
def test_gemm_non_finite_operands(native, M, N, K, b_nk):
    """An inf or NaN of A or B makes every output whose dot product meets it NaN (inf splits into hi = inf, lo = NaN),
    whatever it meets; a finite value that rounds past the largest TF32 number (FLT_MAX) behaves like inf.  Every other
    output stays finite and within the bar of the float64 result."""
    A, B, C0 = operands(M, N, K, b_nk, 51)
    A[3, 5] = float("inf")
    A[7, K - 1] = float("-inf")
    A[11, 0] = float("nan")
    A[13, 2] = 3.4028234e38                       # FLT_MAX
    A[17, 3] = 0.0
    if b_nk:
        B[9, 1] = float("inf")
        B[10, 2] = 0.0
    else:
        B[1, 9] = float("inf")
        B[2, 10] = 0.0
    got = gemm(native, A, B, C0, -1.0, 1.0, b_nk)
    bad = torch.zeros(M, N, dtype=torch.bool, device="cuda")
    bad[[3, 7, 11, 13], :] = True
    bad[:, 9] = True
    assert bool(got[bad].isnan().all())
    assert bool(torch.isfinite(got[~bad]).all())
    A0, B0 = A.clone(), B.clone()
    A0[[3, 7, 11, 13], :] = 0
    if b_nk:
        B0[9, :] = 0
    else:
        B0[:, 9] = 0
    ref, env = ref64(A0, B0, C0, -1.0, 1.0, b_nk)
    assert float(((got.double() - ref).abs() / env)[~bad].max()) < BAR


@pytest.mark.gpu
def test_gemm_rejections_leave_c_unchanged(native):
    """Each of these raises before any launch, and C keeps its bits."""
    M, N, K = 128, 128, 128
    A, B, C0 = operands(M, N, K, 0, 61)

    def flat(n, off):
        return torch.zeros(n + 8, device="cuda")[off:off + n]

    def rejected(A_, B_, C_, status, **kw):
        before = C_.clone()
        with pytest.raises(native.VlmcError) as e:
            native.gemm_tf32x3(A_, B_, C_, **kw)
        torch.cuda.synchronize()
        assert e.value.status == status and same_bits(C_, before)

    UNSUP, BAD = -2, -1
    Ab = torch.zeros(M, 8, device="cuda")
    rejected(Ab[:, :6], torch.zeros(6, N, device="cuda"), C0.clone(), UNSUP)                       # K % 4
    Bb, Cb = torch.zeros(K, 8, device="cuda"), torch.zeros(M, 8, device="cuda")
    rejected(A, Bb[:, :6], Cb[:, :6], UNSUP)                                                      # N % 4
    rejected(torch.zeros(M, K + 2, device="cuda")[:, :K], B, C0.clone(), UNSUP)                  # lda % 4
    rejected(A, torch.zeros(K, N + 2, device="cuda")[:, :N], C0.clone(), UNSUP)                  # ldb % 4
    rejected(A, B, torch.zeros(M, N + 2, device="cuda")[:, :N], UNSUP)                           # ldc % 4
    rejected(flat(M * K, 1).view(M, K), B, C0.clone(), UNSUP)                                      # A not 16-byte aligned
    rejected(A, flat(K * N, 2).view(K, N), C0.clone(), UNSUP)                                      # B
    rejected(A, B, flat(M * N, 3).view(M, N), UNSUP)                                               # C
    rejected(A, B, torch.zeros(M * N, device="cuda").as_strided((M, N), (N - 4, 1)), BAD)          # ldc < N
    # argument errors of the binding itself
    for bad_args in [(A.double(), B, None), (A, B[:64], None), (A, B, torch.zeros(M, N + 4, device="cuda")),
                     (A.t(), B, None), (A[0], B, None)]:
        with pytest.raises(ValueError):
            native.gemm_tf32x3(*bad_args)


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,K,b_nk", [(200, 260, 36, 0), (129, 132, 1000, 1), (1000, 1000, 132, 1)])
def test_gemm_power_of_two_scale_invariance(native, M, N, K, b_nk):
    """gemm(2^s A, B) == 2^s gemm(A, B) bit for bit with beta = 0: the split and the accumulation are exact under
    power-of-two scaling while nothing is subnormal."""
    A, B, C0 = operands(M, N, K, b_nk, 71)
    base = gemm(native, A, B, C0, 1.0, 0.0, b_nk)
    for s in (48, -48):
        got = gemm(native, A * 2.0 ** s, B, C0, 1.0, 0.0, b_nk)
        assert same_bits(got, base * 2.0 ** s), s


# ------------------------------------------------------------------------------------------- the chain at row pitches
PITCHED = [(260, 4), (260, 132), (1408, 4), (1408, 132)]
SENT = -777.25
DT = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}


def acts(T, C, seed, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    gain = torch.exp(torch.rand(C, generator=g) * 2.77 - 1.386)
    off = torch.randn(C, generator=g) * 0.3
    return (torch.randn(T, C, generator=g) * gain + off).to(dtype).cuda()


def hessian(C, seed, damp=0.01):
    """2/T X^T X (T = 4C) in float64, rounded to fp32, plus the pruner's percdamp * mean(diag) on the diagonal."""
    x = acts(4 * C, C, seed).double()
    H = x.T @ x * (2.0 / x.shape[0])
    H += damp * H.diagonal().mean() * torch.eye(C, dtype=H.dtype, device=H.device)
    return H.float()


def x_pitch_extra(C, p):
    return (C + p + 4 + 7) // 8 * 8 - C          # fp16 / bf16 rows need a pitch that is a multiple of 8 elements


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f16", "bf16", "f32"])
@pytest.mark.parametrize("C,p", PITCHED)
def test_hessian_accum_at_row_pitch(native, C, p, tag):
    """Both paths (fp16 / bf16 SYRK, fp32 3xTF32 with A given [K, M]), two calls so that the second reads H.  The SYRK
    takes C % 8 == 0: it runs at C = 264 where the fp32 path runs at 260."""
    if tag != "f32" and C % 8:
        C += 4
    xs = [acts(300, C, 3 + i, DT[tag]) for i in range(2)]
    H = torch.zeros(C, C, device="cuda")
    for i, x in enumerate(xs):
        native.hessian_accum(x, H, i, 1)
    Hbuf, Hv, Hpad = embed(torch.zeros(C, C, device="cuda"), p, SENT)
    for i, x in enumerate(xs):
        xbuf, xv, xpad = embed(x, x_pitch_extra(C, p), float("nan"))
        native.hessian_accum(xv, Hv, i, 1)
        assert pad_kept(xbuf, xpad, float("nan"))
    assert same_bits(Hv, H)
    assert pad_kept(Hbuf, Hpad, SENT)


@pytest.mark.gpu
@pytest.mark.parametrize("C,p", PITCHED)
def test_prepare_and_damp_at_row_pitch(native, C, p):
    H = hessian(C, 5)
    H[7, :] = 0
    H[:, 7] = 0
    H[C - 1, C - 1] = 0                          # two dead channels
    want = H.clone()
    damp, dead = native.hessian_prepare(want, 0.01)
    native.hessian_add_damp(want, damp)
    Hbuf, Hv, Hpad = embed(H, p, SENT)
    damp2, dead2 = native.hessian_prepare(Hv, 0.01)
    native.hessian_add_damp(Hv, damp2)
    assert int(dead.sum()) == 2
    assert same_bits(Hv, want) and same_bits(damp2, damp) and torch.equal(dead2, dead)
    assert pad_kept(Hbuf, Hpad, SENT)


@pytest.mark.gpu
@pytest.mark.parametrize("C,p", PITCHED)
def test_factorisations_at_row_pitch(native, C, p):
    """chol_inv_upper and chol_upper with H at pitch C + p and U at C + 136 - p (the pitches differ, so an ldh / ldu
    swap shows too; U's pitch is the lda / ldb / ldc of the triangular-inverse GEMMs), then gram_upper: bits and status
    words of the contiguous calls."""
    H = hessian(C, 7)
    for fn in (native.chol_inv_upper, native.chol_upper):
        U, st = fn(H)
        Hbuf, Hv, Hpad = embed(H, p, float("nan"))
        Ubuf, Uv, Upad = embed(torch.zeros(C, C, device="cuda"), 136 - p, SENT)
        _, st2 = fn(Hv, U=Uv)
        assert int(st.item()) == 0 and int(st2.item()) == int(st.item())
        assert same_bits(Uv, U), fn.__name__
        assert pad_kept(Ubuf, Upad, SENT) and pad_kept(Hbuf, Hpad, float("nan"))
    G = native.gram_upper(U)
    Ubuf, Uv, _ = embed(U, p, float("nan"))
    Gbuf, Gv, Gpad = embed(torch.zeros(C, C, device="cuda"), 136 - p, SENT)
    native.gram_upper(Uv, out=Gv)
    assert same_bits(Gv, G) and pad_kept(Gbuf, Gpad, SENT)


@pytest.mark.gpu
@pytest.mark.parametrize("C,p", PITCHED)
def test_matrix_helpers_at_row_pitch(native, C, p):
    """diag_abs_mean, matrix_nonfinite_count (NaN only in the padding counts nothing) and matrix_replace_inf (the
    padding holds the infinity being replaced, and keeps it)."""
    A = mixed((C, C), 81)
    A[3, 4] = float("inf")
    A[5, 5] = float("-inf")
    A[C - 1, C - 2] = float("inf")
    A[9, 1] = float("nan")
    Abuf, Av, Apad = embed(A, p, float("nan"))
    assert native.matrix_nonfinite_count(Av) == native.matrix_nonfinite_count(A) == (2, 1, 1)
    Af = A.clone()
    Af[5, 5] = -2.0
    Af[9, 1] = 0.5
    _, Afv, _ = embed(Af, p, float("nan"))
    assert same_bits(native.diag_abs_mean(Afv, 0.01), native.diag_abs_mean(Af, 0.01))
    for negative, inf in ((0, float("inf")), (1, float("-inf"))):
        want = A.clone()
        native.matrix_replace_inf(want, 123.0, negative)
        buf, v, pad = embed(A, p, inf)
        native.matrix_replace_inf(v, 123.0, negative)
        assert same_bits(v, want) and pad_kept(buf, pad, inf)
    assert pad_kept(Abuf, Apad, float("nan"))


@pytest.mark.gpu
@pytest.mark.parametrize("n,m", [(0, 0), (2, 4)])
@pytest.mark.parametrize("tag", ["f16", "bf16"])
@pytest.mark.parametrize("C,p", PITCHED)
def test_obs_sweep_at_row_pitch(native, C, p, tag, n, m):
    """U at a pitch (NaN padding), W a column slice of a wider fp16 / bf16 buffer and the keep mask a slice of a wider
    byte buffer (sentinels): the same weights, mask and importance score as the contiguous call."""
    R = 96
    H = hessian(C, 9)
    H[11, :] = 0
    H[:, 11] = 0
    damp, dead = native.hessian_prepare(H, 0.01)
    U, st = native.chol_inv_upper(H)
    assert int(st.item()) == 0
    g = torch.Generator().manual_seed(C + p)
    W0 = (torch.randn(R, C, generator=g) * 0.05).to(DT[tag]).cuda()
    sp = 0.5 if n == 0 else 0.0
    W = W0.clone()
    keep, score = native.obs_sweep(W, U, sp, n, m, dead=dead, want_mask=True)
    Ubuf, Uv, Upad = embed(U, p, float("nan"))
    Wbuf, Wv, Wpad = embed(W0, x_pitch_extra(C, p), SENT)
    Kbuf, Kv, Kpad = embed(torch.zeros(R, C, dtype=torch.uint8, device="cuda"), p + 16, 0xA5)
    _, score2 = native.obs_sweep(Wv, Uv, sp, n, m, dead=dead, keep=Kv)
    assert same_bits(Wv, W) and torch.equal(Kv, keep.to(torch.uint8)) and same_bits(score2, score)
    assert pad_kept(Wbuf, Wpad, SENT) and pad_kept(Kbuf, Kpad, 0xA5) and pad_kept(Ubuf, Upad, float("nan"))


# ------------------------------------------------------------------------------------------- small and ragged C vs float64
@pytest.mark.gpu
@pytest.mark.parametrize("C", [4, 12, 100, 124, 132, 260])
def test_factorisations_small_c_vs_fp64(native, C):
    """Blocks smaller than 128 are padded with the identity: here they are the whole matrix (C < 128) or its ragged last
    block.  Both factors within REL of float64, exactly upper triangular, H untouched."""
    H = hessian(C, 13 + C)
    H0 = H.clone()
    cases = [(native.chol_inv_upper, torch.linalg.cholesky(torch.linalg.inv(H.double()), upper=True)),
             (native.chol_upper, torch.linalg.cholesky(H.double(), upper=True))]
    for fn, want in cases:
        U, st = fn(H)
        assert int(st.item()) == 0 and same_bits(H, H0)
        assert float(U.tril(-1).abs().max()) == 0.0
        err = float((U.double() - want).abs().max() / want.abs().max())
        print(f"{fn.__name__} C={C}: max-norm error vs fp64 {err:.2e}")
        assert err < REL, fn.__name__


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["dense", "upper"])
@pytest.mark.parametrize("C", [4, 64, 128, 132, 1000, 4100])
def test_gram_upper_vs_fp64(native, C, kind):
    """Hinv = U^T U against float64, relative to |U|^T |U| (the gemm bar).  C <= 128 takes the non-chunked [K, M]
    instance that nothing else reaches; the kernel does not assume U triangular."""
    U = mixed((C, C), 91 + C)
    if kind == "upper":
        U = torch.triu(U)
    got = native.gram_upper(U)
    U64 = U.double()
    err = env_err(got, U64.T @ U64, U64.abs().T @ U64.abs())
    print(f"gram_upper C={C} {kind}: err {err:.3e} (bar {BAR:.1e})")
    assert err < BAR


@pytest.mark.gpu
@pytest.mark.parametrize("C", [4, 260, 1408, 4100])
def test_diag_abs_mean_vs_torch(native, C):
    """scale * mean(|diag|): within 1 ulp of torch's fp32 expression and of the float64 value (the kernel sums in double)."""
    A = mixed((C, C), 101 + C)
    scale = 0.01
    got = np.float32(native.diag_abs_mean(A, scale).item())
    want32 = np.float32((torch.tensor(scale, dtype=torch.float32, device="cuda") * A.diagonal().abs().mean()).item())
    want64 = scale * float(A.diagonal().double().abs().mean())
    assert abs(float(got) - float(want32)) <= float(np.spacing(want32))
    assert abs(float(got) - want64) <= float(np.spacing(np.float32(want64)))
