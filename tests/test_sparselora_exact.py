"""The SparseLoRA tile kernels against an exact reference: K15 (effective weight), K14 (merge, single and batched) and K16
(LoRA gradients).  Every LoRA path of the project is built on these three; K23 and K28-K30 are tested bit-equal to them.

The reference below is torch float64 and runs on any device:
  - fma32: fmaf correctly rounded (exact float64 product, TwoSum, round to odd, one rounding to fp32);
  - K15 and K14 bit for bit, the sign of zero included: the rank-r product with one fma per k, k ascending from +0 (what
    lt_dot computes), then the documented roundings;
  - K16 per element against float64 sums, within (n + 2) 2^-24 sum |terms|, n the depth of the kernel's fixed
    summation order.
The masked-position rule (include/vlmc.h): masked entries of the effective weight are +0 and a masked G contributes
nothing, whatever W, the LoRA product or G hold.  The reference's `(W + d) * mask` gives -0 or NaN there instead.

CPU: fma32 against Fraction arithmetic, the numpy oracle against this reference, and the K16 bar against float64
emulations of real regressions.
GPU: ragged R (R % 4 != 0) and C (partial column tiles), every rank 1-16, row pitches, batched merges whose CTA spans
cross items, Vicuna-7B shapes, non-finite inputs; K16 on both sides of every chunking and template switch.
"""
import math
from fractions import Fraction

import numpy as np
import pytest
import torch

from oracle import oracle

DT = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}
VEC = {"f32": 4, "f16": 8, "bf16": 8}                  # elements per 16-byte vector (Elem<T>::kVec)
# one vector; one column tile (1024 columns, 512 for fp32) plus one vector; 1.375 tiles; 10.75 tiles (21.5 for fp32)
COLS = {"f32": [4, 516, 1408, 11008], "f16": [8, 1032, 1408, 11008], "bf16": [8, 1032, 1408, 11008]}
ROWS = [1, 2, 3, 5, 4097]                               # K14 / K15 take rows in blocks of 4
VICUNA = [(4096, 4096), (11008, 4096), (4096, 11008)]
GRAD_ROWS = [1, 15, 16, 17, 4735, 4736, 4737, 11008]   # K16's chunking changes at 16 rows and at 296 chunks (R > 4736)
GRAD_RANKS = [1, 3, 4, 5, 8, 9, 15, 16]                 # K16's template switches at 4, 8 and 16
U = 2.0 ** -24                                          # unit roundoff of fp32
MAX_GRID = 148 * 5                                      # K14's largest grid: every SM, at most 5 CTAs (__launch_bounds__)


# ------------------------------------------------------------------------------------------- the reference
def fma32(b, a, c):
    """fmaf(b, a, c), correctly rounded, on float64 tensors that hold fp32 values; returns float64.  b * a is exact in
    float64; TwoSum gives the sum and its exact error; an inexact sum is moved to its odd neighbour (round to odd), so the
    one rounding to fp32 that follows is correct.  float32(b * a + c) in float64 is not: that sum can land exactly on an
    fp32 midpoint."""
    p = b * a
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    even = (s.view(torch.int64) & 1) == 0
    toward = torch.where(err > 0, math.inf, -math.inf).to(s.dtype)
    s = torch.where(torch.isfinite(s) & (err != 0) & even, torch.nextafter(s, toward), s)
    return s.to(torch.float32).to(torch.float64)


def add32(x, y):
    """x + y in fp32 (one rounding)."""
    return fma32(x, torch.ones((), dtype=torch.float64, device=x.device), y)


def mul32(x, s):
    """x * s in fp32: the product of two fp32 values is exact in float64, so one rounding."""
    return (x * s).to(torch.float32).to(torch.float64)


def round_dt(x, dt):
    """fp32 values (in float64) rounded to `dt` (round to nearest even), back in float64."""
    return x.to(torch.float32).to(dt).to(torch.float64)


def f32(s):
    """The fp32 scaling the kernels receive."""
    return float(np.float32(s))


def lora_product(A, B):
    """B @ A in fp32 as lt_dot computes it: per element one fma per k, k ascending, from +0.  Returns float64."""
    A64, B64 = A.double(), B.double()
    acc = torch.zeros(B.shape[0], A.shape[1], dtype=torch.float64, device=A.device)
    for k in range(A.shape[0]):
        acc = fma32(B64[:, k:k + 1], A64[k:k + 1], acc)
    return acc


def effective_weight(W, A, B, s, M, sparse):
    """K15's weight in W's dtype: d = round(round(BA) * s); sparse: M ? round(W + d) : +0; dense: round((M ? W : +0) + d)."""
    dt, zero = W.dtype, torch.zeros((), dtype=torch.float64, device=W.device)
    d = round_dt(lora_product(A, B), dt)
    d = round_dt(mul32(d, f32(s)), dt)
    W64 = W.double()
    if sparse:
        out = torch.where(M, round_dt(add32(W64, d), dt), zero)
    else:
        out = round_dt(add32(torch.where(M, W64, zero), d), dt)
    return out.to(dt)


def merge(W, A, B, s, M, remask):
    """K14 in W's dtype: M ? round(W +32 (BA *32 s)) : (remask ? +0 : W)."""
    dt, zero = W.dtype, torch.zeros((), dtype=torch.float64, device=W.device)
    W64 = W.double()
    merged = round_dt(add32(W64, mul32(lora_product(A, B), f32(s))), dt)
    return torch.where(M, merged, zero if remask else W64).to(dt)


def lora_grads(G, A, B, s, M, sparse):
    """K16 in float64 with E as the kernel defines it, keep ? round(G *32 s) : 0 (keep = M, or everywhere when not
    sparse).  Returns (dA, dB, SA, SB); SA and SB are the sums of |term| of each output element."""
    E = round_dt(mul32(G.double(), f32(s)), G.dtype)
    if sparse:
        E = torch.where(M, E, torch.zeros((), dtype=torch.float64, device=G.device))
    A64, B64 = A.double(), B.double()
    return B64.T @ E, E @ A64.T, B64.abs().T @ E.abs(), E.abs() @ A64.abs().T


def grad_depths(R, C, V):
    """Summation depth of each K16 output: dB adds ceil(C / 32V) * V fmas per lane, then 5 shuffle adds; dA adds
    rows_per_chunk fmas per chunk, then nchunks partials.  The chunking mirrors grad_chunks() in csrc/lora_forward.cu
    (at most kNumSMs * 2 = 296 chunks, at least 16 rows each)."""
    chunks = max(1, min(296, -(-R // 16)))
    rows_per_chunk = -(-R // chunks)
    nchunks = -(-R // rows_per_chunk)
    return rows_per_chunk + nchunks, -(-C // (32 * V)) * V + 5


# Measured on an NVIDIA B200 (1000 W power limit): K16's largest error is 0.25 of the bar on both sides, dA and dB.  On
# coherent_case() the float64 emulations of three faults land far over it: E not rounded to the dtype 202x (dA) and 298x
# (dB), the last row of the last chunk dropped 341x, the mask not applied 2.5e5x.
def bar_ratio(got, ref, S, n):
    """Largest |got - ref| / ((n + 2) 2^-24 S) over the elements; an element with S = 0 must be exact."""
    err = (got.double() - ref).abs()
    bar = (n + 2) * U * S
    ratio = torch.where(bar > 0, err / bar, torch.where(err > 0, math.inf, 0.0).to(err.dtype))
    return float(ratio.max())


# ------------------------------------------------------------------------------------------- helpers
def canon_bits(t):
    """The bits of t as integers, every NaN as one pattern: the kernels store canonical NaNs, payloads are not part of
    their results.  The sign of zero counts."""
    t = t.contiguous()
    t = torch.where(torch.isnan(t), torch.full_like(t, math.nan), t)
    return t.view({torch.float32: torch.int32, torch.float16: torch.int16, torch.bfloat16: torch.int16}[t.dtype])


def assert_same_bits(got, want, what):
    g, w = canon_bits(got), canon_bits(want)
    if not torch.equal(g, w):
        bad = (g != w).nonzero()
        i = tuple(bad[0].tolist())
        raise AssertionError(f"{what}: {bad.shape[0]} elements differ, first at {i}: got {got[i].item()!r} "
                             f"({g[i].item() & 0xFFFFFFFF:#x}), want {want[i].item()!r} ({w[i].item() & 0xFFFFFFFF:#x})")


def raw_bits(t):
    return t.contiguous().view({4: torch.int32, 2: torch.int16, 1: torch.uint8}[t.element_size()])


def lora_case(R, C, r, dt, seed, device="cuda"):
    g = torch.Generator(device=device).manual_seed(seed)
    W = (torch.randn(R, C, generator=g, device=device) * 0.05).to(dt)
    A = torch.randn(r, C, generator=g, device=device) * 0.1
    B = torch.randn(R, r, generator=g, device=device) * 0.1
    M = torch.rand(R, C, generator=g, device=device) < 0.5
    return W, A, B, M


# ------------------------------------------------------------------------------------------- CPU: fma32
def f32_of(q):
    """The fp32 nearest to the Fraction q (ties to even), as a float; inf past the largest finite fp32."""
    if q == 0:
        return 0.0
    sign, q = (-1.0 if q < 0 else 1.0), abs(q)
    e = q.numerator.bit_length() - q.denominator.bit_length()
    if Fraction(2) ** e > q:
        e -= 1
    ulp = Fraction(2) ** (max(e, -126) - 23)
    n = q // ulp
    rem = q - n * ulp
    if rem > ulp / 2 or (rem == ulp / 2 and n % 2 == 1):
        n += 1
    v = n * ulp
    return sign * (math.inf if v >= 2 ** 128 else float(v))


def exact_fma(b, a, c):
    return np.array([f32_of(Fraction(float(x)) * Fraction(float(y)) + Fraction(float(z))) for x, y, z in zip(b, a, c)])


def fma32_np(b, a, c):
    t = [torch.from_numpy(np.asarray(v, np.float32)).double() for v in (b, a, c)]
    return fma32(*t).numpy()


def old_fma(b, a, c):
    """The former oracle emulation: float32(float64(b * a) + c), two roundings."""
    return (b.astype(np.float64) * a.astype(np.float64) + c.astype(np.float64)).astype(np.float32).astype(np.float64)


def near_midpoint_triples(n, seed):
    """(b, a, c) fp32 with b * a = U/2 (1 + eps), 0 <= |eps| < 2^-31, and c = +-K U, K a 24-bit integer: b * a + c lies
    within 2^-32 U of a midpoint of c's fp32 grid, closer than half a float64 ulp of the sum, so a float64 sum rounds to
    the midpoint itself.  The mantissas are 24-bit integers ma * mb = 2^47 + r with |r| < 2^16, found by rejection."""
    rng = np.random.default_rng(seed)
    ma, mb = np.zeros(0, np.int64), np.zeros(0, np.int64)
    while ma.size < n:
        x = rng.integers(2 ** 23 + 1, 2 ** 24, size=1 << 20, dtype=np.int64)
        y = (2 ** 47 + x // 2) // x
        ok = np.abs(x * y - 2 ** 47) < 2 ** 16
        ma, mb = np.concatenate([ma, x[ok]]), np.concatenate([mb, y[ok]])
    ma, mb = ma[:n], mb[:n]
    ea, eb = rng.integers(-50, 1, n), rng.integers(-50, 1, n)
    K = rng.integers(2 ** 23, 2 ** 24, n)
    sgn = lambda: rng.choice([-1.0, 1.0], n)                               # noqa: E731
    a = np.ldexp(ma.astype(np.float64), ea) * sgn()
    b = np.ldexp(mb.astype(np.float64), eb) * sgn()
    c = np.ldexp(K.astype(np.float64), ea + eb + 48) * sgn()
    return b.astype(np.float32), a.astype(np.float32), c.astype(np.float32)


def random_triples(n, seed):
    """Ordinary fp32 triples over a wide exponent range, a quarter of them with c = -fl(b * a) (the exact rounding error
    of the product)."""
    rng = np.random.default_rng(seed)
    f = lambda: (rng.standard_normal(n) * np.exp2(rng.integers(-30, 30, n))).astype(np.float32)   # noqa: E731
    b, a, c = f(), f(), f()
    q = n // 4
    c[:q] = -(b[:q].astype(np.float64) * a[:q]).astype(np.float32)
    return b, a, c


def test_fma32_midpoint_example():
    b = np.array([1 - 2.0 ** -12 + 2.0 ** -24], np.float32)
    a = np.array([2.0 ** -24 * (1 + 2.0 ** -12)], np.float32)
    c = np.array([1.0], np.float32)
    assert float(b[0]) == 1 - 2.0 ** -12 + 2.0 ** -24 and float(a[0]) == 2.0 ** -24 * (1 + 2.0 ** -12)
    assert exact_fma(b, a, c)[0] == 1 + 2.0 ** -23
    assert fma32_np(b, a, c)[0] == 1 + 2.0 ** -23
    assert oracle._fma32(b, a, c)[0] == np.float32(1 + 2.0 ** -23)
    assert old_fma(b, a, c)[0] == 1.0                    # the double rounding this reference exists to avoid


def test_fma32_near_midpoints_against_fractions():
    b, a, c = near_midpoint_triples(10000, 1)
    want = exact_fma(b, a, c)
    assert np.array_equal(fma32_np(b, a, c), want)
    assert np.array_equal(oracle._fma32(b, a, c).astype(np.float64), want)
    # the triples are hard ones: the double-rounded form gets thousands of them wrong
    assert (old_fma(b, a, c) != want).sum() > 2000


def test_fma32_random_triples_against_fractions():
    b, a, c = random_triples(10000, 2)
    want = exact_fma(b, a, c)
    got = fma32_np(b, a, c)
    assert np.array_equal(got, want)
    assert np.array_equal(np.signbit(got), np.signbit(want))
    assert np.array_equal(oracle._fma32(b, a, c).astype(np.float64), want)
    # the non-finite cases the kernels meet: inf and NaN operands propagate as IEEE fma does
    t = lambda *v: torch.tensor(v, dtype=torch.float64)                   # noqa: E731
    r = fma32(t(1.0, 1.0, 0.0, 2.0), t(math.inf, math.inf, math.inf, 3.0), t(1.0, -math.inf, 1.0, math.nan))
    assert r[0] == math.inf and r[1:].isnan().all()


# ------------------------------------------------------------------------------------------- CPU: the oracle
@pytest.mark.parametrize("tag", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("R,C,r", [(37, 1032, 5), (64, 516, 16), (5, 1408, 3)])
def test_oracle_equals_reference(tag, R, C, r):
    """The numpy oracle (tests/test_gpu_parity.py compares K14 / K15 with it bit for bit) and this reference agree."""
    W, A, B, M = lora_case(R, C, r, DT[tag], R * C + r, device="cpu")
    s = 16.0 / r
    Wn, An, Bn, Mn = W.float().numpy(), A.numpy(), B.numpy(), M.numpy()
    for remask in (True, False):
        want = merge(W, A, B, s, M, remask).float().numpy()
        got = oracle.sparselora_merge(Wn, tag, An, Bn, s, Mn, remask)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), remask
    for sparse in (True, False):
        want = effective_weight(W, A, B, s, M, sparse).float().numpy()
        got = oracle.sparselora_effective_weight(Wn, tag, An, Bn, s, Mn, sparse)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), sparse


# ------------------------------------------------------------------------------------------- CPU: the K16 bar
def coherent_case(device):
    """bf16 G, fp32 A and B, all positive, and a scaling just above 1: every G * s (exact in fp32) rounds back down to G
    in bf16, so an E left unrounded is off by 2^-10 of every term, all of one sign."""
    g = torch.Generator().manual_seed(5)
    R, C, r = 1000, 1408, 8
    G = (0.5 + 0.5 * torch.rand(R, C, generator=g)).bfloat16()
    A = 0.5 + 0.5 * torch.rand(r, C, generator=g)
    B = 0.5 + 0.5 * torch.rand(R, r, generator=g)
    M = torch.rand(R, C, generator=g) < 0.5
    return [t.to(device) for t in (G, A, B, M)] + [1.0 + 2.0 ** -10]


def test_grad_bar_catches_regressions():
    """Float64 emulations of three K16 faults land at least 10x over the bar the GPU tests hold the kernel to."""
    G, A, B, M, s = coherent_case("cpu")
    R, C = G.shape
    nA, nB = grad_depths(R, C, VEC["bf16"])
    A64, B64 = A.double(), B.double()
    ratios = {}
    for sparse in (True, False):
        dA, dB, SA, SB = lora_grads(G, A, B, s, M, sparse)
        keep = M if sparse else torch.ones_like(M)
        E_raw = torch.where(keep, mul32(G.double(), f32(s)), 0.0)                       # E not rounded to bf16
        ratios[f"unrounded dA {sparse}"] = bar_ratio(B64.T @ E_raw, dA, SA, nA)
        ratios[f"unrounded dB {sparse}"] = bar_ratio(E_raw @ A64.T, dB, SB, nB)
        E = torch.where(keep, round_dt(mul32(G.double(), f32(s)), torch.bfloat16), 0.0)
        ratios[f"last row dropped {sparse}"] = bar_ratio(dA - B64[-1:].T @ E[-1:], dA, SA, nA)
    dA, dB, SA, SB = lora_grads(G, A, B, s, M, True)
    E_all = round_dt(mul32(G.double(), f32(s)), torch.bfloat16)                         # the mask not applied
    ratios["unmasked dA"] = bar_ratio(B64.T @ E_all, dA, SA, nA)
    ratios["unmasked dB"] = bar_ratio(E_all @ A64.T, dB, SB, nB)
    print(f"\nK16 regression emulations, smallest error / bar: {min(ratios.values()):.3g}")
    assert min(ratios.values()) >= 10, ratios


# ------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def native(built_lib):
    from vlmc import native as n
    n.load()
    assert torch.cuda.is_available()
    return n


@pytest.fixture(scope="module")
def grad_ratios():
    r = {"dA": 0.0, "dB": 0.0}
    yield r
    print(f"\nK16 largest error / bar: dA {r['dA']:.3g}, dB {r['dB']:.3g}")


def check_tile_kernels(native, W, A, B, s, M, what):
    """K15 (sparse and dense) and K14 (with and without re-mask) against the reference, bit for bit; K15 leaves W as it
    was."""
    W0 = raw_bits(W).clone()
    for sparse in (True, False):
        got = native.sparselora_effective_weight(W, A, B, s, M, sparse)
        assert_same_bits(got, effective_weight(W, A, B, s, M, sparse), f"K15 sparse={sparse} {what}")
    assert torch.equal(raw_bits(W), W0)
    for remask in (True, False):
        Wm = W.clone()
        native.sparselora_merge(Wm, A, B, s, M, remask=remask)
        assert_same_bits(Wm, merge(W, A, B, s, M, remask), f"K14 remask={remask} {what}")


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("r", range(1, 17))
def test_tile_kernels_every_rank(native, tag, r):
    """R = 4097 (a last block of one row) by one column tile plus one vector: 2050 units, more than the grid, so CTA spans
    cross the column tile and restage A.  Scaling 16 / r (not a power of two for r = 3, 5, 6, 7, ...)."""
    R, C = 4097, COLS[tag][1]
    W, A, B, M = lora_case(R, C, r, DT[tag], 100 + r)
    check_tile_kernels(native, W, A, B, 16.0 / r, M, f"{tag} r={r}")


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("R", ROWS)
@pytest.mark.parametrize("ci", range(4))
def test_tile_kernels_ragged_shapes(native, tag, R, ci):
    C = COLS[tag][ci]
    r = (3, 5, 6, 7)[(ROWS.index(R) + ci) % 4]
    W, A, B, M = lora_case(R, C, r, DT[tag], R * 7 + ci)
    check_tile_kernels(native, W, A, B, 16.0 / r, M, f"{tag} {R}x{C} r={r}")


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("shape", VICUNA)
@pytest.mark.parametrize("r", [8, 16])
def test_tile_kernels_vicuna_shapes(native, tag, shape, r):
    R, C = shape
    W, A, B, M = lora_case(R, C, r, DT[tag], R + C + r)
    check_tile_kernels(native, W, A, B, 16.0 / r, M, f"{tag} {R}x{C} r={r}")


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f32", "f16", "bf16"])
def test_tile_kernels_row_pitches(native, tag):
    """W, mask and out as views with pitches ldw, ldm, ldo different from C and from each other: NaN in W's padding and
    True in the mask's are never used, a sentinel in out's padding survives, K15 writes nothing of W."""
    dt, V = DT[tag], VEC[tag]
    R, C, r, s = 37, 1408, 5, 16.0 / 5
    W, A, B, M = lora_case(R, C, r, dt, 77)
    Wp = torch.full((R, C + 3 * V), math.nan, dtype=dt, device="cuda")
    Wp[:, :C] = W
    Mp = torch.ones((R, C + 16), dtype=torch.bool, device="cuda")
    Mp[:, :C] = M
    Wv, Mv = Wp[:, :C], Mp[:, :C]
    assert Wv.stride(0) != C and Mv.stride(0) != C
    Wp0 = raw_bits(Wp).clone()
    for sparse in (True, False):
        outp = torch.full((R, C + 5 * V), -1234.5, dtype=dt, device="cuda")
        got = native.sparselora_effective_weight(Wv, A, B, s, Mv, sparse, out=outp[:, :C])
        assert got.data_ptr() == outp.data_ptr() and got.stride(0) == C + 5 * V
        assert_same_bits(outp[:, :C], effective_weight(W, A, B, s, M, sparse), f"K15 sparse={sparse} pitched")
        assert bool((outp[:, C:] == -1234.5).all())
        assert torch.equal(raw_bits(Wp), Wp0)
    for remask in (True, False):
        Wq = Wp.clone()
        native.sparselora_merge(Wq[:, :C], A, B, s, Mv, remask=remask)
        assert_same_bits(Wq[:, :C], merge(W, A, B, s, M, remask), f"K14 remask={remask} pitched")
        assert torch.equal(raw_bits(Wq[:, C:]), raw_bits(Wp[:, C:]))


def merge_batch_items(tag, ranks):
    """One R = 4097 item of 2050 units, then fifteen items of 1-3 rows (one to three units each) at every column count.
    The total is more than twice the largest grid, so every CTA span holds two units or more and the spans over the
    small items cover several of them."""
    Cs = COLS[tag][:3] + [2056]
    items = [(4097, COLS[tag][1], ranks[0])] + [(1 + i % 3, Cs[i % 4], ranks[(i + 1) % len(ranks)]) for i in range(15)]
    V = VEC[tag]
    units = sum(-(-C // (128 * V)) * -(-R // 4) for R, C, _ in items)
    assert units > 2 * MAX_GRID
    return items


def merge_inputs(items, dt, seed):
    cases = [lora_case(R, C, r, dt, seed + i) for i, (R, C, r) in enumerate(items)]
    return [c[0] for c in cases], [c[1] for c in cases], [c[2] for c in cases], [c[3] for c in cases]


def merge_batch_abi(native, Ws, As, Bs, scalings, Ms, remask):
    """vlmc_sparselora_merge_batch called directly (the Python wrapper sends ranks above 8 to the single-linear call)."""
    lib = native.load()
    items = (native.MergeItem * len(Ws))(*[native.MergeItem(W.data_ptr(), W.stride(0), W.shape[0], W.shape[1],
                                                            A.data_ptr(), B.data_ptr(), A.shape[0], float(s),
                                                            M.data_ptr(), M.stride(0))
                                           for W, A, B, s, M in zip(Ws, As, Bs, scalings, Ms)])
    assert lib.vlmc_sparselora_merge_batch(items, len(Ws), native._DTYPES[Ws[0].dtype], int(remask),
                                           native._stream(Ws[0])) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f32", "f16", "bf16"])
def test_merge_batch_spans_cross_items(native, tag):
    """The batched merge through the wrapper (more than 16 items, so it chunks them; mixed ranks, one above 8) and through
    the C ABI with ranks 9-16 mixed with low ranks: bit-equal to the single calls and to the reference."""
    dt = DT[tag]
    items = merge_batch_items(tag, [1, 2, 3, 5, 8]) + [(3, 1408, 12), (2, COLS[tag][0], 7), (1, 2056, 4)]
    assert len(items) > 16
    Ws, As, Bs, Ms = merge_inputs(items, dt, 300)
    sc = [16.0 / r for _, _, r in items]
    for remask in (True, False):
        got = [W.clone() for W in Ws]
        native.sparselora_merge_batch(got, As, Bs, sc, Ms, remask=remask)
        for i, (W, A, B, s, M) in enumerate(zip(Ws, As, Bs, sc, Ms)):
            single = W.clone()
            native.sparselora_merge(single, A, B, s, M, remask=remask)
            assert torch.equal(raw_bits(got[i]), raw_bits(single)), i
            assert_same_bits(got[i], merge(W, A, B, s, M, remask), f"batch item {i} {items[i]} remask={remask}")
    items = merge_batch_items(tag, [16, 9, 2, 11, 1, 13, 15, 10, 4, 12, 14, 3])
    assert len(items) == 16 and {r for _, _, r in items} >= set(range(9, 17))
    Ws, As, Bs, Ms = merge_inputs(items, dt, 400)
    sc = [16.0 / r for _, _, r in items]
    for remask in (True, False):
        got = [W.clone() for W in Ws]
        merge_batch_abi(native, got, As, Bs, sc, Ms, remask)
        for i, (W, A, B, s, M) in enumerate(zip(Ws, As, Bs, sc, Ms)):
            single = W.clone()
            native.sparselora_merge(single, A, B, s, M, remask=remask)
            assert torch.equal(raw_bits(got[i]), raw_bits(single)), i
            assert_same_bits(got[i], merge(W, A, B, s, M, remask), f"ABI batch item {i} {items[i]} remask={remask}")


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f32", "f16", "bf16"])
def test_masked_rule_non_finite(native, tag):
    """W = +-inf / NaN at kept and at masked positions, and LoRA products that overflow fp16: K15 and K14 still match the
    reference bit for bit.  Masked entries of K15's sparse weight are +0 whatever W or the product hold."""
    dt = DT[tag]
    R, C, r = 133, 1032, 8
    W, A, B, M = lora_case(R, C, r, dt, 55)
    g = torch.Generator(device="cuda").manual_seed(56)
    for v in (math.inf, -math.inf, math.nan):
        idx = torch.randint(0, R * C, (R * C // 100,), generator=g, device="cuda")
        W.view(-1)[idx] = v
    nonfinite = ~torch.isfinite(W)
    assert bool((nonfinite & M).any()) and bool((nonfinite & ~M).any())
    B[:8], B[8:16], A[:, :64] = 100.0, -100.0, 100.0          # |BA| = 8e4 there: past fp16's 65504
    check_tile_kernels(native, W, A, B, 2.0, M, f"{tag} non-finite")
    weff = native.sparselora_effective_weight(W, A, B, 2.0, M, True)
    assert bool((canon_bits(weff)[~M] == 0).all())
    if tag == "f16":
        kept = M[:16, :64] & torch.isfinite(W[:16, :64])
        assert bool(kept.any()) and bool(torch.isinf(weff[:16, :64][kept]).all())


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f32", "f16", "bf16"])
def test_masked_rule_negative_zero(native, tag):
    """B = 0 and negative W: K15's masked entries are +0 where the reference's expression (W + d) * mask gives -0."""
    dt = DT[tag]
    R, C, r = 64, 1408, 4
    W, A, B, M = lora_case(R, C, r, dt, 66)
    W = -W.abs() - 0.01
    B = torch.zeros_like(B)
    expr = (W + (B @ A).to(dt) * 4.0) * M                                  # lora.py:364-369
    assert bool(torch.signbit(expr[~M]).all())
    weff = native.sparselora_effective_weight(W, A, B, 4.0, M, True)
    assert bool((canon_bits(weff)[~M] == 0).all())
    assert torch.equal(weff, expr)                                          # equal as values: -0 == +0
    check_tile_kernels(native, W, A, B, 4.0, M, f"{tag} B = 0")


# ------------------------------------------------------------------------------------------- GPU: K16
def check_grads(native, G, A, B, s, M, ratios, what):
    """K16 with both values of `sparse` on G and M as given and on pitched copies (NaN in G's padding, True in the
    mask's): the same bits, and every element within the bar of its float64 value."""
    R, C = G.shape
    V = 4 if G.dtype == torch.float32 else 8
    nA, nB = grad_depths(R, C, V)
    Gp = torch.full((R, C + 3 * V), math.nan, dtype=G.dtype, device="cuda")
    Gp[:, :C] = G
    Mp = torch.ones((R, C + 24), dtype=torch.bool, device="cuda")
    Mp[:, :C] = M
    for sparse in (True, False):
        dA, dB = native.sparselora_lora_grads(G, A, B, s, M, sparse)
        dA2, dB2 = native.sparselora_lora_grads(Gp[:, :C], A, B, s, Mp[:, :C], sparse)
        assert torch.equal(raw_bits(dA), raw_bits(dA2)) and torch.equal(raw_bits(dB), raw_bits(dB2)), what
        rA, rB, SA, SB = lora_grads(G, A, B, s, M, sparse)
        qA, qB = bar_ratio(dA, rA, SA, nA), bar_ratio(dB, rB, SB, nB)
        ratios["dA"], ratios["dB"] = max(ratios["dA"], qA), max(ratios["dB"], qB)
        assert qA <= 1 and qB <= 1, (what, sparse, qA, qB)


def grad_case(R, C, r, dt, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    G = (torch.randn(R, C, generator=g, device="cuda") * 0.01).to(dt)
    A = torch.randn(r, C, generator=g, device="cuda") * 0.1
    B = torch.randn(R, r, generator=g, device="cuda") * 0.1
    M = torch.rand(R, C, generator=g, device="cuda") < 0.5
    return G, A, B, M


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("R", GRAD_ROWS)
@pytest.mark.parametrize("ci", range(4))
def test_grads_ragged_shapes(native, grad_ratios, tag, R, ci):
    C = COLS[tag][ci]
    r = GRAD_RANKS[(GRAD_ROWS.index(R) + ci) % len(GRAD_RANKS)]
    G, A, B, M = grad_case(R, C, r, DT[tag], R + ci)
    check_grads(native, G, A, B, 16.0 / r, M, grad_ratios, f"{tag} {R}x{C} r={r}")


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("r", GRAD_RANKS)
def test_grads_every_template(native, grad_ratios, tag, r):
    """R = 4737: 17 rows per chunk, 279 chunks, a last chunk of 11 rows."""
    G, A, B, M = grad_case(4737, 1408, r, DT[tag], 900 + r)
    check_grads(native, G, A, B, 16.0 / r, M, grad_ratios, f"{tag} 4737x1408 r={r}")


@pytest.mark.gpu
def test_grads_coherent_case(native, grad_ratios):
    """The case test_grad_bar_catches_regressions builds its emulations on: the kernel itself stays within the bar."""
    G, A, B, M, s = coherent_case("cuda")
    check_grads(native, G, A, B, s, M, grad_ratios, "coherent")


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f32", "f16", "bf16"])
def test_grads_non_finite(native, grad_ratios, tag):
    """inf / NaN in G at masked positions change nothing (sparse).  At kept positions the outputs are non-finite exactly
    where the float64 reference of the documented rule is, and the finite ones stay within the bar."""
    dt = DT[tag]
    R, C, r = 4737, 1032, 9
    G, A, B, M = grad_case(R, C, r, dt, 31)
    nA, nB = grad_depths(R, C, VEC[tag])
    dA, dB = native.sparselora_lora_grads(G, A, B, 2.0, M, True)
    g = torch.Generator(device="cuda").manual_seed(32)
    Gm = G.clone()
    for v in (math.nan, math.inf, -math.inf):
        Gm[~M & (torch.rand(R, C, generator=g, device="cuda") < 0.05)] = v
    assert int((~torch.isfinite(Gm)).sum()) > 1000
    dAm, dBm = native.sparselora_lora_grads(Gm, A, B, 2.0, M, True)
    assert torch.equal(raw_bits(dA), raw_bits(dAm)) and torch.equal(raw_bits(dB), raw_bits(dBm))
    Gk, Mk = G.clone(), M.clone()
    rows = torch.tensor([5, 17, 2000, 2000, 4736], device="cuda")
    cols = torch.tensor([100, 7, 900, 901, 1031], device="cuda")
    Mk[rows, cols] = True
    Gk[rows, cols] = torch.tensor([math.inf, math.nan, -math.inf, math.inf, -math.inf], device="cuda").to(dt)
    for sparse in (True, False):
        dA, dB = native.sparselora_lora_grads(Gk, A, B, 2.0, Mk, sparse)
        rA, rB, SA, SB = lora_grads(Gk, A, B, 2.0, Mk, sparse)
        for got, ref, S, n in ((dA, rA, SA, nA), (dB, rB, SB, nB)):
            fin = torch.isfinite(ref)
            assert torch.equal(torch.isfinite(got), fin)
            assert 0 < int((~fin).sum()) < fin.numel()
            assert bar_ratio(got[fin], ref[fin], S[fin], n) <= 1


@pytest.mark.gpu
def test_grads_deterministic_through_shared_workspace(native):
    """Repeated calls give the same bits, also after calls of other shapes and ranks, smaller and larger, in between
    (the larger one makes the wrapper allocate a new workspace that still holds its partial sums)."""
    G, A, B, M = grad_case(4737, 1408, 5, torch.bfloat16, 41)
    first = native.sparselora_lora_grads(G, A, B, 3.2, M, True)
    for R, C, r in ((300, 1032, 16), (11008, 4096, 16)):
        Gx, Ax, Bx, Mx = grad_case(R, C, r, torch.bfloat16, R)
        native.sparselora_lora_grads(Gx, Ax, Bx, 2.0, Mx, True)
        again = native.sparselora_lora_grads(G, A, B, 3.2, M, True)
        for x, y in zip(first, again):
            assert torch.equal(raw_bits(x), raw_bits(y))
