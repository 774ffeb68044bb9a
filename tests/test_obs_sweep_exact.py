"""The SparseGPT column-block OBS sweep (K11-K13, csrc/obs.cu) against exact references.

Layer 1, bit for bit.  On a block-diagonal factor (U[i1:i2, i2:] = 0 for every 128-column block) the 3xTF32 trailing
update subtracts exact zeros, and every other step of the kernel rounds as oracle.sparsegpt_fasterprune does in numpy
fp32.  Weights, keep mask, per-block threshold and pruned count must then equal the oracle's exactly, at ragged widths
and row counts, every dtype, every n:m instance, exact ties, dead channels, every schedule switch and every store path.
Layer 2, float64.  On a dense factor the trailing GEMM differs from fp32 matmul in the last bits, so the kernel's own
keep mask is fed to a float64 recursion on the kernel's super-block schedule: kept weights within C_BAR * 2^-24 of the
recursion run on absolute values, pruned ones exactly +0, and the mask valid to a relative ETA on the float64 scores.
A CPU test shows that five plausible schedule defects land far above that bar.
Layer 3: vlmc_obs_sweep_guarded with its flag set, row shards in lock-step, and argument rejections.
"""
import functools
import math

import numpy as np
import pytest
import torch

from oracle import oracle

F32 = np.float32
U24 = 2.0 ** -24
TAGS = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}
CODES = {"f32": 0, "f16": 1, "bf16": 2}
BAD_ARG, UNSUPPORTED = -1, -2

# Layer 2 bars.  Kept weights: |W - W64| <= C_BAR * 2^-24 * env (+ half an ulp of the output dtype), env the recursion on
# absolute values.  Measured on an NVIDIA B200 (1000 W power limit) over F64_CASES: at most 11.2 (f32 weights), 1.3
# beyond the half ulp (f16), 0.2 (bf16).  The smallest margin of the emulated schedule defects is 21x, for a single-pass
# TF32 trailing product.
C_BAR = 32.0
# Masks against the float64 scores of the same recursion: a pruned score may exceed a kept one by this relative amount.
# Measured on the same B200 runs: no pruned score exceeds any kept score of its block or group at all; ETA leaves room
# for the fp32 error of scores near the threshold (C_BAR * 2^-24 of the envelope, relative to |w|).
ETA = 1e-4

SCHEDULE_ENV = ("VLMC_OBS_SUPERBLOCK", "VLMC_OBS_FAR_CHUNKED", "VLMC_CHOL_LOOKAHEAD", "VLMC_OBS_FUSED")


# ------------------------------------------------------------------------------------------- references (CPU)
@functools.lru_cache(maxsize=None)
def factor(C, seed, dense=False, dead_key=(), unit_half=False):
    """U = cholesky(H^-1, upper) in float64 rounded to fp32, from a Hessian that is block-diagonal over 128-column
    blocks (or dense).  Dead channels are prepared as vlmc_hessian_prepare does: zero row and column, H[d, d] = 1.
    unit_half: every row divided by its diagonal and halved, so diag(U) = 0.5 everywhere (exact ties of w^2 / d^2)."""
    rng = np.random.default_rng(seed)
    dead = np.zeros(C, bool)
    dead[list(dead_key)] = True
    U = np.zeros((C, C))
    for a in ([0] if dense else range(0, C, 128)):
        b = C if dense else min(a + 128, C)
        n = b - a
        X = rng.standard_normal((n, min(n, 256) + 8))
        H = X @ X.T / X.shape[1] + 0.1 * np.eye(n)
        d = dead[a:b]
        H[d, :] = 0
        H[:, d] = 0
        H[d, d] = 1
        U[a:b, a:b] = np.linalg.cholesky(np.linalg.inv(H)).T
    if unit_half:
        U = U / np.diag(U)[:, None] * 0.5
    U = np.triu(U).astype(F32)
    U.setflags(write=False)
    return U, dead


def make_w(R, C, seed, tag, quant=False):
    """fp32 values of a `tag` weight, no -0 (the sign of a kept zero is not part of the contract)."""
    rng = np.random.default_rng(seed)
    if quant:
        w = rng.integers(-6, 7, (R, C)).astype(F32) * F32(2.0 ** -5)
    else:
        w = (rng.standard_normal((R, C)) * 0.05).astype(F32)
    return oracle.round_to_dtype(w, tag) + F32(0.0)


def tf32(x):
    """TF32 value of fp32 x as the 3xTF32 split rounds it (round to nearest, ties away from zero), as float64."""
    b = np.asarray(x, F32).view(np.uint32).astype(np.uint64)
    return (((b + 0x1000) & ~np.uint64(0x1FFF)) & 0xFFFFFFFF).astype(np.uint32).view(F32).astype(np.float64)


FAULTS = ("drop_far", "other_err_buffer", "u_rows_offset", "near_short", "tf32_single_pass")


def obs_ref(W0, U, dead, sp=0.0, n=0, m=0, keep=None, dt=np.float64, sb=4, env=False, fault=None):
    """The OBS sweep (sparsegpt_pruner.py:160-215) in `dt` arithmetic, on the kernel's super-block schedule: after a
    block the rest of its super-block gets that block's errors (near), and a finished super-block's errors go to every
    later column at once (far), read from one of two alternating Err buffers.
    keep=None decides the mask the oracle's way: unstructured score <= the int(R*bs*sp)-th block score, n:m the n
    smallest of each group on the compensated values, ties to the lower column.  Otherwise `keep` is used as given.
    env: the same recursion on absolute values (|W0|, |err| = |w| / |d|, products added): the error envelope.
    fault: one of FAULTS, a defect of the trailing update emulated for the CPU self-test.
    Returns (W, keep, decision scores, per-block thresholds)."""
    W = np.array(W0, dt)
    if dead is not None:
        W[:, dead] = 0
    Ud = np.asarray(U, dt)
    if env:
        W, Ud = np.abs(W), np.abs(Ud)
    R, C = W.shape
    pruned = np.zeros((R, C), bool)
    dec = np.zeros((R, C), dt)
    thr = []
    errbuf = np.zeros((2, R, sb * 128), dt)
    diag = np.diag(Ud)
    for blk in range((C + 127) // 128):
        i1, i2 = blk * 128, min(blk * 128 + 128, C)
        bs = i2 - i1
        W1 = W[:, i1:i2]
        d = diag[i1:i2]
        E = errbuf[(blk // sb) & 1, :, (blk % sb) * 128:(blk % sb) * 128 + 128]
        E[:] = 0
        if n == 0:
            s = ((W1 * W1) / (d * d)[None, :]).astype(dt)
            dec[:, i1:i2] = s
            if keep is None:
                kk = int(s.size * sp)
                thr.append(np.partition(s.ravel(), kk)[kk])
                pruned[:, i1:i2] = s <= thr[-1]
        for i in range(bs):
            c = i1 + i
            if n and i % m == 0:
                g = ((W1[:, i:i + m] ** 2) / ((d[i:i + m] ** 2)[None, :])).astype(dt)
                dec[:, c:c + g.shape[1]] = g
                if keep is None:
                    order = np.argsort(g, axis=1, kind="stable")[:, :n]
                    np.put_along_axis(pruned[:, c:c + g.shape[1]], order, True, axis=1)
            if keep is not None:
                pruned[:, c] = ~keep[:, c]
            w = W1[:, i].copy()
            p = pruned[:, c]
            if env:
                err = np.where(p, w / d[i], dt(0))
                W1[:, i:] = W1[:, i:] + err[:, None] * Ud[c, c:i2][None, :]
            else:
                err = ((w - np.where(p, dt(0), w)) / d[i]).astype(dt)
                W1[:, i:] = (W1[:, i:] - (err[:, None] * Ud[c, c:i2][None, :]).astype(dt)).astype(dt)
            W1[p, i] = 0
            E[:, i] = err
        if i2 >= C:
            continue
        slot = blk % sb
        sb_i1 = (blk - slot) * 128
        sb_i2 = min(sb_i1 + sb * 128, C)
        sign = 1 if env else -1

        def prod(A, B):
            if fault == "tf32_single_pass":
                return tf32(A) @ tf32(B)
            return A @ B

        if i2 < sb_i2:
            hi = sb_i2 - 128 if fault == "near_short" else sb_i2
            if hi > i2:
                W[:, i2:hi] = (W[:, i2:hi] + sign * prod(E[:, :bs], Ud[i1:i2, i2:hi])).astype(dt)
        elif sb_i2 < C:
            if fault == "drop_far" and blk // sb == 0:
                continue
            K = i2 - sb_i1
            buf = errbuf[((blk // sb) & 1) ^ (fault == "other_err_buffer"), :, :K]
            off = 1 if fault == "u_rows_offset" else 0
            Ufar = np.zeros((K, C - sb_i2), dt)
            rows = Ud[sb_i1 + off:sb_i1 + off + K, sb_i2:]
            Ufar[:rows.shape[0]] = rows
            W[:, sb_i2:] = (W[:, sb_i2:] + sign * prod(buf, Ufar)).astype(dt)
    return W, ~pruned, dec, thr


def out_bits(x, tag):
    """Integer view of fp32 values rounded to `tag`, as the kernel's output holds them."""
    x = np.asarray(x, F32)
    if tag == "f32":
        return x.view(np.uint32)
    if tag == "f16":
        return x.astype(np.float16).view(np.uint16)
    return (oracle.round_to_dtype(x, "bf16").view(np.uint32) >> 16).astype(np.uint16)


def half_ulp(x, tag):
    if tag == "f32":
        return np.zeros_like(x)
    mant, emin = (10, -14) if tag == "f16" else (7, -126)
    e = np.floor(np.log2(np.maximum(np.abs(x), 2.0 ** emin)))
    return 2.0 ** (e - mant - 1)


def importance_bar(R, score):
    """obs_importance_kernel: each term w^2 / d^2 carries three roundings, a thread adds ceil(R / min(R, 64)) of them in
    fp32, then five shuffle levels, eight warp partials, the fp32 store of the double sum and the fp32 mean: all terms
    are non-negative, so the error is below (that depth) * 2^-24 * score."""
    depth = 3 + math.ceil(R / min(R, 64)) + 5 + 8 + 2
    return depth * U24 * abs(score)


# ------------------------------------------------------------------------------------------- case lists
WIDTHS = [4, 12, 100, 124, 128, 132, 260, 1028, 2180]
ROWS = [1, 3, 5, 31, 33, 127, 129, 300]
NM = [(1, 2), (1, 4), (2, 4), (3, 4), (1, 8), (4, 8), (7, 8), (2, 16), (8, 16), (15, 16)]
NM_WIDTHS = [128, 132, 260]
SPS = [0.0, 0.5, 0.9]
DEAD_C = 260
DEAD_COLS = (3, 77, 100) + tuple(range(128, 256)) + (257,)     # a fully dead block and one in the partial last block


def exact_cases():
    """(R, C, tag, sp, n, m, kind): kind 'rand' | 'quant' (exact ties at constant d) | 'dead'."""
    tags = list(TAGS)
    cases = []
    for j, C in enumerate(WIDTHS):                              # every width, unstructured, rows cycled
        cases.append((ROWS[j % len(ROWS)], C, tags[j % 3], SPS[j % 3], 0, 0, "rand"))
    for j, R in enumerate(ROWS):                                 # every row count at a partial last block
        cases.append((R, 132 if j % 2 else 260, tags[(j + 1) % 3], 0.5, *((0, 0) if j % 2 else (2, 4)), "rand"))
    for j, (n, m) in enumerate(NM):                              # every n:m on every n:m width
        for k, C in enumerate(NM_WIDTHS):
            cases.append((ROWS[(j + k) % len(ROWS)], C, tags[(j + k) % 3], 0.0, n, m, "rand"))
    for j, tag in enumerate(tags):
        cases.append((33, 260, tag, 0.5, 0, 0, "quant"))         # hundreds of exact ties at the threshold
        cases.append((31, 132, tag, 0.0, 0, 0, "quant"))         # sp = 0: the minimum and all its ties
        cases.append((33, DEAD_C, tag, 0.0, 0, 0, "dead"))        # every dead column ties at the minimum score
        cases.append((5, DEAD_C, tag, 0.5, 0, 0, "dead"))
        cases.append((31, DEAD_C, tag, 0.0, 2, 4, "dead"))
        cases.append((25, 132, tag, 0.29, 0, 0, "rand"))          # 4-column last block: numel 100, rank 28 (not 29)
        cases.append((25, 132, tag, 0.57, 0, 0, "rand"))          # rank 56 (not 57)
    return cases


EXACT_CASES = exact_cases()
BIG_R = 14213           # > 3 * 148 CTAs * 32 rows: the grid-stride loop of obs_sweep4_kernel, above the fused capacity

# Layer 2: (R, C, tag, sp, n, m, superblock, far_chunked)
MODES = [(0.5, 0, 0), (0.0, 2, 4), (0.0, 4, 8), (0.0, 8, 16)]
F64_WIDTHS = [132, 260, 1028, 2180, 4100]
F64_ROWS = [1, 5, 33, 300]


def f64_cases():
    cases = []
    for j, tag in enumerate(TAGS):
        for k, mode in enumerate(MODES):
            i = 4 * j + k
            C = F64_WIDTHS[i % len(F64_WIDTHS)]
            R = F64_ROWS[(i + j) % len(F64_ROWS)]
            if C == 4100 and R == 300:
                R = 33                                           # keeps the numpy recursions short
            cases.append((R, C, tag, *mode, (1, 2, 4, 8)[(i + j) % 4], (j + k) % 2))
    return cases


F64_CASES = f64_cases()


# ------------------------------------------------------------------------------------------- CPU tests
def test_case_lists_cover_every_axis():
    ex = EXACT_CASES
    assert {c[1] for c in ex if c[4] == 0} >= set(WIDTHS)
    assert {c[0] for c in ex} >= set(ROWS)
    assert {(c[4], c[5], c[1]) for c in ex if c[4]} >= {(n, m, C) for n, m in NM for C in NM_WIDTHS}
    assert {c[2] for c in ex if c[4] == 0} == set(TAGS) and {c[2] for c in ex if c[4]} == set(TAGS)
    assert {c[3] for c in ex if c[4] == 0} >= set(SPS)
    assert {m for *_, m, _k in ex if m} == {2, 4, 8, 16}
    assert {(c[6], c[4] == 0) for c in ex} >= {("quant", True), ("dead", True), ("dead", False)}
    # int(numel * sp) decided by double rounding on a 4-column last block
    for R, C, tag, sp, n, m, kind in ex:
        if (R, C, sp) in ((25, 132, 0.29), (25, 132, 0.57)):
            assert int(R * 4 * sp) == round(R * 4 * sp) - 1
    assert any((R, C, sp) == (25, 132, 0.29) for R, C, tag, sp, *_ in ex)
    assert any((R, C, sp) == (25, 132, 0.57) for R, C, tag, sp, *_ in ex)
    # widths: single partial blocks, a 4-column last block, and more than 2 * 8 blocks (look-ahead at every superblock)
    assert min(WIDTHS) < 128 and any(C % 128 == 4 for C in WIDTHS) and (max(WIDTHS) + 127) // 128 > 16
    f = F64_CASES
    assert {c[1] for c in f} == set(F64_WIDTHS) and {c[0] for c in f} == set(F64_ROWS)
    assert {(c[2], c[3], c[4], c[5]) for c in f} == {(t, *mo) for t in TAGS for mo in MODES}
    assert {c[6] for c in f} == {1, 2, 4, 8} and {c[7] for c in f} == {0, 1}
    assert max(R * C for R, C, *_ in f) <= 300 * 2180


@pytest.mark.parametrize("sp,n,m,kind,sb", [(0.5, 0, 0, "rand", 1), (0.0, 2, 4, "dead", 1), (0.3, 0, 0, "quant", 1),
                                            (0.0, 1, 8, "rand", 1), (0.5, 0, 0, "dense", 1), (0.0, 2, 4, "dense", 1)])
def test_fp32_reference_equals_the_oracle(sp, n, m, kind, sb):
    """obs_ref in fp32 on the reference's block-by-block schedule is the oracle bit for bit (its mask and thresholds are
    what layer 1 compares the kernel's with); in float64 it agrees with the oracle to fp32 rounding."""
    R, C = 13, 260
    dead_key = (5, 130, 257) if kind == "dead" else ()
    U, dead = factor(C, 5, dense=kind == "dense", dead_key=dead_key, unit_half=kind == "quant")
    W0 = make_w(R, C, 6, "f32", quant=kind == "quant")
    Wo, so, _ = oracle.sparsegpt_fasterprune(W0, "f32", None, sp, n, m, U=U, dead=dead)
    W, keep, _, thr = obs_ref(W0, U, dead, sp, n, m, dt=np.float32, sb=sb)
    assert np.array_equal(W.view(np.uint32), Wo.view(np.uint32))
    nz = (W0 != 0) & ~dead[None, :]
    assert np.array_equal(keep[nz], (Wo != 0)[nz])
    W64, keep64, _, _ = obs_ref(W0, U, dead, sp, n, m, keep=keep)
    env = obs_ref(W0, U, dead, sp, n, m, keep=keep, env=True)[0]
    assert np.all(np.abs(W64 - Wo) <= C_BAR * U24 * env)
    assert np.array_equal(keep64, keep)
    # a different super-block size changes only the order of the trailing sums
    W4 = obs_ref(W0, U, dead, sp, n, m, keep=keep, sb=4)[0]
    assert np.all(np.abs(W4 - W64) <= 1e-12 * (env + 1e-30))


def _fault_margins():
    R, C = 33, 1028
    U, dead = factor(C, 11, dense=True)
    W0 = make_w(R, C, 12, "f32")
    _, keep, _, _ = obs_ref(W0, U, dead, 0.5)
    ref = obs_ref(W0, U, dead, keep=keep)[0]
    bar = C_BAR * U24 * obs_ref(W0, U, dead, keep=keep, env=True)[0]
    out = {}
    for f in FAULTS:
        got = obs_ref(W0, U, dead, keep=keep, fault=f)[0]
        out[f] = float(np.max(np.abs(got - ref)[keep] / bar[keep]))
    return out


def test_schedule_faults_land_far_above_the_bar():
    """Five defects of the trailing update, emulated in float64 with the mask held fixed: each must miss the layer-2 bar
    by 10x or more on this case (dense factor, 9 blocks: two full super-blocks with a far update each)."""
    margins = _fault_margins()
    print("fault margins (x bar):", {k: round(v, 1) for k, v in margins.items()}, "smallest", round(min(margins.values()), 1))
    for f, v in margins.items():
        assert v >= 10, (f, v)


# ------------------------------------------------------------------------------------------- GPU helpers
@pytest.fixture(scope="module")
def native(built_lib):
    from vlmc import native as n
    n.load()
    assert torch.cuda.is_available()
    return n


@pytest.fixture
def schedule(monkeypatch):
    """Default schedule unless a test sets it; the kernel reads these on every call."""
    for k in SCHEDULE_ENV:
        monkeypatch.delenv(k, raising=False)

    def set_(**kv):
        for k, v in kv.items():
            monkeypatch.setenv(k, str(v))
    return set_


def dev_w(W0, tag):
    return torch.from_numpy(np.ascontiguousarray(W0)).to(TAGS[tag]).cuda()


def dev_u(U):
    return torch.from_numpy(np.array(U)).cuda()


def dev_dead(dead):
    return torch.from_numpy(dead.astype(np.uint8)).cuda()


def bits(t):
    t = t.detach().cpu().contiguous()
    return t.view(torch.int32 if t.dtype == torch.float32 else torch.int16).numpy()


def run(native, W0, tag, U, dead, sp, n, m, keep=None):
    W = dev_w(W0, tag)
    k, score = native.obs_sweep(W, dev_u(U), sp, n, m, dead=dev_dead(dead), want_mask=keep is None, keep=keep)
    torch.cuda.synchronize()
    return W, k, score


@functools.lru_cache(maxsize=64)
def exact_ref(R, C, tag, sp, n, m, kind, seed):
    dead_key = DEAD_COLS if kind == "dead" else ()
    U, dead = factor(C, seed, dead_key=dead_key, unit_half=kind == "quant")
    W0 = make_w(R, C, seed + 1, tag, quant=kind == "quant")
    Wo, _, _ = oracle.sparsegpt_fasterprune(W0, tag, None, sp, n, m, U=U, dead=dead)
    W32, keep, _, thr = obs_ref(W0, U, dead, sp, n, m, dt=np.float32, sb=1)
    assert np.array_equal(oracle.round_to_dtype(W32, tag).view(np.uint32), Wo.view(np.uint32))
    return W0, U, dead, Wo, keep, thr


def check_exact(native, R, C, tag, sp, n, m, kind, seed=1):
    W0, U, dead, Wo, keep_ref, thr = exact_ref(R, C, tag, sp, n, m, kind, seed)
    W, keep, score = run(native, W0, tag, U, dead, sp, n, m)
    got = bits(W)
    assert np.array_equal(got, out_bits(Wo, tag).view(got.dtype)), "weights differ from the oracle"
    keep = keep.cpu().numpy()
    assert np.array_equal(keep, keep_ref), "keep mask differs from the oracle's"
    nz = W0 != 0
    if dead is not None:
        nz[:, dead] = False
    assert np.array_equal(keep[nz], (W.float().cpu().numpy() != 0)[nz])
    if n == 0:
        Wd = np.where(dead[None, :], F32(0), W0)
        d = np.diag(U)
        for b, t in enumerate(thr):
            i1, i2 = 128 * b, min(128 * b + 128, C)
            # the block scores the threshold was taken from are the block-start values: W0 itself on this factor
            s = ((Wd[:, i1:i2] * Wd[:, i1:i2]) / (d[i1:i2] * d[i1:i2])[None, :]).astype(F32)
            assert np.sort(s.ravel())[int(R * (i2 - i1) * sp)] == t
            assert (~keep[:, i1:i2]).sum() == (s <= t).sum() >= int(R * (i2 - i1) * sp) + 1
    else:
        for c0 in range(0, C, m):
            w = min(m, C - c0)
            assert bool(((~keep[:, c0:c0 + w]).sum(1) == min(n, w)).all())
    Wd = np.where(dead[None, :], 0.0, W0.astype(np.float64))
    s64 = float(np.mean(Wd ** 2 / np.diag(U).astype(np.float64)[None, :] ** 2))
    assert abs(score.item() - s64) <= importance_bar(R, s64), (score.item(), s64)
    return abs(score.item() - s64) / max(s64, 1e-300)


# ------------------------------------------------------------------------------------------- layer 1: bit for bit
@pytest.mark.gpu
@pytest.mark.parametrize("R,C,tag,sp,n,m,kind", EXACT_CASES)
def test_sweep_is_bit_exact_on_a_block_diagonal_factor(native, schedule, R, C, tag, sp, n, m, kind):
    rel = check_exact(native, R, C, tag, sp, n, m, kind)
    print(f"importance rel err {rel:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("sp,n,m,fused", [(0.0, 2, 4, None), (0.5, 0, 0, "1"), (0.5, 0, 0, "0")])
def test_grid_stride_rows_are_bit_exact(native, schedule, sp, n, m, fused):
    """R = 14213 rows at C = 132 reach the grid-stride loop of obs_sweep4_kernel; a fused request there exceeds the
    cooperative capacity and falls back to the three-pass path, still exact."""
    if fused is not None:
        schedule(VLMC_OBS_FUSED=fused)
    check_exact(native, BIG_R, 132, "bf16", sp, n, m, "rand")


@pytest.mark.gpu
@pytest.mark.parametrize("sp,n,m,tag", [(0.5, 0, 0, "bf16"), (0.0, 2, 4, "f16")])
def test_every_schedule_switch_gives_the_same_bits(native, schedule, sp, n, m, tag):
    """C = 2180 (18 blocks): near and far updates at every super-block size, the look-ahead side stream, chunked and
    one-pass far GEMMs, fused and three-pass unstructured blocks - all the oracle's bits on a block-diagonal factor."""
    for sb in (1, 2, 4, 8):
        for far in (0, 1):
            for la in (0, 1):
                for fused in ((0, 1) if n == 0 else (1,)):
                    schedule(VLMC_OBS_SUPERBLOCK=sb, VLMC_OBS_FAR_CHUNKED=far, VLMC_CHOL_LOOKAHEAD=la,
                             VLMC_OBS_FUSED=fused)
                    check_exact(native, 129, 2180, tag, sp, n, m, "rand")


def _padded(W0, tag, layout):
    """W and keep as views that force element-wise stores: 'odd_ldw' (row pitch C + 1), 'offset' (W one element past
    a 16-byte boundary), 'ldm' (mask pitch C + 3).  Padding holds sentinels."""
    R, C = W0.shape
    pw = {"odd_ldw": 1, "offset": 4, "ldm": 0}[layout]
    Wb = torch.full((R, C + pw), 3.0, dtype=TAGS[tag], device="cuda")
    W = Wb[:, 1:C + 1] if layout == "offset" else Wb[:, :C]
    W.copy_(dev_w(W0, tag))
    pm = 3 if layout == "ldm" else 0
    Kb = torch.full((R, C + pm), 0xA5, dtype=torch.uint8, device="cuda")
    return Wb, W, Kb


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["odd_ldw", "offset", "ldm"])
@pytest.mark.parametrize("tag", list(TAGS))
@pytest.mark.parametrize("sp,n,m,fused", [(0.5, 0, 0, "1"), (0.5, 0, 0, "0"), (0.0, 2, 4, None)])
def test_element_wise_stores_equal_the_vector_stores(native, schedule, layout, tag, sp, n, m, fused):
    if fused is not None:
        schedule(VLMC_OBS_FUSED=fused)
    R, C = 33, 260
    W0, U, dead, Wo, keep_ref, _ = exact_ref(R, C, tag, sp, n, m, "rand", 3)
    Wv, kv, _ = run(native, W0, tag, U, dead, sp, n, m)
    Wb, W, Kb = _padded(W0, tag, layout)
    pad_w, pad_k = bits(Wb).copy(), Kb.cpu().numpy().copy()
    keep = Kb[:, :C].view(torch.bool)
    native.obs_sweep(W, dev_u(U), sp, n, m, dead=dev_dead(dead), keep=keep)
    torch.cuda.synchronize()
    assert np.array_equal(bits(W), bits(Wv))
    assert np.array_equal(bits(W), out_bits(Wo, tag).view(bits(W).dtype))
    k8 = Kb.cpu().numpy()
    assert np.array_equal(k8[:, :C], keep_ref.astype(np.uint8)) and np.array_equal(k8[:, :C].astype(bool), kv.cpu().numpy())
    # sentinels outside the matrix survive
    wb = bits(Wb)
    inside = np.zeros(wb.shape, bool)
    c0 = 1 if layout == "offset" else 0
    inside[:, c0:c0 + C] = True
    assert np.array_equal(wb[~inside], pad_w[~inside])
    assert np.array_equal(k8[:, C:], pad_k[:, C:])


# ------------------------------------------------------------------------------------------- layer 2: float64
def _f64_check(native, R, C, tag, sp, n, m, seed=21):
    dead_key = (7, C - 3)
    U, dead = factor(C, seed, dense=True, dead_key=dead_key)
    W0 = make_w(R, C, seed + 1, tag)
    W, keep, _ = run(native, W0, tag, U, dead, sp, n, m)
    keep = keep.cpu().numpy()
    got = W.float().cpu().numpy().astype(np.float64)
    W64, _, dec, _ = obs_ref(W0, U, dead, sp, n, m, keep=keep)
    env = obs_ref(W0, U, dead, sp, n, m, keep=keep, env=True)[0]
    gbits = bits(W)
    assert np.all(gbits[~keep] == 0), "pruned weights must be +0"
    excess = np.abs(got - W64) - half_ulp(np.maximum(np.abs(got), np.abs(W64)), tag)
    ratio = float(np.max(np.where(keep, excess / (U24 * env + 1e-300), 0.0)))
    assert ratio <= C_BAR, f"kept weights {ratio:.1f} x 2^-24 env off float64"
    # mask validity on the float64 decision scores
    worst = 0.0
    if n == 0:
        for b in range((C + 127) // 128):
            i1, i2 = 128 * b, min(128 * b + 128, C)
            s, k = dec[:, i1:i2], keep[:, i1:i2]
            kk = int(s.size * sp)
            assert (~k).sum() >= kk + 1
            if k.any() and (~k).any():
                worst = max(worst, float(s[~k].max() / s[k].min()) - 1 if s[k].min() > 0 else 0.0)
                assert s[~k].max() <= s[k].min() * (1 + ETA)
            sk = np.partition(s.ravel(), kk)[kk]
            assert (~k).sum() - (kk + 1) <= int((np.abs(s - sk) <= ETA * sk).sum())
    else:
        for c0 in range(0, C, m):
            w = min(m, C - c0)
            s, k = dec[:, c0:c0 + w], keep[:, c0:c0 + w]
            assert bool(((~k).sum(1) == min(n, w)).all())
            if w > n:
                pmax = np.where(~k, s, -np.inf).max(1)
                kmin = np.where(k, s, np.inf).min(1)
                assert bool((pmax <= kmin * (1 + ETA)).all())
                with np.errstate(divide="ignore", invalid="ignore"):
                    r = np.where(kmin > 0, pmax / kmin - 1, 0.0)
                worst = max(worst, float(r.max()))
    return ratio, worst, W, keep


@pytest.mark.gpu
@pytest.mark.parametrize("R,C,tag,sp,n,m,sb,far", F64_CASES)
def test_dense_factor_against_float64(native, schedule, R, C, tag, sp, n, m, sb, far):
    schedule(VLMC_OBS_SUPERBLOCK=sb, VLMC_OBS_FAR_CHUNKED=far)
    ratio, worst, _, _ = _f64_check(native, R, C, tag, sp, n, m)
    print(f"f64 {tag} R={R} C={C} sp={sp} {n}:{m} sb={sb} far={far}: err {ratio:.2f} x 2^-24 env "
          f"({ratio / C_BAR:.3f} of bar), mask excess {worst:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("tag", list(TAGS))
def test_dense_factor_f32_output(native, schedule, tag):
    """The same cases in f32 weights: the fp32 error without the output rounding."""
    for R, C, t, sp, n, m, sb, far in F64_CASES:
        if t == tag and C <= 1028:
            schedule(VLMC_OBS_SUPERBLOCK=sb, VLMC_OBS_FAR_CHUNKED=far)
            ratio, worst, _, _ = _f64_check(native, R, C, "f32", sp, n, m)
            print(f"f64 f32-out R={R} C={C} {n}:{m}: err {ratio:.2f} x 2^-24 env, mask excess {worst:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("C,sp,n,m", [(2180, 0.5, 0, 0), (4100, 0.0, 2, 4), (1028, 0.5, 0, 0)])
def test_dense_factor_identities(native, schedule, C, sp, n, m):
    """Fused and three-pass, look-ahead on and off, two runs and a run on a second stream: the same bits."""
    R, tag = 65, "bf16"
    U, dead = factor(C, 21, dense=True, dead_key=(7, C - 3))
    W0 = make_w(R, C, 32, tag)

    def once(stream=None):
        if stream is None:
            W, k, s = run(native, W0, tag, U, dead, sp, n, m)
        else:
            with torch.cuda.stream(stream):
                W, k, s = run(native, W0, tag, U, dead, sp, n, m)
            stream.synchronize()
        return bits(W), k.cpu().numpy(), s.item()

    base = once()
    outs = {"again": once(), "stream": once(torch.cuda.Stream())}
    schedule(VLMC_CHOL_LOOKAHEAD=0)
    outs["no_lookahead"] = once()
    schedule(VLMC_CHOL_LOOKAHEAD=1)
    if n == 0:
        schedule(VLMC_OBS_FUSED=0)
        outs["three_pass"] = once()
        schedule(VLMC_OBS_FUSED=1)
    for name, o in outs.items():
        assert np.array_equal(o[0], base[0]), name
        assert np.array_equal(o[1], base[1]), name
        assert o[2] == base[2], name


# ------------------------------------------------------------------------------------------- layer 3
def _guard_setup(tag, sp, n, m):
    R, C = 37, 132
    U, dead = factor(C, 41, dense=True, dead_key=(2,))
    W0 = make_w(R, C, 42, tag)
    return R, C, U, dead, W0


@pytest.mark.gpu
@pytest.mark.parametrize("sp,n,m,fused", [(0.5, 0, 0, "1"), (0.5, 0, 0, "0"), (0.0, 2, 4, None)])
def test_guarded_sweep_with_the_flag_set_leaves_w_and_mask(native, schedule, sp, n, m, fused):
    """A non-zero flag: W (with its sentinel padding) and the keep mask are bit-unchanged.  importance_score is still
    written - vlmc_obs_begin computes it before the flag is read - and equals the unflagged call's.  Then, with the
    scratch of the failed call still in the workspace, a good factor and a zero flag give a fresh sweep's bits."""
    if fused is not None:
        schedule(VLMC_OBS_FUSED=fused)
    tag = "bf16"
    R, C, U, dead, W0 = _guard_setup(tag, sp, n, m)
    Ud, dd = dev_u(U), dev_dead(dead)
    Wf, kf, sf = run(native, W0, tag, U, dead, sp, n, m)             # fresh sweep

    Wb = torch.full((R, C + 4), -7.0, dtype=TAGS[tag], device="cuda")
    W = Wb[:, :C]
    W.copy_(dev_w(W0, tag))
    Kb = torch.full((R, C + 4), 0xA5, dtype=torch.uint8, device="cuda")
    keep = Kb[:, :C].view(torch.bool)
    before_w, before_k = bits(Wb).copy(), Kb.cpu().numpy().copy()
    Ubad = Ud.clone()
    Ubad[5, 5:] = float("nan")                                       # scratch of the failed call is poisoned
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    flag.fill_(1)                                                    # on the sweep's stream, before the call
    _, score = native.obs_sweep(W, Ud, sp, n, m, dead=dd, keep=keep, fail_flag=flag)
    _, score_bad = native.obs_sweep(W, Ubad, sp, n, m, dead=dd, keep=keep, fail_flag=flag)
    torch.cuda.synchronize()
    assert np.array_equal(bits(Wb), before_w)
    assert np.array_equal(Kb.cpu().numpy(), before_k)
    assert score.item() == sf.item()                                 # pinned: the score is written with the flag set
    # damp-and-retry: the good factor, flag cleared
    flag.zero_()
    native.obs_sweep(W, Ud, sp, n, m, dead=dd, keep=keep, fail_flag=flag)
    torch.cuda.synchronize()
    assert np.array_equal(bits(W), bits(Wf))
    assert np.array_equal(Kb[:, :C].cpu().numpy().astype(bool), kf.cpu().numpy())
    assert np.array_equal(bits(Wb)[:, C:], before_w[:, C:])


@pytest.mark.gpu
@pytest.mark.parametrize("sp,n,m", [(0.5, 0, 0), (0.0, 4, 8)])
def test_guarded_sweep_with_a_zero_flag_equals_the_unguarded_call(native, schedule, sp, n, m):
    tag = "f16"
    R, C, U, dead, W0 = _guard_setup(tag, sp, n, m)
    Wa, ka, sa = run(native, W0, tag, U, dead, sp, n, m)
    W = dev_w(W0, tag)
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    kb, sb = native.obs_sweep(W, dev_u(U), sp, n, m, dead=dev_dead(dead), want_mask=True, fail_flag=flag)
    torch.cuda.synchronize()
    assert np.array_equal(bits(W), bits(Wa)) and torch.equal(ka, kb) and sa.item() == sb.item()


@pytest.mark.gpu
@pytest.mark.parametrize("C", [132, 1028])
@pytest.mark.parametrize("sp,n,m", [(0.5, 0, 0), (0.0, 2, 4), (0.0, 8, 16)])
@pytest.mark.parametrize("bounds", [((0, 20), (20, 37)), ((0, 5), (5, 18), (18, 37))])
def test_row_shards_in_lockstep_equal_the_unsharded_sweep(native, schedule, C, sp, n, m, bounds):
    """Two or three uneven row shards driven in lock-step, their block histograms summed between passes (the all-reduce
    across ranks): the unsharded sweep's bits."""
    lib = native.load()
    R, tag = 37, "bf16"
    U, dead = factor(C, 51, dense=True, dead_key=(1, C - 1))
    W0 = make_w(R, C, 52, tag)
    Wfull, kfull, _ = run(native, W0, tag, U, dead, sp, n, m)
    Ud, dd = dev_u(U), dev_dead(dead)
    W = dev_w(W0, tag)
    keep = torch.empty((R, C), dtype=torch.bool, device="cuda")
    nblk = (C + 127) // 128
    st = torch.cuda.current_stream().cuda_stream
    shards = []
    for s, e in bounds:
        ws = torch.zeros(lib.vlmc_workspace_bytes(native.OP_OBS, e - s, C, 128), dtype=torch.uint8, device="cuda")
        hist = torch.zeros((nblk, 3, 2048), dtype=torch.int32, device="cuda")
        shards.append((s, e, ws, hist))
        assert lib.vlmc_obs_begin(W[s:e].data_ptr(), CODES[tag], e - s, C, W.stride(0), Ud.data_ptr(), C,
                                  dd.data_ptr(), None, ws.data_ptr(), ws.numel(), st) == 0
    for blk in range(nblk):
        if n == 0:
            for ps in range(3):
                for s, e, ws, hist in shards:
                    assert lib.vlmc_obs_block_hist(e - s, C, Ud.data_ptr(), C, blk, ps, R, sp, hist.data_ptr(),
                                                   ws.data_ptr(), ws.numel(), st) == 0
                total = sum(h[blk, ps] for *_, h in shards)
                for *_, h in shards:
                    h[blk, ps].copy_(total)
        for s, e, ws, hist in shards:
            assert lib.vlmc_obs_block_finish(W[s:e].data_ptr(), CODES[tag], e - s, C, W.stride(0), Ud.data_ptr(), C,
                                             blk, R, sp, n, m, keep[s:e].data_ptr(), C,
                                             hist.data_ptr() if n == 0 else None, ws.data_ptr(), ws.numel(), st) == 0
    torch.cuda.synchronize()
    assert np.array_equal(bits(W), bits(Wfull)) and torch.equal(keep, kfull)


REJECTIONS = [  # (name, overrides, status)
    ("m=3", dict(n=1, m=3), BAD_ARG), ("m=12", dict(n=1, m=12), BAD_ARG), ("m=32", dict(n=1, m=32), BAD_ARG),
    ("n=m", dict(n=4, m=4), BAD_ARG), ("n>m", dict(n=5, m=4), BAD_ARG),
    ("sp=1", dict(sp=1.0), BAD_ARG), ("sp<0", dict(sp=-0.25), BAD_ARG), ("sp=nan", dict(sp=float("nan")), BAD_ARG),
    ("C%4", dict(C=130), UNSUPPORTED), ("blocksize", dict(bsz=64), UNSUPPORTED), ("ldm<C", dict(ldm=131), BAD_ARG),
    ("U unaligned", dict(uoff=1), UNSUPPORTED), ("ldu%4", dict(ldu=133), UNSUPPORTED),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,over,status", REJECTIONS, ids=[r[0] for r in REJECTIONS])
def test_bad_arguments_are_rejected_before_any_launch(native, name, over, status):
    """The documented status, and W, the keep mask and the importance score (written by the first launch of a
    sweep) all left as they were."""
    lib = native.load()
    R, C = 9, 132
    a = dict(n=0, m=0, sp=0.5, C=C, bsz=128, ldm=C, uoff=0, ldu=C + 4)
    a.update(over)
    Wb = torch.full((R, C + 4), 0.25, dtype=torch.float16, device="cuda")
    Ub = torch.zeros((C + 8) * (C + 8), dtype=torch.float32, device="cuda")
    Ub[:: C + 9] = 1.0
    keep = torch.full((R, C + 4), 0xA5, dtype=torch.uint8, device="cuda")
    score = torch.full((1,), -3.0, device="cuda")
    ws = native.workspace(Wb, lib.vlmc_workspace_bytes(native.OP_OBS, R, C + 4, 128))
    before = (bits(Wb).copy(), keep.cpu().numpy().copy())
    torch.cuda.synchronize()
    for fn in ("vlmc_obs_sweep", "vlmc_obs_sweep_guarded"):
        args = [Wb.data_ptr(), 1, R, a["C"], C + 4, Ub.data_ptr() + 4 * a["uoff"], a["ldu"], None, a["sp"], a["n"],
                a["m"], a["bsz"], keep.data_ptr(), a["ldm"], score.data_ptr()]
        if fn == "vlmc_obs_sweep_guarded":
            args.append(None)
        args += [ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream]
        assert getattr(lib, fn)(*args) == status, fn
    torch.cuda.synchronize()
    assert np.array_equal(bits(Wb), before[0]) and np.array_equal(keep.cpu().numpy(), before[1])
    assert score.item() == -3.0
