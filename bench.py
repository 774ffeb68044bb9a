#!/usr/bin/env python
"""bench.py - seconds per Vicuna-7B block pruned (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--method wanda_nm|wanda_unstructured|sparsegpt|dsnot]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...     # the unmodified reference on the host cores (oracle/ref_arm.py; port fallback)

A "step" prunes ONE Vicuna-7B decoder layer (q,k,v,o 4096x4096; gate,up 11008x4096; down 4096x11008, fp16,
random init) the way the reference's per-layer wrapper API dictates: for each of the 7 linears, calibration
statistics over its 128 x 2048 synthetic fp16 tokens (WrappedGPT.add_batch / SparseGPT.add_batch), then the
mask selection (Wanda 2:4 / unstructured, DSnoT refine) or the Cholesky-inverse + OBS sweep (SparseGPT 50 %).
Block forwards are excluded (activations are the synthetic inputs), SURVEY 8(d).  No de-duplication of the
statistics of linears that share an input: 7 accumulations per block, like the reference.

N > 1 (strong scaling, SURVEY 8e): calibration sequences are split across ranks and ONE all-reduce per statistic
merges them; output rows are split for selection / the OBS sweep and all-gathered; the SparseGPT factorisations
of a block are spread over the ranks and broadcast.

value     device-resident inputs, CUDA-event timed, max over ranks
e2e       the same step through the public wrapper API from PINNED HOST buffers (activations + weights H2D,
          pruned weights + masks D2H inside the timed region)
roofline  the kernel with the largest share of the step, timed live with CUDA events on the launching stream
The default run times --method (wanda_nm) and appends a short measurement of the other methods under "methods".
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "vlm-compression_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

D, FF = 4096, 11008
LINEARS = [  # name, rows, cols, input id
    ("q_proj", D, D, "attn_in"), ("k_proj", D, D, "attn_in"), ("v_proj", D, D, "attn_in"),
    ("o_proj", D, D, "attn_out"), ("gate_proj", FF, D, "mlp_in"), ("up_proj", FF, D, "mlp_in"),
    ("down_proj", D, FF, "mlp_mid"),
]
INPUT_DIMS = {"attn_in": D, "attn_out": D, "mlp_in": D, "mlp_mid": FF}
N_SEQ, SEQ_LEN = 128, 2048
METHODS = ["wanda_nm", "wanda_unstructured", "sparsegpt", "dsnot", "dsnot_elided", "wanda_nm_shared", "sparsegpt_shared"]
METRIC, UNIT = "s_per_vicuna7b_block_pruned", "s/block"
WORKLOAD = {
    "wanda_nm": "Wanda 2:4", "wanda_unstructured": "Wanda 50% unstructured (per-row)",
    "sparsegpt": "SparseGPT 50% unstructured (blocksize 128, percdamp 0.01)",
    "dsnot": "Wanda-initialised DSnoT refine at 60% (reference semantics, swap loop executed)",
    "dsnot_elided": "Wanda-initialised DSnoT at 60% (reference semantics; the self-cancelling swap loop elided: same masks)",
    "wanda_nm_shared": "Wanda 2:4, statistics of linears fed by the same activations (q/k/v, gate/up) accumulated once "
                       "(4 accumulations per block instead of 7; same masks)",
    "sparsegpt_shared": "SparseGPT 50% unstructured (blocksize 128, percdamp 0.01), Hessians of linears fed by the same "
                        "activations accumulated and factorised once (4 per block instead of 7; same weights)",
}


def stat_groups(shared):
    """[(leader linear, [member linears])]: per linear like the reference's hooks, or one group per distinct input."""
    if not shared:
        return [(n, [n]) for n, *_ in LINEARS]
    by_inp = {}
    for n, _, _, inp in LINEARS:
        by_inp.setdefault(inp, []).append(n)
    return [(m[0], m) for m in by_inp.values()]


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return {"hbm": float(d["hbm_gbs"]), "tensor": float(d["bf16_tflops"]),
                "tensor_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm": 6650.0, "tensor": 1650.0, "tensor_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


def measure_tf32_peak(torch, dev, n=8192, reps=5):
    """SURVEY 8(d): "TF32 peak not yet measured - the builder must measure it".  torch.matmul of two fp32 n^3 matrices
    with allow_tf32 (cuBLAS TF32 tensor-core GEMM), best of `reps`, CUDA events: dense TF32 TFLOP/s of THIS GPU, the
    denominator for the 3xTF32 GEMMs of K10 / K13 (executed flop = 3 x logical)."""
    prev = torch.backends.cuda.matmul.allow_tf32
    try:
        torch.backends.cuda.matmul.allow_tf32 = True
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        c = torch.empty(n, n, device=dev)
        torch.matmul(a, b, out=c)
        torch.cuda.synchronize()
        best = None
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b, out=c)
            e1.record()
            torch.cuda.synchronize()
            t = e0.elapsed_time(e1)
            best = t if best is None or t < best else best
        del a, b, c
        return 2.0 * n ** 3 / best / 1e9
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


class ClockSampler:
    """SM clock and throttle reasons sampled through NVML DURING the timed region (a few ms period)."""

    def __init__(self, index):
        self.index, self.sm, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thread = None
        self._nvml = self._handle = None
        try:        # NVML is initialised HERE (~10 ms), not inside the timed region; start() only starts the thread
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and vis.split(",")[0].isdigit() else self.index
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._handle, pynvml.NVML_CLOCK_SM)
            self._nvml = pynvml
        except Exception as e:  # noqa: BLE001
            self.reasons.add(f"nvml unavailable: {type(e).__name__}")

    def start(self):
        if self._nvml is None:
            return
        pynvml, h = self._nvml, self._handle
        names = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

        def loop():
            while not self._stop.is_set():
                try:
                    self.sm.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                    r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for n, bit in names.items():
                        if r & bit:
                            self.reasons.add(n)
                except Exception:  # noqa: BLE001
                    pass
                time.sleep(0.002)
        self._thread = threading.Thread(target=loop, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=1.0)
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ GPU arm
def make_block(torch, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    return {name: (torch.randn(r, c, device=dev, generator=g) * 0.02).half() for name, r, c, _ in LINEARS}


def make_inputs(torch, dev, n_seq, seed):
    """Synthetic calibration activations [n_seq, SEQ_LEN, C] fp16: N(0,1) * per-channel gain + offset (SURVEY 8d)."""
    out = {}
    for i, (name, C) in enumerate(INPUT_DIMS.items()):
        g = torch.Generator(device=dev).manual_seed(seed + i)
        gain = torch.exp(torch.rand(C, device=dev, generator=g) * 2.77 - 1.386)
        off = torch.randn(C, device=dev, generator=g) * 0.3
        x = torch.empty(n_seq, SEQ_LEN, C, device=dev, dtype=torch.float16)
        for j in range(n_seq):  # chunked: never materialise the fp32 copy of the whole set
            x[j] = (torch.randn(SEQ_LEN, C, device=dev, generator=g) * gain + off).half()
        out[name] = x
    return out


class Ctx:
    """Everything a step needs: torch, the bindings, rank / world, persistent device buffers."""

    def __init__(self, torch, native, parallel, dev, rank, world, calib_batch):
        from vlmc import schedule
        self.torch, self.native, self.parallel, self.schedule = torch, native, parallel, schedule
        self.dev, self.rank, self.world, self.calib_batch = dev, rank, world, calib_batch
        self.events = None          # list of (tag, start, end, work) when kernel timing is on
        self.launches = 0
        self.H = self.U = None

    def timed(self, tag, work, fn):
        if self.events is None:
            return fn()
        a, b = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
        a.record()
        r = fn()
        b.record()
        self.events.append((tag, a, b, work))
        return r

    def sparsegpt_buffers(self):
        if self.H is None:
            t = self.torch
            self.H = {n: t.empty(c, c, device=self.dev) for n, _, c, _ in LINEARS}
            self.U = {n: t.empty(c, c, device=self.dev) for n, _, c, _ in LINEARS}
        return self.H, self.U


def accumulate(ctx, fn, x, state, work_per_seq, tag):
    """Statistics of one linear over this rank's sequences.  One rank: running mean, calib_batch sequences per
    add_batch call.  Several ranks: raw partial sums with the global divisor, merged by the caller."""
    n_local = x.shape[0]
    if ctx.world > 1:
        ctx.timed(tag, work_per_seq * n_local, lambda: fn(x, state, 0, N_SEQ))
        ctx.launches += 1
        return
    n = 0
    for j in range(0, n_local, ctx.calib_batch):
        xb = x[j:j + ctx.calib_batch]
        ctx.timed(tag, work_per_seq * xb.shape[0], lambda xb=xb, n=n: fn(xb, state, n, xb.shape[0]))
        n += xb.shape[0]
        ctx.launches += 1


class _NoFork:
    """Same interface as vlmc.schedule.Fork, everything on the current stream."""

    def __enter__(self):
        return self

    def stream(self, i):
        import contextlib
        return contextlib.nullcontext()

    def __exit__(self, *exc):
        return False


def schedule_fork(ctx, n):
    return ctx.schedule.Fork(ctx.dev, n) if n > 1 else _NoFork()


def step_wanda(ctx, weights, inputs, method, shared=False):
    torch, native, parallel = ctx.torch, ctx.native, ctx.parallel
    shape = {n: (R, C, inp) for n, R, C, inp in LINEARS}
    scalers = {}
    groups = stat_groups(shared)
    # the scaler_rows of the block are views of ONE packed fp32 buffer: one memset, and on several GPUs one in-place
    # all-reduce (no gather / scatter copies around the collective)
    flat = torch.zeros(sum(shape[l][1] for l, _ in groups), device=ctx.dev, dtype=torch.float32)
    off = 0
    # phase 1: statistics (per-linear API unless `shared`).  The accumulations are independent of each other: they
    # alternate between two streams so that the ramp-up of one launch covers the drain + finalize of the previous one
    # (each stream has its own scratch).  Per-span events (eager pass only) need the launches on one stream.
    nstreams = 1 if ctx.events is not None else 2
    # ONE multi-tensor launch for the statistics of the block (vlmc_sqnorm_accum_batch): one ramp-up and one drain instead of
    # seven.  Several GPUs: a rank's share of a linear is a 40-100 us launch.  One GPU (r02): 2.92 -> 2.68-2.71 ms per block
    # (18.66 GB in 2.55 ms = 7.3 TB/s; a 0.33 ms launch at C = 4096 loses ~6 % to its own ramp and drain, A/B on one box).
    # VLMC_BENCH_STATS_BATCH=0 restores one launch per linear on two alternating streams; the calibration-batch sweep
    # (calib_batch < 128: several add_batch calls per linear) always uses per-linear launches.
    batch_stats = ctx.world > 1 or (ctx.calib_batch >= N_SEQ and os.environ.get("VLMC_BENCH_STATS_BATCH") != "0")
    if batch_stats:
        # Partial sums carry the divisor of the whole set (0, N_SEQ) on several GPUs.
        xs, ss = [], []
        for leader, members in groups:
            _, C, inp = shape[leader]
            sl = flat[off:off + C]
            off += C
            xs.append(inputs[inp])
            ss.append(sl)
            for m in members:
                scalers[m] = sl
        n_local = xs[0].shape[0]
        nb, bb = (0, N_SEQ) if ctx.world > 1 else (0, n_local)
        ctx.timed("sqnorm_accum", sum(x.numel() * 2 for x in xs), lambda: native.sqnorm_accum_batch(xs, ss, nb, bb))
        ctx.launches += 1
    with schedule_fork(ctx, nstreams) as fk:
        for gi, (leader, members) in enumerate(groups if not batch_stats else []):
            _, C, inp = shape[leader]
            s = flat[off:off + C]
            off += C
            with fk.stream(gi):
                accumulate(ctx, native.sqnorm_accum, inputs[inp], s, SEQ_LEN * C * 2, "sqnorm_accum")
            for m in members:
                scalers[m] = s
    if ctx.world > 1:
        parallel.allreduce_sum(flat)
    masks = {}
    if method == "wanda_nm":
        # phase 2, n:m: a group decision needs its m scores and nothing else, and the pruned weights + masks must end
        # up on EVERY rank anyway (5 B/weight to rewrite the replica) - exactly the traffic of running the selection
        # itself.  So every rank selects on its whole replica: no row split, no exchange, identical results.
        # ... and all 7 linears go through ONE launch (vlmc_wanda_nm_batch): one ramp-up and one drain per block.
        names = [n for n, *_ in LINEARS]
        keeps, _ = ctx.timed("wanda_select", sum(R * C for _, R, C, _ in LINEARS) * 5, lambda: native.wanda_nm_batch(
            [weights[n] for n in names], [scalers[n] for n in names], 2, 4))
        ctx.launches += 2
        return dict(zip(names, keeps))
    if ctx.world > 1 and all(R % ctx.world == 0 for _, R, _, _ in LINEARS):
        # phase 2, per-row top-k, sharded: select on this rank's rows, ONE all-gather of the bit-packed masks of all 7
        # linears, the other rows of the replicated weights are zeroed locally from the received bits
        def make_sel(name, C):
            return lambda Wr, keep: native.wanda_rowselect(Wr, scalers[name], int(C * 0.5), keep_mask=keep)[1]
        names = [n for n, *_ in LINEARS]
        total = sum(R * C for _, R, C, _ in LINEARS)
        def sel_batch(Wrs, keeps_r):        # the row shards of all linears in one call (one launch per distinct row length)
            return native.wanda_rowselect_batch(Wrs, [scalers[n] for n in names], [int(C * 0.5) for _, _, C, _ in LINEARS],
                                                keep_masks=keeps_r)[1]
        batch = sel_batch if os.environ.get("VLMC_BENCH_SELECT_BATCH") != "0" else None
        res = ctx.timed("wanda_select", total * 5, lambda: parallel.prune_block_rows_packed(
            [weights[n] for n in names], [make_sel(n, C) for n, _, C, _ in LINEARS], native.mask_pack,
            lambda W, bits, keep, rps, stride: native.mask_apply_packed(W, bits, keep, True, rps, stride),
            ctx.rank, ctx.world, select_batch_fn=batch, pack_batch_fn=native.mask_pack_batch if batch else None,
            apply_batch_fn=(lambda Ws, bits, keeps, rps, stride: native.mask_apply_packed_batch(
                Ws, bits, keeps, True, rps, stride)) if batch else None))
        ctx.launches += 5 if batch else 7 * 3
        return {n: k for n, (k, _) in zip(names, res)}
    if ctx.world == 1:
        # phase 2, per-row top-k on one GPU: one launch per linear (the reference's per-linear API), longest first, dealt
        # over a few streams: a warp owns whole rows (1-5 per launch), so the tail of one launch - warps that got one row
        # fewer - is filled by the next linear's rows instead of idling.  Masks are allocated on the caller's stream.
        nsel = 1 if ctx.events is not None else max(1, int(os.environ.get("VLMC_BENCH_SELECT_STREAMS", "3")))
        keeps = {name: torch.empty((R, C), dtype=torch.bool, device=ctx.dev) for name, R, C, _ in LINEARS}
        if os.environ.get("VLMC_BENCH_SELECT_BATCH") != "0":
            # ONE call for the block (vlmc_wanda_rowselect_batch): the linears of equal row length share a launch whose CTAs
            # walk the concatenated rows - 2 launches instead of 7, 25-30 rows per CTA instead of 5.  Same masks and weights.
            names = [n for n, *_ in LINEARS]
            ctx.timed("wanda_select", sum(R * C for _, R, C, _ in LINEARS) * 5, lambda: native.wanda_rowselect_batch(
                [weights[n] for n in names], [scalers[n] for n in names], [int(C * 0.5) for _, _, C, _ in LINEARS],
                keep_masks=[keeps[n] for n in names]))
            ctx.launches += 3
            return keeps
        with schedule_fork(ctx, nsel) as fk:
            for i, (name, R, C, _) in enumerate(sorted(LINEARS, key=lambda l: -l[1] * l[2])):
                with fk.stream(i):
                    ctx.timed("wanda_select", R * C * 5, lambda: native.wanda_rowselect(
                        weights[name], scalers[name], int(C * 0.5), keep_mask=keeps[name]))
                ctx.launches += 2
        return keeps
    for name, R, C, _ in LINEARS:                         # phase 2: score + select + apply on this rank's rows
        def sel(Wr, s, keep, C=C):
            return native.wanda_rowselect(Wr, s, int(C * 0.5), keep_mask=keep)[1]
        masks[name], _ = ctx.timed("wanda_select", R * C * 5 // ctx.world, lambda: parallel.prune_linear_row_sharded(
            weights[name], scalers[name], sel, ctx.rank, ctx.world))
        ctx.launches += 2
    return masks


def step_dsnot(ctx, weights, inputs, elide=False):
    torch, native, parallel = ctx.torch, ctx.native, ctx.parallel
    stats = {}
    # one stream: two concurrent DSnoT statistics kernels (256-byte row segments, multi-wave grids) ran 50 % SLOWER than
    # one after the other (measured), unlike the Wanda statistics in step_wanda
    if os.environ.get("VLMC_BENCH_STATS_BATCH") != "0":
        # ONE launch for the 7 wrappers (vlmc_dsnot_stats_batch, r02): per item the plan and the results of vlmc_dsnot_stats;
        # the grid walks the calls with the linears interleaved, so q / k / v (gate / up) read a call's activations at
        # the same time and the repeats hit in L2
        xs = []
        for name, R, C, inp in LINEARS:
            stats[name] = [torch.zeros(C, device=ctx.dev) for _ in range(4)]   # scaler_row, sum_metric_row, mean, var
            xs.append(inputs[inp])
        n_local = xs[0].shape[0]
        ctx.timed("dsnot_stats", sum(x.numel() * 2 for x in xs), lambda: native.dsnot_stats_batch(
            xs, [stats[name] for name, *_ in LINEARS], 0, 1, 0, nseg=n_local))
        ctx.launches += 1
    with schedule_fork(ctx, 1) as fk:
        for li, (name, R, C, inp) in enumerate(LINEARS if not stats else []):
            st = [torch.zeros(C, device=ctx.dev) for _ in range(4)]       # scaler_row, sum_metric_row, mean, var
            x = inputs[inp]
            n_local = x.shape[0]
            # every sequence is one reference add_batch call (nseg segments): var is a mean of per-call variances
            with fk.stream(li):
                ctx.timed("dsnot_stats", x.numel() * 2, lambda: native.dsnot_stats(x, st[0], st[1], st[2], st[3], 0, 1, 0,
                                                                                   nseg=n_local))
            ctx.launches += 1
            stats[name] = st
    if ctx.world > 1:
        n_local = next(iter(inputs.values())).shape[0]
        parallel.merge_running_means([t for st in stats.values() for t in st], n_local, n_total=N_SEQ)
    masks = {}
    # one GPU: the per-linear launches are dealt over a few streams, longest first (see step_wanda); several GPUs: one
    # after the other, each followed by its mask exchange
    nref = 1
    if ctx.world == 1 and ctx.events is None:
        nref = max(1, int(os.environ.get("VLMC_BENCH_SELECT_STREAMS" if elide else "VLMC_BENCH_REFINE_STREAMS", "3")))
    order = sorted(LINEARS, key=lambda l: -l[1] * l[2]) if nref > 1 else LINEARS
    keeps = {name: torch.empty((R, C), dtype=torch.bool, device=ctx.dev) for name, R, C, _ in LINEARS}
    if elide and os.environ.get("VLMC_BENCH_SELECT_BATCH") != "0" and all(R % ctx.world == 0 for _, R, _, _ in LINEARS):
        # shipped semantics (the mask is the initial selection): the block's selections as ONE batched call, like step_wanda
        names = [n for n, *_ in LINEARS]
        ks = [round(C * 0.6) for _, _, C, _ in LINEARS]
        total = sum(R * C for _, R, C, _ in LINEARS)
        if ctx.world == 1:
            ctx.timed("wanda_select", total * 5, lambda: native.wanda_rowselect_batch(
                [weights[n] for n in names], [stats[n][0] for n in names], ks, keep_masks=[keeps[n] for n in names]))
            ctx.launches += 3
            return keeps
        res = ctx.timed("wanda_select", total * 5, lambda: parallel.prune_block_rows_packed(
            [weights[n] for n in names], [None] * len(names), native.mask_pack, None, ctx.rank, ctx.world,
            select_batch_fn=lambda Wrs, kr: native.wanda_rowselect_batch(Wrs, [stats[n][0] for n in names], ks, keep_masks=kr)[1],
            pack_batch_fn=native.mask_pack_batch,
            apply_batch_fn=lambda Ws, bits, kp, rps, stride: native.mask_apply_packed_batch(Ws, bits, kp, True, rps, stride)))
        ctx.launches += 5
        return {n: k for n, (k, _) in zip(names, res)}
    with schedule_fork(ctx, nref) as fk:
        for li, (name, R, C, _) in enumerate(order):
            W = weights[name]
            s, e = parallel.row_range(R, ctx.rank, ctx.world)
            keep = keeps[name]
            st = stats[name]
            with fk.stream(li):
                if elide:      # shipped semantics: the swaps are written back (SURVEY F4), the mask is the initial selection
                    ctx.timed("wanda_select", (e - s) * C * 5, lambda: native.wanda_rowselect(
                        W[s:e], st[0], round(C * 0.6), keep_mask=keep[s:e]))
                else:
                    ctx.timed("dsnot_refine", (e - s) * C * 7, lambda: native.dsnot_refine(
                        W[s:e], st[0], st[1], st[3], round(C * 0.6), keep_mask=keep[s:e],
                        reduce_ncycles=parallel.allreduce_max if ctx.world > 1 else None))
            ctx.launches += 2
            if ctx.world > 1:      # masks travel as bits; the replicated weights are zeroed locally
                parallel.exchange_rows_packed(
                    W, keep, native.mask_pack,
                    lambda Wf, bits, kp, rps, stride: native.mask_apply_packed(Wf, bits, kp, True, rps, stride),
                    ctx.rank, ctx.world)
            masks[name] = keep
    return masks


def step_sparsegpt(ctx, weights, inputs, shared=False):
    """Phase 1: H = (2/N) sum X^T X on the tensor cores (tokens split over ranks, SUM all-reduce).
    Phase 2 + 3: the factorisation and the OBS sweep of a linear are sequential chains of small kernels, independent
    between linears: on one GPU they run concurrently, one stream per chain (vlmc.schedule); on several GPUs WHOLE
    linears are spread over the ranks (longest chain first), each rank runs its chains concurrently and the pruned
    weights are broadcast from their owners - no per-column-block exchange, no broadcast of U."""
    torch, native, parallel, schedule = ctx.torch, ctx.native, ctx.parallel, ctx.schedule
    H, U = ctx.sparsegpt_buffers()
    shape = {n: (R, C, inp) for n, R, C, inp in LINEARS}
    Hof = {}
    for leader, members in stat_groups(shared):
        _, C, inp = shape[leader]
        accumulate(ctx, native.hessian_accum, inputs[inp], H[leader], 2.0 * SEQ_LEN * C * C, "hessian_accum")
        if ctx.world > 1:
            parallel.allreduce_sum(H[leader])
        for m in members:
            Hof[m] = leader
    names = [n for n, *_ in LINEARS]

    def run(indices):
        mine = [names[i] for i in indices]
        leaders = list(dict.fromkeys(Hof[n] for n in mine))
        flop = sum(2.0 / 3.0 * shape[l][1] ** 3 for l in leaders) + sum(float(shape[n][0]) * shape[n][1] ** 2 for n in mine)
        ctx.timed("sparsegpt_chains", flop, lambda: schedule.sparsegpt_block(
            [(weights[n], H[Hof[n]], 0.5, 0, 0) for n in mine], 0.01, 128, [U[l] for l in leaders]))
        ctx.launches += len(leaders) + sum(5 * ((shape[n][1] + 127) // 128) for n in mine)
    parallel.prune_linears_task_parallel([weights[n] for n in names], run, ctx.rank, ctx.world)
    return None


def run_step(ctx, method, weights, inputs):
    shared = method.endswith("_shared")
    if shared:
        method = method[:-len("_shared")]
    if method == "sparsegpt":
        return step_sparsegpt(ctx, weights, inputs, shared)
    if method in ("dsnot", "dsnot_elided"):
        return step_dsnot(ctx, weights, inputs, elide=method == "dsnot_elided")
    return step_wanda(ctx, weights, inputs, method, shared)


GRAPH_METHODS = ("wanda_nm", "wanda_unstructured", "dsnot", "dsnot_elided", "wanda_nm_shared")   # no host round trip inside the step (SparseGPT's
                                                                # conditional damping reads a status word)


DUMP_ROWS = 128     # rows per linear in --dump-outputs: the 7 weights + masks of a block in 35 MB
DUMP_SEED = 200     # weight set of the last timed step of either pass when outputs are kept: same inputs in both passes


def sample_outputs(torch, weights, masks):
    """{file name: float32 array} of what a caller of one step receives: every pruned weight and, for the methods that
    return them, the keep masks, each cut to the same DUMP_ROWS rows (a fixed seeded choice per linear)."""
    import numpy as np
    out = {}
    for li, (name, R, _, _) in enumerate(LINEARS):
        W = weights[name]
        rows = torch.from_numpy(np.sort(np.random.default_rng(li).choice(R, DUMP_ROWS, replace=False))).to(W.device)
        out[f"{name}.weight"] = W.index_select(0, rows).float().cpu().numpy()
        if masks:
            out[f"{name}.mask"] = masks[name].index_select(0, rows).float().cpu().numpy()
    return out


def time_method(ctx, method, inputs, steps, warmup, sample_clocks, dist, use_graph=True, keep_outputs=False):
    """W untimed + K timed steps of one method, a fresh weight set per step.

    Pass A (eager launches): per-span CUDA events -> the kernel shares behind `roofline`.
    Pass B (Wanda / DSnoT, unless --no-graph): the K timed steps (each on its own weight set) captured into ONE CUDA
    graph (kernels + NCCL collectives) and replayed once inside the timed region: neither the Python launch overhead
    (~100 small launches per 3 ms step) nor the host's graph-launch latency between steps (0.15-0.2 ms, measured)
    sits between the steps.  The headline is the faster of the two passes (both time exactly K steps on the device, max over ranks).
    keep_outputs: the last timed step of each pass prunes a fresh weight set of seed DUMP_SEED, and out["outputs"] holds
    sample_outputs() of that step in the pass behind the headline (out["outputs_pass"]), taken after both passes.
    Returns dict(ms_per_step, launches, kernels, ...)."""
    torch = ctx.torch
    nsets = min(steps + warmup, 24)
    wsets = [make_block(torch, ctx.dev, seed=s) for s in range(nsets)]

    def barrier():
        if ctx.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    step_ms = []

    def timed_loop(step_fn):
        for i in range(warmup):
            step_fn(i)
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        marks = [t0]
        t0.record()
        for i in range(steps):
            step_fn(warmup + i)
            if i + 1 < steps:                # step boundaries (diagnostic: one stalled step shows up in step_ms)
                marks.append(torch.cuda.Event(enable_timing=True))
                marks[-1].record()
        t1.record()
        marks.append(t1)
        barrier()
        step_ms.clear()
        step_ms.extend(round(a.elapsed_time(b), 3) for a, b in zip(marks[:-1], marks[1:]))
        ms = torch.tensor([t0.elapsed_time(t1)], device=ctx.dev)
        if ctx.world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / steps

    # ---- pass A: eager, with per-span events on the launching stream
    sampler = ClockSampler(ctx.dev.index)
    ctx.events = None
    last = {}                                # pass -> (weights, masks) of its last timed step, with keep_outputs
    wlast = make_block(torch, ctx.dev, seed=DUMP_SEED) if keep_outputs else None

    def eager_step(i):
        if i == warmup:                      # the timed region starts here
            ctx.events, ctx.launches = [], 0
            if sample_clocks:
                sampler.start()
        w = wlast if wlast is not None and i == warmup + steps - 1 else wsets[i % nsets]
        masks = run_step(ctx, method, w, inputs)
        if w is wlast:
            last["eager"] = (w, masks)
    eager_ms = timed_loop(eager_step)
    clocks = sampler.stop() if sample_clocks else None
    kern = {}
    for tag, a, b, work in ctx.events:
        k = kern.setdefault(tag, {"ms": 0.0, "work": 0.0, "spans": 0})
        k["ms"] += a.elapsed_time(b)
        k["work"] += work
        k["spans"] += 1
    ctx.events = None
    out = {"ms_per_step": eager_ms, "eager_ms_per_step": eager_ms, "launches": ctx.launches, "kernels": kern, "method": method,
           "clocks": clocks, "steps": steps, "cuda_graph": False, "weight_sets": nsets, "world": ctx.world,
           "calib_batch": ctx.calib_batch, "shared": method.endswith("_shared"), "eager_step_ms": list(step_ms)}

    # ---- pass B: ONE CUDA graph holding the K timed steps
    if use_graph and method in GRAPH_METHODS:
        try:
            del wsets
            torch.cuda.empty_cache()
            nsets = min(steps, 24)
            wsets = [make_block(torch, ctx.dev, seed=100 + s) for s in range(nsets)]
            wlast = make_block(torch, ctx.dev, seed=DUMP_SEED) if keep_outputs else None
            barrier()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for i in range(steps):
                    w = wlast if wlast is not None and i == steps - 1 else wsets[i % nsets]
                    masks = run_step(ctx, method, w, inputs)
            barrier()
            # warm-up: whole replays (K >= 1 steps each, at least W steps in all; the first one also uploads the graph to
            # the device), then the weights the warm replays pruned are restored (the selection kernels are data dependent)
            for _ in range(max(1, -(-warmup // steps))):
                g.replay()
            restore = [(100 + si, w) for si, w in enumerate(wsets)]
            if wlast is not None:
                restore.append((DUMP_SEED, wlast))
            for seed, w in restore:
                for name, t in make_block(torch, ctx.dev, seed=seed).items():
                    w[name].copy_(t)
            barrier()
            sampler = ClockSampler(ctx.dev.index)
            if sample_clocks:
                sampler.start()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            g.replay()                       # exactly K steps, one launch: no host work between the steps
            t1.record()
            barrier()
            ms = torch.tensor([t0.elapsed_time(t1)], device=ctx.dev)
            if ctx.world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            graph_ms = float(ms.item()) / steps
            out["graph_ms_per_step"] = graph_ms
            gclocks = sampler.stop() if sample_clocks else None
            if keep_outputs:
                last["graph"] = (wlast, masks)
            del masks, wlast
            # both passes time exactly K steps on the device, max over ranks; the headline is the faster way of launching
            # the same work (at 8 GPUs the replay of a graph that holds NCCL collectives measured SLOWER than eager launches)
            if graph_ms <= out["ms_per_step"]:
                out["ms_per_step"] = graph_ms
                out["cuda_graph"] = True
                out["weight_sets"] = nsets
                if sample_clocks:
                    out["clocks"] = gclocks
            del g
        except Exception as e:  # noqa: BLE001  (capture unsupported somewhere: the eager number stands)
            out["cuda_graph_error"] = f"{type(e).__name__}: {e}"[:200]
            torch.cuda.synchronize()
    if keep_outputs:
        out["outputs_pass"] = "graph" if out["cuda_graph"] else "eager"
        out["outputs"] = sample_outputs(torch, *last[out["outputs_pass"]])
    del wsets, last
    torch.cuda.empty_cache()
    return out


def ncu_traffic(tag, res):
    """DRAM bytes (read + write) of the span `tag` per step, from the committed ncu capture of the same bench command
    (profiles/ncu_traffic.json, written by scripts/ncu_traffic.py from `ncu --metrics dram__bytes_read.sum,
    dram__bytes_write.sum`), divided by the spans per step: per launch like `achieved`.  None when no capture matches the
    timed configuration (several GPUs, another calibration batch)."""
    if res.get("world", 1) != 1 or res.get("calib_batch") != N_SEQ:
        return None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            cap = json.load(f)
        method = res.get("method", "")
        per_step = cap["per_step_bytes"][method][tag]
        spans_per_step = res["kernels"][tag]["spans"] / max(res["steps"], 1)
        return per_step / max(spans_per_step, 1)
    except (OSError, KeyError, ValueError, TypeError):
        return None


def roofline_of(res, pk):
    """The span with the largest share of the step -> roofline object (HBM GB/s or tensor TFLOP/s)."""
    total = res["eager_ms_per_step"] * res["steps"]      # spans were timed in the eager pass
    tag, k = max(res["kernels"].items(), key=lambda kv: kv[1]["ms"])
    info = {
        "sqnorm_accum": ("hbm", "colstats_batch_kernel<half,0> (vlmc_sqnorm_accum_batch: the block's statistics in one launch) / "
                                "colstats_kernel<half,0> (vlmc_sqnorm_accum): T*C*2 B per tensor"),
        "dsnot_stats": ("hbm", "colstats_batch_kernel<half,1> (vlmc_dsnot_stats_batch: the block's 7 wrappers in one launch) / "
                               "colstats_kernel<half,1> (vlmc_dsnot_stats): T*C*2 B per tensor"),
        "wanda_select": ("hbm", "nm_batch_kernel (all linears of the block in one launch) / rowselect_cta_kernel: 5 B per weight"),
        "dsnot_refine": ("hbm", "dsnot_walk2_kernel + dsnot_apply_kernel: 7 B per weight (latency / issue-bound, see DESIGN.md)"),
        "hessian_accum": ("tensor", "hessian_syrk_kernel (vlmc_hessian_accum): 2*T*C^2 logical flop per call (SYRK executes half)"),
        "chol_inv_upper": ("tensor", "blocked Cholesky + triangular inverse (3xTF32 tcgen05 GEMMs, the chains of the block run concurrently): 2/3 C^3 flop per Hessian"),
        "sparsegpt_chains": ("tensor", "factorisation (blocked Cholesky + triangular inverse) and OBS sweep chains of the block, pipelined "
                                       "per Hessian on concurrent streams (3xTF32 tcgen05 GEMMs): 2/3 C^3 + R*C^2 flop"),
        "obs_sweep": ("tensor", "OBS block sweeps + trailing 3xTF32 tcgen05 GEMMs (the chains of the block run concurrently): R*C^2 flop per linear"),
    }[tag]
    bound, desc = info
    if bound == "hbm":
        achieved = k["work"] / (k["ms"] * 1e-3) / 1e9
        peak, unit = pk["hbm"], "GB/s"
    else:
        achieved = k["work"] / (k["ms"] * 1e-3) / 1e12
        peak, unit = pk["tensor"], "TFLOP/s"
    out = {"bound": bound, "kernel": desc, "achieved": achieved, "peak": peak, "peak_source": pk["source"],
           "unit": unit, "frac": achieved / peak if achieved else None, "traffic": ncu_traffic(tag, res), "spans": k["spans"],
           "avg_span_ms": k["ms"] / max(k["spans"], 1), "share_of_step": k["ms"] / total,
           "spans_ms_per_step": {t: v["ms"] / res["steps"] for t, v in res["kernels"].items()}}
    if bound == "hbm" and out["traffic"] and k["spans"]:
        alg = k["work"] / k["spans"]                     # algorithmic bytes per launch
        out["traffic_over_algorithmic"] = out["traffic"] / alg
        out["dram_achieved"] = out["traffic"] / (out["avg_span_ms"] * 1e-3) / 1e9       # GB/s that actually crossed the HBM interface
    batched = os.environ.get("VLMC_BENCH_STATS_BATCH") != "0" and (res.get("world", 1) > 1 or res.get("calib_batch", 0) >= N_SEQ)
    if bound == "hbm" and tag in ("sqnorm_accum", "dsnot_stats") and not res.get("shared") and batched:
        # SURVEY 8(d): "18.66 GB per-linear, 12.21 GB if the 4 distinct inputs are de-duplicated - report which".  The block's
        # statistics are ONE launch in which the linears fed the same activations (q / k / v, gate / up) read them at the same
        # time, so the repeats hit in L2 and DRAM sees the distinct tensors only (`traffic`, when a capture matches).  `achieved` /
        # `frac` are therefore quoted on the DISTINCT bytes (what the memory system has to deliver); the per-linear figure is
        # kept beside them.
        dims = {}
        for _, _, C, inp in LINEARS:
            dims[inp] = C
        frac_distinct = sum(dims.values()) / float(sum(C for _, _, C, _ in LINEARS))
        out["achieved_per_linear_bytes"] = achieved
        out["frac_per_linear_bytes"] = achieved / peak
        out["achieved"] = achieved * frac_distinct
        out["frac"] = achieved * frac_distinct / peak
        out["bytes_basis"] = ("distinct activation tensors of the block (12.21 of the 18.66 GB per-linear bytes at 1 GPU); "
                              "`*_per_linear_bytes` count every linear's read; `dram_achieved` = measured DRAM traffic / time")
        if out.get("traffic") and k["spans"]:
            out["traffic_over_algorithmic"] = out["traffic"] / (k["work"] / k["spans"] * frac_distinct)
    if tag == "hessian_accum":
        # the SYRK executes the upper 256 x 256 tiles only: executed flop next to the logical (full-square) figure
        ex = 0.0
        for _, _, C, _ in LINEARS:
            nt = (C + 255) // 256
            ex += 2.0 * N_SEQ * SEQ_LEN * (nt * (nt + 1) // 2) * 256.0 * 256.0
        logical = sum(2.0 * N_SEQ * SEQ_LEN * C * C for _, _, C, _ in LINEARS)
        out["executed_tflops"] = achieved * ex / logical
        out["executed_frac_of_peak"] = out["executed_tflops"] / peak
        out["note"] = "achieved = LOGICAL flop (full square, SURVEY 8d); the SYRK executes the upper tiles only: executed_tflops"
    if tag in ("sparsegpt_chains", "chol_inv_upper", "obs_sweep") and pk.get("tf32"):
        # 3xTF32: three tensor-core MMAs per logical product; quoted against the TF32 peak measured on this GPU
        out["executed_tf32_tflops"] = 3.0 * achieved
        out["tf32_peak_measured"] = pk["tf32"]
        out["executed_frac_of_tf32_peak"] = 3.0 * achieved / pk["tf32"]
    return out


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from vlmc import native, parallel
    native.load()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    s0, s1 = parallel.sample_range(N_SEQ, rank, world)
    inputs = make_inputs(torch, dev, s1 - s0, seed=1000 + 17 * rank)
    ctx = Ctx(torch, native, parallel, dev, rank, world, args.calib_batch)
    if args.one_step:
        # for `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum` (scripts/ncu_traffic.py): exactly one eager step
        # of --method on a fresh weight set, nothing else; never a bench value
        w = make_block(torch, dev, seed=0)
        torch.cuda.synchronize()
        run_step(ctx, args.method, w, inputs)
        torch.cuda.synchronize()
        print(json.dumps({"one_step": args.method}), flush=True)
        return

    main = time_method(ctx, args.method, inputs, args.steps, args.warmup, rank == 0, dist, not args.no_graph,
                       keep_outputs=args.dump_outputs is not None)
    if args.dump_outputs is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in main.pop("outputs").items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    others = {}
    if args.all_methods:
        for m in METHODS:
            if m != args.method:
                # the millisecond methods get enough steps to average out rank skew; SparseGPT steps are ~0.1 s each
                r = time_method(ctx, m, inputs, 3 if m.startswith("sparsegpt") else 10, 3, rank == 0, dist, not args.no_graph)
                others[m] = r
    # VERDICT r1 weak #5: the headline hands all 128 sequences to ONE add_batch per linear; the reference's hooks call once
    # per sequence and vlmc's driver once per chunk of 16 stacked sequences (layerwise.stack_calibration).  Same step,
    # eager launches (hooks cannot be graph-captured), for both.
    calib = {}
    if args.all_methods and world == 1:
        for cb in (1, 16):
            c2 = Ctx(torch, native, parallel, dev, rank, world, cb)
            r = time_method(c2, args.method, inputs, 3, 3, False, dist, use_graph=False)
            calib[str(cb)] = {"eager_ms_per_step": r["eager_ms_per_step"], "add_batch_calls_per_linear": N_SEQ // cb,
                              "launches": r["launches"]}
    ctx.H = ctx.U = None
    torch.cuda.empty_cache()

    # the whole model through the drop-in driver (every rank takes part when world > 1)
    full_models = {}
    if args.all_methods and args.method == "wanda_nm" and not args.no_full_model:
        del inputs
        torch.cuda.empty_cache()
        # the third run adds the 12 Q-Former layers north_star names (SURVEY F9: the reference never prunes them; vlmc's
        # qformer_prune_spec extension does) - VERDICT r1 missing #7
        for key, m, nq in (("wanda_nm", "wanda_nm", 0), ("sparsegpt", "sparsegpt", 0), ("wanda_nm_with_qformer", "wanda_nm", 12)):
            try:
                full_models[f"full_model_instructblip_vicuna7b_{key}"] = full_model_vicuna(torch, native, dev, m, rank, world,
                                                                                         n_qformer=nq)
            except Exception as e:  # noqa: BLE001  (the headline line must not depend on it)
                full_models[f"full_model_instructblip_vicuna7b_{key}"] = {"error": f"{type(e).__name__}: {e}"[:300]}
                torch.cuda.synchronize()
        inputs = make_inputs(torch, dev, s1 - s0, seed=1000 + 17 * rank)

    e2e = run_e2e(torch, native, parallel, dev, args, rank, world, inputs)
    if world > 1:
        t = torch.tensor([e2e["ms"]], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e["ms"] = float(t.item())

    if rank == 0:
        pk = peaks()
        try:
            pk["tf32"] = measure_tf32_peak(torch, dev)
        except Exception:  # noqa: BLE001
            pk["tf32"] = None
        out = {
            "metric": METRIC, "value": main["ms_per_step"] / 1e3, "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": main["ms_per_step"],
            "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": f"{WORKLOAD[args.method]} on one InstructBLIP-Vicuna-7B LLM block (7 linears, fp16 "
                                   f"weights, random init), {N_SEQ}x{SEQ_LEN} fp16 calibration tokens per linear",
                       "method": args.method, "calib_batch": args.calib_batch, "cuda_graph": main["cuda_graph"],
                       "dump_outputs": {"dir": args.dump_outputs, "pass": main["outputs_pass"], "weight_seed": DUMP_SEED,
                                        "rows_per_linear": DUMP_ROWS} if args.dump_outputs is not None else None,
                       "eager_ms_per_step": main["eager_ms_per_step"], "eager_step_ms": main["eager_step_ms"],
                       "graph_ms_per_step": main.get("graph_ms_per_step"), "weight_sets": main["weight_sets"],
                       "l2": "inputs larger than L2 (12.2 GB of activations per step, fresh weight set per step)",
                       "statistics_launch": ("one launch per linear, two alternating streams"
                                             if (os.environ.get("VLMC_BENCH_STATS_BATCH") == "0" and world == 1) or args.calib_batch < N_SEQ
                                             else "one multi-tensor launch per block (vlmc_sqnorm_accum_batch)")
                       if args.method.startswith("wanda") else "one launch per linear",
                       "parallelism": ("tokens/%d + allreduce, rows/%d + allgather" % (world, world)) if world > 1 else "1 GPU"},
            "gpu_launches": main["launches"],
            "clocks": main["clocks"],
            "e2e": {"value": e2e["ms"] / 1e3, "unit": UNIT, "h2d_bytes_per_step": e2e["h2d"],
                    "d2h_bytes_per_step": e2e["d2h"]},
            "roofline": roofline_of(main, pk),
            "peaks": {"hbm_gbs": pk["hbm"], "bf16_tflops": pk["tensor"], "bf16_tflops_sustained": pk["tensor_sustained"],
                      "tf32_tflops_measured_here": pk.get("tf32"), "source": pk["source"]},
        }
        if calib:
            out["config"]["calib_batch_sweep"] = dict(calib, note="seconds per block of the same step with 1 / 16 sequences per "
                                                      "add_batch call (eager launches): 1 = the reference's per-sample hooks, 16 = what "
                                                      "vlmc's drop-in driver issues (calib_batch default)")
        if others:
            out["methods"] = {m: {"value": r["ms_per_step"] / 1e3, "unit": UNIT, "steps": r["steps"],
                                  "cuda_graph": r["cuda_graph"], "eager_ms_per_step": r["eager_ms_per_step"],
                                  "graph_ms_per_step": r.get("graph_ms_per_step"),
                                  "eager_step_ms": r["eager_step_ms"], "clocks": r["clocks"],
                                  "roofline": roofline_of(r, pk)} for m, r in others.items()}
        if "cuda_graph_error" in main:
            out["config"]["cuda_graph_error"] = main["cuda_graph_error"]
        if full_models:
            out.setdefault("workloads", {}).update(full_models)
        if world == 1 and args.all_methods and args.method == "wanda_nm":
            out.setdefault("workloads", {}).update({"config2_instructblip_flant5xl_wanda_2of4": full_model_wanda_nm(torch, native, dev),
                                "config5_sparselora_and_hessian_sweep": config5_lora_and_hessian_sweep(torch, native, dev, inputs),
                                "f4_global_sparsity_allocation": f4_global_allocation(torch, native, dev,
                                                                                      cpu=not args.no_cpu_baseline)})
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(args.method)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_e2e(torch, native, parallel, dev, args, rank, world, dev_inputs):
    """Host buffers in, host buffers out, through the wrapper classes: per distinct input, pinned chunks stream H2D on
    a copy stream while the statistics kernels consume the previous chunk; weights H2D, pruned weights (and masks)
    D2H.  Same per-linear work as the device-resident step."""
    from vlmc.compression.pruners.wanda_pruner import WrappedGPT
    from vlmc.compression.pruners.sparsegpt_pruner import SparseGPT
    from vlmc.compression.pruners import dsnot_pruner
    method = args.method
    shared = method.endswith("_shared")
    if shared:
        method = method[:-len("_shared")]
    elide = method == "dsnot_elided"
    if elide:
        method = "dsnot"
    n_local = next(iter(dev_inputs.values())).shape[0]
    chunk = min(8, n_local)
    host_in = {}
    for k, x in dev_inputs.items():
        h = torch.empty(x.shape, dtype=x.dtype, pin_memory=True)
        h.copy_(x)
        host_in[k] = h
    torch.cuda.synchronize()
    host_w = {name: (torch.randn(r, c) * 0.02).half().pin_memory() for name, r, c, _ in LINEARS}
    host_out_w = {name: torch.empty(r, c, dtype=torch.float16, pin_memory=True) for name, r, c, _ in LINEARS}
    host_out_m = {name: torch.empty(r, c, dtype=torch.bool, pin_memory=True) for name, r, c, _ in LINEARS}
    copy_stream = torch.cuda.Stream(device=dev)
    main = torch.cuda.current_stream(dev)
    bufs = {C: [torch.empty(chunk, SEQ_LEN, C, device=dev, dtype=torch.float16) for _ in range(2)] for C in (D, FF)}
    h2d = sum(h.numel() * 2 for h in host_in.values()) + sum(w.numel() * 2 for w in host_w.values())
    with_mask = method != "sparsegpt"
    d2h = sum(w.numel() * (3 if with_mask else 2) for w in host_w.values())

    class Lin(torch.nn.Module):   # the wrappers only need .weight (shape, device, dtype)
        def __init__(self, w):
            super().__init__()
            self.weight = torch.nn.Parameter(w, requires_grad=False)

    def make_wrapper(w):
        if method == "sparsegpt":
            lin = torch.nn.Linear(1, 1, bias=False)
            lin.weight = torch.nn.Parameter(w, requires_grad=False)
            return SparseGPT(lin)
        if method == "dsnot":
            return dsnot_pruner.WrappedGPT(Lin(w))
        return WrappedGPT(Lin(w))

    def step():
        dW = {}
        with torch.cuda.stream(copy_stream):
            for name in host_w:
                dW[name] = host_w[name].to(dev, non_blocking=True)
        w_ready = torch.cuda.Event()
        w_ready.record(copy_stream)
        main.wait_event(w_ready)
        wrappers = {name: make_wrapper(dW[name]) for name, *_ in LINEARS}
        for inp, C in INPUT_DIMS.items():
            users = [n for n, _, _, i in LINEARS if i == inp]
            free = [torch.cuda.Event(), torch.cuda.Event()]
            for ci, j in enumerate(range(0, n_local, chunk)):
                b = bufs[C][ci % 2]
                n = min(chunk, n_local - j)
                with torch.cuda.stream(copy_stream):
                    if ci >= 2:
                        copy_stream.wait_event(free[ci % 2])
                    b[:n].copy_(host_in[inp][j:j + n], non_blocking=True)
                    ready = torch.cuda.Event()
                    ready.record(copy_stream)
                main.wait_event(ready)
                for u in (users[:1] if shared else users):   # per-linear API: each linear reads the chunk itself
                    if method == "dsnot":            # one reference call per sequence (var is a mean of per-call variances)
                        for q in range(n):
                            wrappers[u].add_batch(b[q:q + 1], None)
                    else:
                        wrappers[u].add_batch(b[:n], None)
                free[ci % 2] = torch.cuda.Event()
                free[ci % 2].record(main)
        if method == "sparsegpt":         # the block's chains run concurrently (sparsegpt_pruner.fasterprune_block)
            from vlmc.compression.pruners.sparsegpt_pruner import fasterprune_block
            ws = [wrappers[name] for name, *_ in LINEARS]
            if shared:                    # what layerwise.InputSharing does in the driver: followers adopt the leader's H
                for leader, members in stat_groups(True):
                    for m in members[1:]:
                        wrappers[m].H = wrappers[leader].H
            fasterprune_block(ws, [0.5] * len(ws), percdamp=0.01, blocksize=128)
            for wr, (name, *_) in zip(ws, LINEARS):
                wr.free()
                host_out_w[name].copy_(wr.layer.weight.data, non_blocking=True)
            return
        for name, R, C, _ in LINEARS:
            wr = wrappers[name]
            if shared and method != "sparsegpt":
                lead = next(l for l, ms in stat_groups(True) if name in ms)
                wr.scaler_row, wr.nsamples = wrappers[lead].scaler_row, wrappers[lead].nsamples
            if method == "dsnot":
                dsnot_pruner.dsnot_prune_linear(wr.layer, wr, 0.6, elide_noop_swaps=elide)
            elif method == "wanda_nm":
                continue                       # pruned below, the whole block in one launch
            else:
                from vlmc.compression.pruners.wanda_pruner import wanda_prune_linear
                wanda_prune_linear(wr.layer, wr.scaler_row, 0.5)
            host_out_w[name].copy_(wr.layer.weight.data, non_blocking=True)
            host_out_m[name].copy_(wr.layer.mask, non_blocking=True)
        if method == "wanda_nm":
            from vlmc.compression.pruners.wanda_pruner import wanda_prune_block_nm
            ws = [wrappers[name] for name, *_ in LINEARS]
            wanda_prune_block_nm([w.layer for w in ws], [w.scaler_row for w in ws], 2, 4)
            for wr, (name, *_) in zip(ws, LINEARS):
                host_out_w[name].copy_(wr.layer.weight.data, non_blocking=True)
                host_out_m[name].copy_(wr.layer.mask, non_blocking=True)

    if world > 1:
        return run_e2e_sharded(torch, native, parallel, dev, args, rank, world, host_in, host_w, host_out_w,
                               host_out_m, bufs, copy_stream, main, h2d, d2h, chunk)
    step()
    torch.cuda.synchronize()
    k = max(2, min(args.steps, 3))
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    wall0 = time.perf_counter()
    t0.record()
    for _ in range(k):
        step()
    t1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - wall0) * 1e3
    return {"ms": max(t0.elapsed_time(t1), wall) / k, "h2d": h2d, "d2h": d2h, "steps": k}


def run_e2e_sharded(torch, native, parallel, dev, args, rank, world, host_in, host_w, host_out_w, host_out_m, bufs,
                    copy_stream, main, h2d, d2h, chunk):
    """N > 1: every rank streams ITS sequences from its pinned host buffers, then the same sharded step as the
    device-resident arm; rank-local H2D / D2H bytes are reported (weights go to every rank)."""
    ctx = Ctx(torch, native, parallel, dev, rank, world, args.calib_batch)
    n_local = next(iter(host_in.values())).shape[0]
    dev_in = {k: torch.empty(v.shape, dtype=v.dtype, device=dev) for k, v in host_in.items()}

    # every rank moves 1 / world of the block over ITS PCIe link: its calibration sequences, its row shard of the weights
    # up (the replicas are completed over NVLink with one all-gather per linear) and its row shard of the pruned weights
    # and masks down - together the host receives exactly one copy of the result (VERDICT r1 weak #8: every rank used to
    # upload all weights and download all results through one host)
    shard = {name: parallel.row_range(r, rank, world) for name, r, c, _ in LINEARS}
    even = all(r % world == 0 for _, r, _, _ in LINEARS)
    h2d = sum(h.numel() * 2 for h in host_in.values()) + sum((shard[n][1] - shard[n][0]) * c * 2 for n, r, c, _ in LINEARS)
    d2h = sum((shard[n][1] - shard[n][0]) * c * (3 if args.method.split("_")[0] != "sparsegpt" else 2) for n, r, c, _ in LINEARS)
    if not even:
        h2d = sum(h.numel() * 2 for h in host_in.values()) + sum(w.numel() * 2 for w in host_w.values())

    def step():
        dW = {name: torch.empty(r, c, dtype=torch.float16, device=dev) for name, r, c, _ in LINEARS}
        with torch.cuda.stream(copy_stream):
            for name in host_w:
                a, b = shard[name] if even else (0, host_w[name].shape[0])
                dW[name][a:b].copy_(host_w[name][a:b], non_blocking=True)
            for k in host_in:
                for j in range(0, n_local, chunk):
                    dev_in[k][j:j + chunk].copy_(host_in[k][j:j + chunk], non_blocking=True)
            ready = torch.cuda.Event()
            ready.record(copy_stream)
        main.wait_event(ready)
        if even:
            for name in host_w:
                parallel.gather_rows(dW[name], rank, world)
        masks = run_step(ctx, args.method, dW, dev_in)
        for name in host_w:
            a, b = shard[name]
            host_out_w[name][a:b].copy_(dW[name][a:b], non_blocking=True)
            if masks:
                host_out_m[name][a:b].copy_(masks[name][a:b], non_blocking=True)

    step()
    torch.cuda.synchronize()
    torch.distributed.barrier()
    k = 2
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.perf_counter()
    t0.record()
    for _ in range(k):
        step()
    t1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - wall0) * 1e3
    return {"ms": max(t0.elapsed_time(t1), wall) / k, "h2d": h2d, "d2h": d2h, "steps": k}


# ------------------------------------------------------------------------------------------------ config 2
# BASELINE.json configs[1]: Wanda 2:4 on the full InstructBLIP-FlanT5-XL (EVA ViT-g + FlanT5-XL), 1 B200, SURVEY 8(d).
VIT_BLOCK = [("qkv", 4224, 1408, "f32"), ("proj", 1408, 1408, "f16"), ("fc1", 6144, 1408, "f32"), ("fc2", 1408, 6144, "f16")]
T5_ENC = [(n, 2048, 2048, "bf16") for n in ("q", "k", "v", "o")] + [("wi_0", 5120, 2048, "bf16"), ("wi_1", 5120, 2048, "bf16"),
                                                                   ("wo", 2048, 5120, "bf16")]
T5_DEC = [(f"{a}.{n}", 2048, 2048, "bf16") for a in ("self", "cross") for n in ("q", "k", "v", "o")] + T5_ENC[4:]
FULL_MODEL = [("eva_vit_g", VIT_BLOCK, 39, 257, "f16"), ("t5_encoder", T5_ENC, 24, 512, "bf16"),
              ("t5_decoder", T5_DEC, 24, 512, "bf16")]


def full_model_wanda_nm(torch, native, dev, reps=2):
    """Every linear of every block: WrappedGPT statistics over its 128-sequence calibration input, then 2:4 selection.
    Inputs rotate through buffers larger than L2; ViT qkv / fc1 inputs are fp32 (nn.LayerNorm under autocast), the
    rest half precision (SURVEY App. A).  Returns seconds per model and the bytes streamed."""
    dt = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}
    g = torch.Generator(device=dev).manual_seed(7)
    plan, total_bytes, total_weights = [], 0, 0
    for name, linears, nblocks, seq, wtag in FULL_MODEL:
        T = N_SEQ * seq
        acts, wts = {}, []
        for _, R, C, xtag in linears:
            key = (C, xtag)
            if key not in acts:        # 3 rotating copies, each >= 93 MB: consecutive uses never hit in L2
                acts[key] = [torch.randn(T, C, device=dev, generator=g, dtype=torch.float32).to(dt[xtag]) for _ in range(3)]
        for _ in range(4):             # 4 rotating weight sets per block type
            wts.append([(torch.randn(R, C, device=dev, generator=g) * 0.02).to(dt[wtag]) for _, R, C, _ in linears])
        plan.append((linears, nblocks, acts, wts, T))
        for _, R, C, xtag in linears:
            total_bytes += nblocks * (T * C * (4 if xtag == "f32" else 2) + R * C * 5)
            total_weights += nblocks * R * C

    def one_model():
        use = 0
        for linears, nblocks, acts, wts, T in plan:
            for b in range(nblocks):
                W = wts[b % len(wts)]
                scal = []
                for i, (_, R, C, xtag) in enumerate(linears):
                    x = acts[(C, xtag)][use % 3]
                    use += 1
                    s = torch.zeros(C, device=dev, dtype=torch.float32)
                    native.sqnorm_accum(x.view(N_SEQ, -1, C), s, 0, N_SEQ)
                    scal.append(s)
                native.wanda_nm_batch(W, scal, 2, 4)      # the block's linears in one launch
    one_model()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        one_model()
    b.record()
    torch.cuda.synchronize()
    eager_sec = a.elapsed_time(b) / reps / 1e3
    sec, graphed = eager_sec, False
    try:    # ~2400 launches of 30-100 us kernels: replayed from one CUDA graph the host leaves the timed region
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            one_model()
        g.replay()
        torch.cuda.synchronize()
        a.record()
        for _ in range(reps):
            g.replay()
        b.record()
        torch.cuda.synchronize()
        sec, graphed = a.elapsed_time(b) / reps / 1e3, True
        del g
    except Exception:  # noqa: BLE001
        torch.cuda.synchronize()
    del plan
    torch.cuda.empty_cache()
    return {"value": sec, "unit": "s/model", "workload": "Wanda 2:4 on full InstructBLIP-FlanT5-XL: 39 EVA ViT-g blocks (fp16, "
            "128x257 tokens, fp32 qkv/fc1 inputs) + 24 + 24 FlanT5-XL blocks (bf16, 128x512 tokens), random init",
            "linears": sum(len(l) * n for _, l, n, _, _ in FULL_MODEL), "weights": total_weights,
            "algorithmic_bytes": total_bytes, "achieved_gbs": total_bytes / sec / 1e9, "reps": reps,
            "cuda_graph": graphed, "eager_s_per_model": eager_sec}


# ------------------------------------------------------------------------------------------------ full model (row g)
VICUNA_LAYER = [("self_attn.q_proj", D, D, "attn_in"), ("self_attn.k_proj", D, D, "attn_in"), ("self_attn.v_proj", D, D, "attn_in"),
                ("self_attn.o_proj", D, D, "attn_out"), ("mlp.gate_proj", FF, D, "mlp_in"), ("mlp.up_proj", FF, D, "mlp_in"),
                ("mlp.down_proj", D, FF, "mlp_mid")]
VIT_G_BLOCK = [("attn.qkv", 4224, 1408, "ln1_f32"), ("attn.proj", 1408, 1408, "attn_out"), ("mlp.fc1", 6144, 1408, "ln2_f32"),
               ("mlp.fc2", 1408, 6144, "mlp_mid")]
QFORMER_LAYER = [("attention.self.query", 768, 768, "q_in"), ("attention.self.key", 768, 768, "q_in"),
                 ("attention.self.value", 768, 768, "q_in"), ("attention.output.dense", 768, 768, "q_ctx"),
                 ("crossattention.self.query", 768, 768, "q_mid"), ("crossattention.self.key", 768, 1408, "img"),
                 ("crossattention.self.value", 768, 1408, "img"), ("crossattention.output.dense", 768, 768, "q_ctx2"),
                 ("intermediate_query.dense", 3072, 768, "q_ff"), ("output_query.dense", 768, 3072, "q_ffmid")]


def build_stand_in_model(torch, dev, n_local, n_llm=32, n_vit=39, n_qformer=0, seed=0):
    """Random-init stand-in of InstructBLIP-Vicuna-7B for the drop-in driver: real nn.Linear modules of the named shapes
    (32 LLaMA layers, 39 EVA ViT-g blocks, optionally the 12 Q-Former layers of SURVEY F9) under the attribute paths the
    composite pruners walk.  Block forwards are excluded from the metric (SURVEY 8d): every linear's forward is skipped,
    Module.__call__ still fires the calibration hooks with that linear's resident synthetic input (fp32 after the ViT's
    LayerNorms, fp16 elsewhere, SURVEY App. A).  Returns (model, data_loader)."""
    import contextlib
    import types
    nn = torch.nn
    g = torch.Generator(device=dev).manual_seed(seed)

    class Feeds:
        """One resident [n_local, S, C] tensor per distinct input of a block type, shared by its blocks (and never the same
        tensor for two different linears unless the real model feeds them the same activation)."""

        def __init__(self):
            self.t = {}

        def get(self, key, S, C, dtype):
            if key not in self.t:
                x = torch.empty(n_local, S, C, device=dev, dtype=dtype)
                gain = torch.exp(torch.rand(C, device=dev, generator=g) * 2.77 - 1.386)
                off = torch.randn(C, device=dev, generator=g) * 0.3
                for j in range(n_local):
                    x[j] = (torch.randn(S, C, device=dev, generator=g) * gain + off).to(dtype)
                self.t[key] = x
            return self.t[key]
    feeds = Feeds()

    class Block(nn.Module):
        def __init__(self, spec, S, wdtype, kind, first_input):
            super().__init__()
            self.spec, self.S, self.kind, self.first_input, self.pos = spec, S, kind, first_input, 0
            dummy = torch.zeros(1, 1, 1, device=dev, dtype=wdtype)
            for name, R, C, _ in spec:
                lin = nn.Linear(C, R, bias=False, device="meta")
                lin.weight = nn.Parameter((torch.randn(R, C, device=dev, generator=g) * 0.02).to(wdtype), requires_grad=False)
                lin.forward = types.MethodType(lambda self_, x, _d=dummy: _d, lin)      # no GEMM; hooks still fire
                parent = self
                *path, leaf = name.split(".")
                for part in path:
                    if not hasattr(parent, part):
                        setattr(parent, part, nn.Module())
                    parent = getattr(parent, part)
                setattr(parent, leaf, lin)

        def forward(self, x, *args, **kwargs):
            b = x.shape[0]
            lo = self.pos % n_local
            if lo + b > n_local:
                lo = 0
            self.pos = lo + b
            for name, R, C, inp in self.spec:
                if inp == self.first_input:
                    xin = x
                else:
                    dt = torch.float32 if inp.endswith("_f32") else x.dtype
                    S = 257 if inp == "img" else self.S
                    xin = feeds.get((self.kind, inp), S, C, dt)[lo:lo + b]
                self.get_submodule(name)(xin)
            return x if self.kind == "vit" else (x,)

    class Model(nn.Module):
        def __init__(self):
            super().__init__()
            self.visual_encoder = nn.Module()
            self.visual_encoder.blocks = nn.ModuleList([Block(VIT_G_BLOCK, 257, torch.float16, "vit", "none") for _ in range(n_vit)])
            if n_qformer:
                self.Qformer = nn.Module()
                self.Qformer.bert = nn.Module()
                self.Qformer.bert.encoder = nn.Module()
                self.Qformer.bert.encoder.layer = nn.ModuleList([Block(QFORMER_LAYER, 32, torch.float32, "qformer", "q_in")
                                                                 for _ in range(n_qformer)])
            self.llm_model = nn.Module()
            self.llm_model.config = types.SimpleNamespace(use_cache=True)
            self.llm_model.model = nn.Module()
            self.llm_model.model.layers = nn.ModuleList([Block(VICUNA_LAYER, SEQ_LEN, torch.float16, "llm", "attn_in")
                                                         for _ in range(n_llm)])

        def maybe_autocast(self, dtype=torch.float16):
            return contextlib.nullcontext()

        def forward(self, batch):
            # only the stack whose first block is being captured runs (the others would be block forwards: excluded)
            def capturing(layers):
                return len(layers) > 0 and type(layers[0]).__name__ == "Catcher"
            if capturing(self.visual_encoder.blocks):
                x = batch["image"]
                for blk in self.visual_encoder.blocks:
                    x = blk(x, None)
            if n_qformer and capturing(self.Qformer.bert.encoder.layer):
                q = batch["query"]
                for layer in self.Qformer.bert.encoder.layer:
                    q = layer(q, None, None, batch["image"], None, None, False, q.shape[1])[0]
            if capturing(self.llm_model.model.layers):
                h = batch["llm_in"]
                for layer in self.llm_model.model.layers:
                    h = layer(h, attention_mask=None, position_ids=None)[0]
            return None

    model = Model().eval()
    img = feeds.get(("loader", "image"), 257, 1408, torch.float16)
    llm_in = feeds.get(("loader", "llm_in"), SEQ_LEN, D, torch.float16)
    query = feeds.get(("loader", "query"), 32, 768, torch.float32) if n_qformer else None
    loader = []
    for j in range(n_local):
        d = {"image": img[j:j + 1], "llm_in": llm_in[j:j + 1], "text_input": ["a"]}
        if n_qformer:
            d["query"] = query[j:j + 1]
        loader.append(d)
    return model, loader


def full_model_vicuna(torch, native, dev, method, rank, world, n_llm=32, n_vit=39, n_qformer=0):
    """Row g of the verdict / north_star Target: the WHOLE InstructBLIP-Vicuna-7B stand-in (39 ViT-g blocks + 32 LLaMA
    layers, optionally + 12 Q-Former layers) through the registered drop-in entry point
    load_pruner(...).prune() - hooks, calibration batching, shared inputs, per-block selection - with block forwards
    excluded.  On several GPUs the driver runs data-parallel (calibration samples split, statistics merged per block).
    Wall-clock seconds per model, synchronised on both sides; masks checked for structure."""
    import contextlib
    import io
    import vlmc.compression as comp
    n_local = len(range(rank, N_SEQ, world))
    nm = method == "wanda_nm"
    name = "blipt5_wanda_pruner" if method.startswith("wanda") else "blipt5_sparsegpt_pruner"
    if not getattr(full_model_vicuna, "_warm", {}).get(name):
        # one-time costs of a process (lazy cubin loads of every kernel of the path, workspace and allocator growth) are paid
        # on a ONE-block model first: the timed run then measures the steady state of a 71-block model
        wm, wl = build_stand_in_model(torch, dev, N_SEQ, 1, 1, 1 if n_qformer else 0, seed=1)
        wcfg = dict(t5_prune_spec="1-0.5-1.0-1.0", vit_prune_spec="1-0.5-1.0-1.0", t5_pruning_method="none",
                    vit_pruning_method="none", t5_model_prefix="llm_model", num_samples=N_SEQ, sparsity_ratio_granularity=None,
                    score_method="obd_avg", prune_n=2 if nm else 0, prune_m=4 if nm else 0, data_parallel=world > 1)
        with contextlib.redirect_stdout(io.StringIO()):
            comp.load_pruner(name, wm, wl, cfg=wcfg).prune()
        torch.cuda.synchronize()
        del wm, wl
        full_model_vicuna._warm = dict(getattr(full_model_vicuna, "_warm", {}), **{name: True})
    model, loader = build_stand_in_model(torch, dev, N_SEQ, n_llm, n_vit, n_qformer)
    cfg = dict(t5_prune_spec="24-0.5-1.0-1.0", vit_prune_spec="39-0.5-1.0-1.0", t5_pruning_method="none",
               vit_pruning_method="none", t5_model_prefix="llm_model", num_samples=N_SEQ, sparsity_ratio_granularity=None,
               score_method="obd_avg", prune_n=2 if nm else 0, prune_m=4 if nm else 0, data_parallel=world > 1)
    if n_qformer:
        cfg["qformer_prune_spec"] = "12-0.5-1.0-1.0"
    pruner = comp.load_pruner(name, model, loader, cfg=cfg)
    torch.cuda.empty_cache()         # blocks cached by earlier phases of the bench are not this run's to free (cudaFree is synchronous)
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        pruner.prune()
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([sec], device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        sec = float(t.item())
    # structure checks on the pruned replica
    lins = [m for m in model.modules() if isinstance(m, torch.nn.Linear)]
    total = sum(m.weight.numel() for m in lins)
    nz = int(native.count_nonzero([m.weight.data for m in lins]).sum().item())
    sparsity = 1.0 - float(nz) / total
    ok = abs(sparsity - 0.5) < 2e-3
    if nm:
        for m in (lins[0], lins[len(lins) // 2], lins[-1]):
            ok = ok and bool((m.mask.view(m.mask.shape[0], -1, 4).sum(-1) == 2).all())
    digest = nz
    del pruner, model, loader
    torch.cuda.empty_cache()
    return {"value": sec, "unit": "s/model", "workload": f"{WORKLOAD[method]} on the whole InstructBLIP-Vicuna-7B stand-in: {n_vit} EVA "
            f"ViT-g blocks + {n_llm} LLaMA layers" + (f" + {n_qformer} Q-Former layers" if n_qformer else "") +
            f" through load_pruner('{name}').prune(), {N_SEQ} calibration samples (2048 LLM tokens, 257 image tokens), "
            "block forwards excluded, random init", "linears": len(lins), "weights": total, "sparsity": sparsity,
            "structure_ok": ok, "nonzero_digest": digest, "n_gpus": world, "data_parallel": world > 1,
            "calib_batch": 16, "warmup": "one 1-block model through the same entry point (untimed)"}


# ------------------------------------------------------------------------------------------------ config 5
def config5_lora_and_hessian_sweep(torch, native, dev, inputs):
    """BASELINE.json configs[4]: (i) SparseLoRA masked merge (K14) and the masked-forward weight build (K15) over the 7
    linears of a Vicuna-7B block (r = 8, random 50 % mask), 5 B / weight each; (ii) Hessian accumulation at calibration
    scales 128..1024 x 2048 tokens for C = 4096 and C = 11008 (the resident 128-sequence input is fed repeatedly with a
    growing n_before: same kernel work as a longer calibration set)."""
    g = torch.Generator(device=dev).manual_seed(11)
    out = {}
    items = []
    for name, R, C, _ in LINEARS:
        W = (torch.randn(R, C, device=dev, generator=g) * 0.02).half()
        A = torch.randn(8, C, device=dev, generator=g) * 0.1
        B = torch.randn(R, 8, device=dev, generator=g) * 0.1
        M = torch.rand(R, C, device=dev, generator=g) < 0.5
        items.append((W, A, B, M, torch.empty_like(W)))
    nbytes = sum(W.numel() for W, *_ in items) * 5

    def timed(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps
    ms = timed(lambda: [native.sparselora_merge(W, A, B, 2.0, M, remask=True) for W, A, B, M, _ in items])
    out["sparselora_merge_block"] = {"ms": ms, "achieved_gbs": nbytes / ms / 1e6, "bytes": nbytes}
    ms = timed(lambda: native.sparselora_merge_batch([i[0] for i in items], [i[1] for i in items], [i[2] for i in items],
                                                     [2.0] * len(items), [i[3] for i in items], remask=True))
    out["sparselora_merge_block_one_launch"] = {"ms": ms, "achieved_gbs": nbytes / ms / 1e6, "bytes": nbytes}
    ms = timed(lambda: [native.sparselora_effective_weight(W, A, B, 2.0, M, True, out=o) for W, A, B, M, o in items])
    out["sparselora_forward_weight_block"] = {"ms": ms, "achieved_gbs": nbytes / ms / 1e6, "bytes": nbytes}
    del items
    sweep = {}
    for inp, C in (("attn_in", D), ("mlp_mid", FF)):
        x = inputs[inp]
        H = torch.zeros(C, C, device=dev)
        native.hessian_accum(x, H, 0, N_SEQ)
        for nseq in (128, 256, 512, 1024):
            reps = nseq // N_SEQ
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for r in range(reps):
                native.hessian_accum(x, H, r * N_SEQ, N_SEQ)
            b.record()
            torch.cuda.synchronize()
            t = a.elapsed_time(b)
            nt = (C + 255) // 256                          # the SYRK executes the upper 256 x 256 tiles only
            executed = 2.0 * nseq * SEQ_LEN * (nt * (nt + 1) // 2) * 256.0 * 256.0
            sweep[f"C{C}_T{nseq}x{SEQ_LEN}"] = {"ms": t, "logical_tflops": 2.0 * nseq * SEQ_LEN * C * C / t / 1e9,
                                                  "executed_tflops": executed / t / 1e9}
        del H
    out["hessian_accum_sweep"] = sweep
    torch.cuda.empty_cache()
    return out


def f4_global_allocation(torch, native, dev, cpu=True):
    """SURVEY 8f-4: LayerSparsity on the parameters of one Vicuna-7B block (7 linears, 202 M fp32 scores, 0.81 GB): the
    first-order score build (K22), the group sums (K21) and get_mask(p = 0.5, max_sparsity_per_layer = 0.8) = per-tensor
    protection (K18 + K19), the whole-block exact threshold (K18) and masks with the fused `param *= mask` (K20).
    The reference runs the same on the CPU (v.cpu(), torch.topk over the concatenation); `cpu_reference` times its op
    sequence (oracle/cpu_port.global_get_mask) on q_proj alone (16.8 M scores) on the host cores."""
    from vlmc.compression.pruners import layer_sparsity as ls
    g = torch.Generator(device=dev).manual_seed(13)
    params = [(torch.randn(R, C, device=dev, generator=g) * 0.02).half() for _, R, C, _ in LINEARS]
    grads = [(torch.randn(R, C, device=dev, generator=g) * 1e-3).half() for _, R, C, _ in LINEARS]
    acc = [torch.zeros(p.shape, device=dev) for p in params]
    scores = [torch.empty_like(a) for a in acc]
    n = sum(p.numel() for p in params)

    def timed(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps
    out = {"scores": n}
    ms = timed(lambda: native.importance_accum(acc, grads, "obd"))
    out["importance_accum"] = {"ms": ms, "achieved_gbs": n * 10 / ms / 1e6, "bytes_per_score": 10}
    ms = timed(lambda: native.importance_finalize(acc, params, scores, "obd", 4))
    out["importance_finalize"] = {"ms": ms, "achieved_gbs": n * 10 / ms / 1e6, "bytes_per_score": 10}
    ms = timed(lambda: native.scores_sum(scores))
    out["scores_sum"] = {"ms": ms, "achieved_gbs": n * 4 / ms / 1e6, "bytes_per_score": 4}
    ms = timed(lambda: native.scores_kth(scores, [0] * len(scores), [n // 2]))
    out["scores_kth_global"] = {"ms": ms, "achieved_gbs": n * 12 / ms / 1e6, "bytes_per_score": 12, "passes": 3}
    named = {name: s for (name, *_), s in zip(LINEARS, scores)}
    pd = {name: p for (name, *_), p in zip(LINEARS, params)}
    ms = timed(lambda: ls.get_mask(named, 0.5, 0.8, params=pd))
    # protect: 3 reads + 1 read/partial write; select: 3 reads; mask: read 4 + write 4 + read/write 2 + 2
    out["get_mask_protect_select_mask_prune"] = {"ms": ms, "achieved_gbs": n * 40 / ms / 1e6, "bytes_per_score": 40}
    if cpu:
        from oracle import cpu_port
        torch.set_num_threads(os.cpu_count() or 1)
        gq = torch.Generator().manual_seed(3)
        sc = {"q_proj": torch.randn(D, D, generator=gq) ** 2 * 1e-6}
        t0 = time.perf_counter()
        cpu_port.global_get_mask(sc, 0.5, 0.8)
        t = time.perf_counter() - t0
        out["cpu_reference"] = {"seconds_q_proj_only": t, "scores": D * D, "cores": os.cpu_count() or 1, "kind": "port",
                                "scaled_to_block_s": t * n / (D * D)}
    del params, grads, acc, scores
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------ CPU arm
def _ref_available():
    try:
        from oracle import ref_loader
        return ref_loader.available()
    except Exception:  # noqa: BLE001
        return False


def cpu_block_seconds(method, threads, budget="small"):
    """The reference on the host cores.  When the unmodified reference files are present (build container:
    /root/reference; GPU box: the verbatim copy under baseline/_ref, oracle/fetch_ref.py) the reference's OWN composite
    pruner runs the whole block through its public entry point (oracle/ref_arm.py, kind "reference"); otherwise the torch
    port of its op sequence (oracle/cpu_port.py, kind "port") runs a bounded sample.
    Returns (seconds per block, description of the sample, kind)."""
    import torch
    if method.endswith("_shared"):        # the reference has no such mode: its per-linear schedule is the baseline
        method = method[:-len("_shared")]
    if method == "dsnot_elided":
        method = "dsnot"
    if _ref_available():
        from oracle import ref_arm
        if method == "wanda_nm":
            sec, _ = ref_arm.run_composite("wanda", ref_arm.VICUNA_BLOCK, N_SEQ, SEQ_LEN, torch.float16, 0.5, 2, 4, threads=threads)
            return sec, (f"the WHOLE block through the unmodified BLIPT5LayerWandaPruner.prune(): {N_SEQ} per-sequence add_batch "
                         "hook calls per linear + the 2:4 topk loop of the 7 linears (block forwards skipped, 8 distinct "
                         "resident sequences per input cycled)"), "reference"
        if method == "wanda_unstructured":
            sec, _ = ref_arm.run_composite("wanda", ref_arm.VICUNA_BLOCK, N_SEQ, SEQ_LEN, torch.float16, 0.5, threads=threads)
            return sec, (f"the WHOLE block through the unmodified BLIPT5LayerWandaPruner.prune(): {N_SEQ} per-sequence add_batch "
                         "hook calls per linear + the stable row sort of the 7 linears"), "reference"
        if method == "dsnot":
            rows_div, seqs = 8, 16
            small = [(n, R // rows_div, C, i) for n, R, C, i in ref_arm.VICUNA_BLOCK]
            # two runs separate the statistics (linear in sequences) from the refine (linear in rows)
            t_a, _ = ref_arm.run_composite("dsnot", small, seqs, SEQ_LEN, torch.float16, 0.6, threads=threads)
            t_b, _ = ref_arm.run_composite("dsnot", small, seqs // 2, SEQ_LEN, torch.float16, 0.6, threads=threads)
            per_seq = max(t_a - t_b, 0.0) / (seqs // 2)
            refine = max(t_a - per_seq * seqs, 0.0)
            return per_seq * N_SEQ + refine * rows_div, (
                f"unmodified BLIPT5LayerDSnoTPruner.prune() on 1/{rows_div} of the rows of each linear with {seqs} and "
                f"{seqs // 2} sequences ({t_a:.1f} s, {t_b:.1f} s): statistics scaled to {N_SEQ} sequences, refine scaled x{rows_div} "
                "(rows are independent; extrapolated)"), "reference"
        sec, note = ref_arm.sparsegpt_block_seconds(ref_arm.VICUNA_BLOCK, N_SEQ, SEQ_LEN, torch.float16, 0.5, threads=threads)
        return sec, "unmodified SparseGPT class: " + note, "reference"
    from oracle import cpu_port
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(0)
    xs = {inp: (torch.randn(SEQ_LEN, C, generator=g)).half() for inp, C in INPUT_DIMS.items()}
    if method in ("wanda_nm", "wanda_unstructured", "dsnot"):
        n_sample = 2
        t_stats, scal = 0.0, {}
        for name, R, C, inp in LINEARS:
            st = cpu_port.DSnoTStat(C) if method == "dsnot" else cpu_port.WandaStat(C)
            t0 = time.perf_counter()
            for _ in range(n_sample):
                st.add_batch(xs[inp].unsqueeze(0))
            t_stats += time.perf_counter() - t0
            scal[name] = st.scaler_row
        t_sel = 0.0
        for name, R, C, _ in LINEARS:
            W = (torch.randn(R, C, generator=g) * 0.02).half()
            t0 = time.perf_counter()
            if method == "wanda_nm":
                cpu_port.wanda_select(W, scal[name], 0.5, 2, 4)
            elif method == "dsnot":       # as shipped the DSnoT mask is the Wanda mask (SURVEY F4): its selection cost is a lower bound
                cpu_port.wanda_select(W, scal[name], 0.6)
            else:
                cpu_port.wanda_select(W, scal[name], 0.5)
            t_sel += time.perf_counter() - t0
        total = t_stats * (N_SEQ / n_sample) + t_sel
        return total, (f"statistics on {n_sample} of {N_SEQ} sequences per linear ({t_stats:.2f} s, scaled x{N_SEQ // n_sample}, "
                       f"extrapolated) + full selection of the 7 linears ({t_sel:.2f} s)"
                       + ("; DSnoT's swap loop not timed (lower bound)" if method == "dsnot" else "")), "port"
    # sparsegpt: Hessian accumulation on 1 sequence for C=4096 and C=11008, fasterprune on a 1024-column problem;
    # both scaled by their flop counts to the 7 linears of the block
    t_h = {}
    for C in (D, FF):
        p = cpu_port.SparseGPTPort(torch.zeros(8, C).half())
        t0 = time.perf_counter()
        p.add_batch(xs["attn_in" if C == D else "mlp_mid"].unsqueeze(0))
        t_h[C] = time.perf_counter() - t0
    t_hess = (6 * t_h[D] + t_h[FF]) * N_SEQ
    Rs, Cs = 1024, 1024
    p = cpu_port.SparseGPTPort((torch.randn(Rs, Cs, generator=g) * 0.02).half())
    x = torch.randn(4 * Cs, Cs, generator=g).half()
    p.add_batch(x.unsqueeze(0))
    t0 = time.perf_counter()
    p.fasterprune(0.5)
    t_fp = time.perf_counter() - t0
    # fasterprune cost model: C^3 (factorisations) + R*C^2 (sweep); scale the measured 1024^3 + 1024^3
    unit = t_fp / (Cs ** 3 + Rs * Cs ** 2)
    t_prune = sum(unit * (C ** 3 + R * C ** 2) for _, R, C, _ in LINEARS)
    return t_hess + t_prune, (f"SparseGPT.add_batch on 1 of {N_SEQ} sequences for C=4096 ({t_h[D]:.2f} s) and C=11008 "
                              f"({t_h[FF]:.2f} s) scaled to 7 linears x {N_SEQ} sequences, + fasterprune on a "
                              f"{Rs}x{Cs} linear ({t_fp:.2f} s) scaled by C^3 + R*C^2 to the 7 linears (extrapolated)"), "port"


def config1_cpu_reference(threads):
    """BASELINE.json configs[0]: Wanda 50 % unstructured on one FlanT5-XL encoder block (bf16, 128 x 512 calibration
    tokens), on the CPU through the unmodified reference, in full."""
    import torch
    if not _ref_available():
        return None
    from oracle import ref_arm
    sec, _ = ref_arm.run_composite("wanda", ref_arm.T5XL_ENC_BLOCK, N_SEQ, 512, torch.bfloat16, 0.5, threads=threads)
    return {"value": sec, "unit": "s/block", "cores": threads, "kind": "reference",
            "sample": "whole FlanT5-XL encoder block (7 linears) through the unmodified BLIPT5LayerWandaPruner.prune(), "
                      f"{N_SEQ} x 512 bf16 tokens per linear"}


def same_gpu_torch_eager(method):
    """SURVEY 8d (2): the reference is torch code that its users run on the GPU that holds the model: the unmodified
    composite pruner (oracle/ref_arm.py) with every tensor on this B200, torch eager, whole block.  Falls back to the port
    of its op sequence (oracle/cpu_port.py) when the reference files are absent.  A reported baseline like the CPU
    figure; only for the Wanda methods; never raises (the bench line must not depend on it)."""
    try:
        import torch
        if method not in ("wanda_nm", "wanda_unstructured") or not torch.cuda.is_available():
            return None
        dev = torch.device("cuda", torch.cuda.current_device())
        if _ref_available():
            from oracle import ref_arm
            nm = (2, 4) if method == "wanda_nm" else (0, 0)
            ref_arm.run_composite("wanda", ref_arm.VICUNA_BLOCK, 2, SEQ_LEN, torch.float16, 0.5, *nm, device=dev)   # warm-up
            sec, _ = ref_arm.run_composite("wanda", ref_arm.VICUNA_BLOCK, N_SEQ, SEQ_LEN, torch.float16, 0.5, *nm, device=dev)
            torch.cuda.empty_cache()
            return {"value": sec, "unit": UNIT, "kind": "reference",
                    "sample": f"whole block through the unmodified BLIPT5LayerWandaPruner.prune() with the model on the same B200 "
                              f"(torch eager): {N_SEQ} per-sequence add_batch hook calls per linear + selection of the 7 linears"}
        from oracle import cpu_port
        g = torch.Generator(device=dev).manual_seed(5)
        xs = {inp: torch.randn(8, SEQ_LEN, C, device=dev, generator=g).half() for inp, C in INPUT_DIMS.items()}
        Ws = {name: (torch.randn(R, C, device=dev, generator=g) * 0.02).half() for name, R, C, _ in LINEARS}

        def block(n_seq):
            for name, R, C, inp in LINEARS:
                st = cpu_port.WandaStat(C, device=dev)
                for j in range(n_seq):
                    st.add_batch(xs[inp][j % 8].unsqueeze(0))
                if method == "wanda_nm":
                    cpu_port.wanda_select(Ws[name], st.scaler_row, 0.5, 2, 4)
                else:
                    cpu_port.wanda_select(Ws[name], st.scaler_row, 0.5)
        block(1)                                           # warm-up: allocator, kernel load
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        block(N_SEQ)
        b.record()
        torch.cuda.synchronize()
        del xs, Ws
        torch.cuda.empty_cache()
        return {"value": a.elapsed_time(b) / 1e3, "unit": UNIT, "kind": "port",
                "sample": f"whole block: {N_SEQ} per-sequence add_batch calls per linear (8 distinct resident sequences reused) + "
                          "selection of the 7 linears, torch eager on the same B200"}
    except Exception as e:                                 # noqa: BLE001
        return {"error": f"{type(e).__name__}: {e}"[:200]}


def cpu_baseline(method):
    threads = os.cpu_count() or 1
    total, sample, kind = cpu_block_seconds(method, threads)
    out = {"value": total, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample}
    same_gpu = same_gpu_torch_eager(method)
    if same_gpu is not None:
        out["same_gpu_torch_eager"] = same_gpu
    return out


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the step on all host cores.  A step is the whole
    block for the Wanda methods."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    vals, sample, kind = [], "", "port"
    warm = 0
    if args.warmup > 0:
        total, sample, kind = cpu_block_seconds(args.method, threads)       # one untimed pass: page cache, thread pool
        warm = 1
    for _ in range(args.steps):
        total, sample, kind = cpu_block_seconds(args.method, threads)
        vals.append(total)
    v = sum(vals) / len(vals)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT,
        "n_gpus": args.gpus, "steps": len(vals), "warmup": warm, "ms_per_step": v * 1e3,
        "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{WORKLOAD[args.method]} on one InstructBLIP-Vicuna-7B LLM block (7 linears, fp16 weights, "
                               f"random init), {N_SEQ}x{SEQ_LEN} fp16 calibration tokens per linear",
                   "method": args.method},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": kind, "sample": "each step: " + sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="vlmc", choices=["vlmc", "reference"])
    ap.add_argument("--method", default="wanda_nm", choices=METHODS)
    ap.add_argument("--calib-batch", type=int, default=N_SEQ,
                    help="sequences per add_batch call (reference hooks use 1; the wrapper API takes any b)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--one-step", action="store_true", help="run ONE eager step of --method and exit (ncu traffic captures)")
    ap.add_argument("--no-full-model", action="store_true", help="skip the whole-model runs through load_pruner().prune()")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches only (no CUDA-graph replay pass)")
    ap.add_argument("--no-other-methods", dest="all_methods", action="store_false",
                    help="skip the short measurement of the methods other than --method")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of --method returned (pruned weights, keep masks; the same "
                         f"{DUMP_ROWS} seeded rows of every linear) as DIR/<linear>.<weight|mask>.npy, float32; one GPU only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "vlmc" or args.gpus != 1 or args.one_step):
        ap.error("--dump-outputs needs --impl vlmc, --gpus 1 and timed steps")
    if args.warmup < 3 and args.impl == "vlmc":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
