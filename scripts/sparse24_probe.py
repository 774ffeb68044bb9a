"""Compressed 2:4 linear (K26) against dense F.linear and against expand (K25) + F.linear on the 7 linears of a Vicuna-7B
block, fp16 and bf16, T = 1 .. 8192 tokens.  Sets vlmc.sparse24.DENSE_EXPAND_MIN_TOKENS and the DESIGN.md K24-K26 rows.

    python scripts/sparse24_probe.py [--reps 15] [--out sparse24_probe.json]

One timed sample = the whole block (404 MB of dense / 227 MB of compressed weights, both far above the 126 MB L2, so a
weight is never read from L2 across samples); the three arms are alternated inside every repetition; CUDA events around
each arm; median, min and max over the repetitions.  GB/s are on the algorithmic bytes (weights + x + y), quoted
against the copy peak measured in the same run (b.copy_(a), 2 GiB moved).  K24 / K25 are timed on the same block.
Each arm is timed twice: eager (host enqueue included: what a Python loop pays) and replayed from a CUDA graph of the
block's 7 calls (device time: what a decode loop captured in a graph pays).
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "vlm-compression_b200"))
from vlmc import native  # noqa: E402

SHAPES = [(4096, 4096)] * 4 + [(11008, 4096)] * 2 + [(4096, 11008)]      # q k v o, gate up, down  (R, C)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def timed(fn, reps=1):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def copy_peak():
    a = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    ms = sorted(timed(lambda: b.copy_(a)) for _ in range(10))[5]
    return 2 * a.numel() / ms / 1e6           # GB/s


def stats(v):
    v = sorted(v)
    return {"median": v[len(v) // 2], "min": v[0], "max": v[-1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--out", default=None, help="also write the rows as JSON here")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the probe measures the GPU; there is no CPU arm"
    torch.manual_seed(0)
    peak = copy_peak()
    cap = torch.cuda.Stream()
    res = {"gpu": gpu_info(), "copy_peak_gbs": peak, "reps": args.reps, "rows": []}
    print(f"# {res['gpu']}; copy peak {peak:.0f} GB/s", flush=True)
    for dt in (torch.float16, torch.bfloat16):
        Ws, comp = [], []
        for R, C in SHAPES:
            W = torch.randn(R, C, device="cuda", dtype=dt) * 0.02
            keep = torch.rand(R, C // 4, 4, device="cuda").argsort(-1) < 2
            W = (W.view(R, C // 4, 4) * keep).view(R, C)
            Ws.append(W)
            comp.append(native.sparse24_compress(W))
        wbytes_dense = sum(W.numel() * 2 for W in Ws)
        wbytes_comp = sum(v.numel() * 2 + m.numel() * 2 for v, m in comp)
        scratch = torch.empty(max(W.numel() for W in Ws), dtype=dt, device="cuda")
        t_comp = stats([timed(lambda: [native.sparse24_compress(W) for W in Ws]) for _ in range(5)])
        t_dec = stats([timed(lambda: [native.sparse24_decompress(v, m, W.shape[1], out=scratch[:W.numel()].view(W.shape))
                                      for W, (v, m) in zip(Ws, comp)]) for _ in range(5)])
        name = str(dt).replace("torch.", "")
        res[f"{name}_compress_ms"] = t_comp
        res[f"{name}_decompress_ms"] = t_dec
        print(f"# {name}: weights {wbytes_dense / 1e6:.1f} MB dense, {wbytes_comp / 1e6:.1f} MB compressed; "
              f"K24 block {t_comp['median']:.3f} ms ({(wbytes_dense + wbytes_comp) / t_comp['median'] / 1e6:.0f} GB/s), "
              f"K25 block {t_dec['median']:.3f} ms ({(wbytes_dense + wbytes_comp) / t_dec['median'] / 1e6:.0f} GB/s)",
              flush=True)
        print("dtype  T      dense_ms  fused_ms  expand_ms  fused/dense  dense_GBs fused_GBs (frac of copy peak)", flush=True)
        T = 1
        while T <= 8192:
            xs = {C: torch.randn(T, C, device="cuda", dtype=dt) for C in (4096, 11008)}
            arms = {
                "dense": lambda: [F.linear(xs[W.shape[1]], W) for W in Ws],
                "fused": lambda: [native.sparse24_linear(xs[W.shape[1]], v, m, W.shape[1]) for W, (v, m) in zip(Ws, comp)],
                "expand": lambda: [F.linear(xs[W.shape[1]], native.sparse24_decompress(
                    v, m, W.shape[1], out=scratch[:W.numel()].view(W.shape))) for W, (v, m) in zip(Ws, comp)],
            }
            for fn in arms.values():
                for _ in range(3):
                    fn()
            # warm up on the capture stream too: the library's per-stream workspace reaches this T's size before the
            # capture, so no buffer a captured kernel points to is replaced (freed) while capturing
            with torch.cuda.stream(cap):
                for fn in arms.values():
                    fn()
            torch.cuda.synchronize()
            graphs = []
            for k in list(arms):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=cap):
                    arms[k]()
                graphs.append(g)
                arms[k + "_graph"] = g.replay
                for _ in range(2):
                    g.replay()
            times = {k: [] for k in arms}
            order = list(arms)
            for r in range(args.reps):
                for k in (order if r % 2 == 0 else order[::-1]):
                    times[k].append(timed(arms[k]))
            act = sum(T * (R + C) * 2 for R, C in SHAPES)
            row = {"dtype": name, "T": T}
            for k in arms:
                row[k] = stats(times[k])
            md, mf, me = row["dense"]["median"], row["fused"]["median"], row["expand"]["median"]
            row["dense_gbs"] = (wbytes_dense + act) / md / 1e6
            row["fused_gbs"] = (wbytes_comp + act) / mf / 1e6
            row["speedup_fused_vs_dense"] = md / mf
            gd, gf, ge = row["dense_graph"]["median"], row["fused_graph"]["median"], row["expand_graph"]["median"]
            row["graph_dense_gbs"] = (wbytes_dense + act) / gd / 1e6
            row["graph_fused_gbs"] = (wbytes_comp + act) / gf / 1e6
            row["graph_speedup_fused_vs_dense"] = gd / gf
            res["rows"].append(row)
            print(f"{name:6s} {T:5d}  {md:8.3f}  {mf:8.3f}  {me:9.3f}  {md / mf:10.2f}x  {row['dense_gbs']:8.0f} "
                  f"{row['fused_gbs']:8.0f} ({row['dense_gbs'] / peak:.2f} / {row['fused_gbs'] / peak:.2f})  "
                  f"spread fused {row['fused']['min']:.3f}-{row['fused']['max']:.3f} dense "
                  f"{row['dense']['min']:.3f}-{row['dense']['max']:.3f}", flush=True)
            print(f"{name:6s} {T:5d}  graph: dense {gd:.3f} fused {gf:.3f} expand {ge:.3f} ms  fused/dense {gd / gf:.2f}x  "
                  f"GB/s dense {row['graph_dense_gbs']:.0f} fused {row['graph_fused_gbs']:.0f} "
                  f"({row['graph_dense_gbs'] / peak:.2f} / {row['graph_fused_gbs'] / peak:.2f} of copy peak)  spread fused "
                  f"{row['fused_graph']['min']:.3f}-{row['fused_graph']['max']:.3f} dense "
                  f"{row['dense_graph']['min']:.3f}-{row['dense_graph']['max']:.3f}", flush=True)
            T *= 2
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
