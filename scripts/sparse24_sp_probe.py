"""The sparse tensor-core 2:4 linear (K31) against dense F.linear, expand (K25) + F.linear and K26 on the 7 linears of a
Vicuna-7B block, fp16 and bf16, T = 1 .. 16384 tokens.  Sets the vlmc.sparse24.SPARSE_MMA_{MIN,MAX}_TOKENS window and the
DESIGN.md K31 row.

    python scripts/sparse24_sp_probe.py [--reps 9] [--out sparse24_sp_probe.json] [--tokens 1,16,...]

One timed sample = the whole block (404 MB of dense / 227 MB of compressed weights, both far above the 126 MB L2, so a
weight is never read from L2 across samples); the four arms are alternated inside every repetition; CUDA events around
each arm; median, min and max over the repetitions.  Each arm is timed eager and replayed from a CUDA graph of the
block's 7 calls (every arm warmed up on the capture stream first).  TFLOP/s are quoted on the dense-equivalent flop
2 T R C and on the flop the sparse tensor cores execute (half of it).  Peak memory of one block forward at T = 8192 is
measured for expand (dense scratch buffer) and for K31 (none).
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
TOKENS = [1, 16, 128, 512, 2048, 8192, 16384]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name()


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def stats(v):
    v = sorted(v)
    return {"median": v[len(v) // 2], "min": v[0], "max": v[-1]}


def peak_forward_mb(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fn()
    torch.cuda.synchronize()
    return (torch.cuda.max_memory_allocated() - base) / 1e6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--tokens", default=",".join(map(str, TOKENS)))
    ap.add_argument("--out", default=None, help="also write the rows as JSON here")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the probe measures the GPU; there is no CPU arm"
    torch.manual_seed(0)
    cap = torch.cuda.Stream()
    res = {"gpu": gpu_info(), "reps": args.reps, "rows": []}
    print(f"# {res['gpu']}", flush=True)
    flop_per_token = sum(2 * R * C for R, C in SHAPES)
    for dt in (torch.float16, torch.bfloat16):
        name = str(dt).replace("torch.", "")
        Ws, comp = [], []
        for R, C in SHAPES:
            W = torch.randn(R, C, device="cuda", dtype=dt) * 0.02
            keep = torch.rand(R, C // 4, 4, device="cuda").argsort(-1) < 2
            W = (W.view(R, C // 4, 4) * keep).view(R, C)
            Ws.append(W)
            comp.append(native.sparse24_compress(W))
        scratch = torch.empty(max(W.numel() for W in Ws), dtype=dt, device="cuda")
        print("dtype     T   dense_ms  expand_ms    k26_ms    k31_ms  k31/dense  k31/expand  (graph replay, median; "
              "TFLOP/s dense-equivalent | executed)", flush=True)
        for T in (int(t) for t in args.tokens.split(",")):
            xs = {C: torch.randn(T, C, device="cuda", dtype=dt) for C in (4096, 11008)}
            arms = {
                "dense": lambda: [F.linear(xs[W.shape[1]], W) for W in Ws],
                "expand": lambda: [F.linear(xs[W.shape[1]], native.sparse24_decompress(
                    v, m, W.shape[1], out=scratch[:W.numel()].view(W.shape))) for W, (v, m) in zip(Ws, comp)],
                "k26": lambda: [native.sparse24_linear(xs[W.shape[1]], v, m, W.shape[1]) for W, (v, m) in zip(Ws, comp)],
                "k31": lambda: [native.sparse24_linear_sp(xs[W.shape[1]], v, m, W.shape[1])
                                for W, (v, m) in zip(Ws, comp)],
            }
            for fn in arms.values():
                for _ in range(2):
                    fn()
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
                g.replay()
            torch.cuda.synchronize()
            times = {k: [] for k in arms}
            order = list(arms)
            for r in range(args.reps):
                for k in (order if r % 2 == 0 else order[::-1]):
                    times[k].append(timed(arms[k]))
            row = {"dtype": name, "T": T}
            for k in arms:
                row[k] = stats(times[k])
                row[k + "_tflops_dense_equiv"] = T * flop_per_token / row[k]["median"] / 1e9
            row["k31_graph_tflops_executed"] = row["k31_graph_tflops_dense_equiv"] / 2
            g = {k: row[k + "_graph"]["median"] for k in ("dense", "expand", "k26", "k31")}
            row["graph_speedup_k31_vs_dense"] = g["dense"] / g["k31"]
            row["graph_speedup_k31_vs_expand"] = g["expand"] / g["k31"]
            res["rows"].append(row)
            print(f"{name:8s} {T:5d}  {g['dense']:8.3f}  {g['expand']:9.3f}  {g['k26']:8.3f}  {g['k31']:8.3f}  "
                  f"{g['dense'] / g['k31']:8.2f}x  {g['expand'] / g['k31']:9.2f}x  "
                  f"TFLOP/s dense {row['dense_graph_tflops_dense_equiv']:.0f} k31 "
                  f"{row['k31_graph_tflops_dense_equiv']:.0f} | {row['k31_graph_tflops_executed']:.0f}  spread k31 "
                  f"{row['k31_graph']['min']:.3f}-{row['k31_graph']['max']:.3f} dense "
                  f"{row['dense_graph']['min']:.3f}-{row['dense_graph']['max']:.3f}; eager dense "
                  f"{row['dense']['median']:.3f} expand {row['expand']['median']:.3f} k26 {row['k26']['median']:.3f} "
                  f"k31 {row['k31']['median']:.3f}", flush=True)
            del graphs
        if name == "float16":
            x8 = {C: torch.randn(8192, C, device="cuda", dtype=dt) for C in (4096, 11008)}
            scratch = None
            torch.cuda.empty_cache()
            from vlmc import sparse24
            sparse24._scratch.clear()
            mods = [sparse24.Sparse24Linear(v, m, W.shape[1]) for W, (v, m) in zip(Ws, comp)]
            with torch.no_grad():
                res["peak_mb_block_T8192_expand"] = peak_forward_mb(lambda: [mod(x8[mod.in_features]) for mod in mods])
                sparse24._scratch.clear()
                torch.cuda.empty_cache()
                res["peak_mb_block_T8192_k31"] = peak_forward_mb(
                    lambda: [native.sparse24_linear_sp(x8[mod.in_features], mod.values, mod.meta, mod.in_features)
                             for mod in mods])
            print(f"# peak memory above the resident weights and inputs, one block forward at T = 8192: expand "
                  f"{res['peak_mb_block_T8192_expand']:.1f} MB, K31 {res['peak_mb_block_T8192_k31']:.1f} MB", flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
