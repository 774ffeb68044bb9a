"""SparseLoRA fine-tuning on compressed 2:4 weights against the dense SparseLoRA layer, on the 7 linears of a Vicuna-7B
block (r = 8, sparse=True), fp16 and bf16, T = 2048 / 8192 / 16384 tokens per step.  Sets the DESIGN.md K27-K30 rows.

    python scripts/sparse24_lora_probe.py [--reps 10] [--out sparse24_lora_probe.json]

Per block and dtype:
  - K15 against K28 (the masked training weight) and K16 against K29 (the LoRA gradients), the 7 calls of the block per
    sample; GB/s on algorithmic bytes: K15 5 B / weight (W + mask in, W_eff out), K28 3.125 B / weight (values + meta in,
    W_eff out), K16 6 B / weight (two reads of G + mask), K29 4.25 B / weight (two reads of G + meta);
  - forward + backward of the 7 layers (vlmc.peft.lora.Linear against vlmc.sparse24.Sparse24LoRALinear), per T;
  - resident frozen-weight bytes, and torch.cuda.max_memory_allocated over one step with only that arm's layers resident.
Dense and compressed arms alternate inside every repetition; CUDA events around each arm; median, min and max.  The
block's weights (607 MB dense + mask, 228 MB compressed) are far above the 126 MB L2.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "vlm-compression_b200"))
from vlmc import native  # noqa: E402
from vlmc.peft.lora import Linear  # noqa: E402
from vlmc.sparse24 import Sparse24LoRALinear  # noqa: E402

SHAPES = [(4096, 4096)] * 4 + [(11008, 4096)] * 2 + [(4096, 11008)]      # q k v o, gate up, down  (R, C)
RANK = 8
TOKENS = (2048, 8192, 16384)


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


def dense_block(dt):
    layers = []
    for R, C in SHAPES:
        lin = Linear(C, R, r=RANK, lora_alpha=16, bias=False, device="cuda", dtype=dt)
        lin.lora_A.cuda(); lin.lora_B.cuda()
        lin.lora_B.weight.data.normal_(0, 0.02)
        with torch.no_grad():
            lin.weight.normal_(0, 0.02)
            lin.mask, _ = native.wanda_nm(lin.weight, torch.rand(C, device="cuda") + 0.1, 2, 4, zero_w=False)
        lin.sparse = True
        layers.append(lin)
    return layers


def step(layers, xs, gys):
    for lin, x, gy in zip(layers, xs, gys):
        lin(x).backward(gy)


def step_peak(layers, xs, gys):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    step(layers, xs, gys)
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the rows as JSON here")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the probe measures the GPU; there is no CPU arm"
    torch.manual_seed(0)
    res = {"gpu": gpu_info(), "reps": args.reps, "rank": RANK, "rows": []}
    print(f"# {res['gpu']}", flush=True)
    nweights = sum(R * C for R, C in SHAPES)
    for dt in (torch.float16, torch.bfloat16):
        tag = str(dt).split(".")[-1]
        # ---- memory: one arm resident at a time
        dense = dense_block(dt)
        Tm = TOKENS[-1]
        xs = [torch.randn(Tm, C, device="cuda", dtype=dt, requires_grad=True) for _, C in SHAPES]
        gys = [torch.randn(Tm, R, device="cuda", dtype=dt) * 1e-3 for R, _ in SHAPES]
        res_dense = sum(m.weight.numel() * m.weight.element_size() + m.mask.numel() for m in dense)
        step(dense, xs, gys)
        peak_dense = step_peak(dense, xs, gys)
        comp = [Sparse24LoRALinear.from_lora_linear(m) for m in dense]
        del dense
        res_comp = sum(m.values.numel() * 2 + m.meta.numel() * 2 for m in comp)
        step(comp, xs, gys)
        peak_comp = step_peak(comp, xs, gys)
        del xs, gys
        dense = [m.to_lora_linear() for m in comp]               # back to dense for the timed arms (same masks)
        mem = {"dtype": tag, "kind": "memory", "T": Tm, "resident_dense_bytes": res_dense,
               "resident_comp_bytes": res_comp, "step_peak_dense_bytes": peak_dense, "step_peak_comp_bytes": peak_comp}
        res["rows"].append(mem)
        print(f"{tag} resident frozen weights: dense+mask {res_dense / 1e6:.1f} MB, compressed {res_comp / 1e6:.1f} MB; "
              f"max_memory_allocated over a T={Tm} step, one arm resident: dense {peak_dense / 1e6:.1f} MB, "
              f"compressed {peak_comp / 1e6:.1f} MB", flush=True)

        # ---- kernels: K15 vs K28, K16 vs K29 over the block
        As = [m.lora_A.weight.data for m in dense]
        Bs = [m.lora_B.weight.data for m in dense]
        outs = [torch.empty(R, C, device="cuda", dtype=dt) for R, C in SHAPES]
        Gs = [torch.randn(R, C, device="cuda", dtype=dt) for R, C in SHAPES]

        def k15():
            for m, A, B, o in zip(dense, As, Bs, outs):
                native.sparselora_effective_weight(m.weight, A, B, 2.0, m.mask, True, out=o)

        def k28():
            for m, A, B, o in zip(comp, As, Bs, outs):
                native.sparse24_lora_effective_weight(m.values, m.meta, m.in_features, A, B, 2.0, True, out=o)

        def k16():
            for m, A, B, G in zip(dense, As, Bs, Gs):
                native.sparselora_lora_grads(G, A, B, 2.0, m.mask, True)

        def k29():
            for m, A, B, G in zip(comp, As, Bs, Gs):
                native.sparse24_lora_grads(G, m.meta, A, B, 2.0, True)

        arms = {"k15": k15, "k28": k28, "k16": k16, "k29": k29}
        for f in arms.values():
            f(); f()
        t = {k: [] for k in arms}
        for _ in range(args.reps):
            for k, f in arms.items():
                t[k].append(timed(f))
        bpw = {"k15": 5.0, "k28": 3.125, "k16": 6.0, "k29": 4.25}
        krow = {"dtype": tag, "kind": "kernels"}
        for k in arms:
            s = stats(t[k])
            krow[k] = {**s, "gbs": bpw[k] * nweights / s["median"] / 1e6}
        res["rows"].append(krow)
        print(f"{tag} block K15 {krow['k15']['median']:.3f} ms ({krow['k15']['gbs']:.0f} GB/s) | K28 "
              f"{krow['k28']['median']:.3f} ms ({krow['k28']['gbs']:.0f} GB/s) | K16 {krow['k16']['median']:.3f} ms "
              f"({krow['k16']['gbs']:.0f} GB/s) | K29 {krow['k29']['median']:.3f} ms ({krow['k29']['gbs']:.0f} GB/s)  "
              f"[min/max K28 {krow['k28']['min']:.3f}/{krow['k28']['max']:.3f}, K15 {krow['k15']['min']:.3f}/"
              f"{krow['k15']['max']:.3f}]", flush=True)
        del outs, Gs

        # ---- forward + backward of the 7 layers
        for T in TOKENS:
            xs = [torch.randn(T, C, device="cuda", dtype=dt, requires_grad=True) for _, C in SHAPES]
            gys = [torch.randn(T, R, device="cuda", dtype=dt) * 1e-3 for R, _ in SHAPES]
            for _ in range(2):
                step(dense, xs, gys); step(comp, xs, gys)
            td, tc = [], []
            for _ in range(args.reps):
                td.append(timed(lambda: step(dense, xs, gys)))
                tc.append(timed(lambda: step(comp, xs, gys)))
            row = {"dtype": tag, "kind": "step", "T": T, "dense_ms": stats(td), "comp_ms": stats(tc)}
            res["rows"].append(row)
            print(f"{tag} T={T:5d} fwd+bwd block: dense {row['dense_ms']['median']:.3f} ms "
                  f"[{row['dense_ms']['min']:.3f}, {row['dense_ms']['max']:.3f}] | compressed "
                  f"{row['comp_ms']['median']:.3f} ms [{row['comp_ms']['min']:.3f}, {row['comp_ms']['max']:.3f}] | "
                  f"ratio {row['comp_ms']['median'] / row['dense_ms']['median']:.3f}", flush=True)
            del xs, gys
        del dense, comp
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
