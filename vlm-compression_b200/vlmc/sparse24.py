"""Inference on compressed 2:4 weights (format: include/vlmc.h, "Compressed 2:4 weights").

A model pruned to 2:4 (Wanda / SparseGPT / DSnoT with prune_n = 2, prune_m = 4) still holds dense weights with explicit
zeros.  `compress_model` swaps its 2:4 fp16 / bf16 `nn.Linear`s for `Sparse24Linear`, which keeps half the values and
one bit of index per weight (0.5625x the bytes) resident, and multiplies from that form:
  - below DENSE_EXPAND_MIN_TOKENS tokens: K26 reads the compressed weight and expands it on chip;
  - from DENSE_EXPAND_MIN_TOKENS tokens on: K25 expands the weight into a scratch buffer shared by all layers on the
    stream, then the library GEMM runs on it.
Both give y = F.linear(x, W, bias) of the dense pruned weight W within the library GEMM's error; the second bit for bit.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from vlmc import native

# Token count from which expand + library GEMM is faster than K26 on a Vicuna-7B block.  Measured on a B200 (1000 W
# limit), fp16 and bf16, T = 1 .. 8192 (profiles/r03_sparse24_probe.log): expand wins at every T (graph replay, T = 1:
# 0.26 against 0.34 ms per block; T = 16: 0.23 against 0.75 ms), so K26 takes no call here until it beats it.
DENSE_EXPAND_MIN_TOKENS = 1

_scratch = {}


def _dense_scratch(ref, R, C):
    """One dense [R, C] buffer per (device, stream, dtype), grown to the largest layer: stream order keeps the K25
    write of one layer behind the GEMM that read the previous one."""
    key = (ref.device.index, native._stream(ref), ref.dtype)
    buf = _scratch.get(key)
    if buf is None or buf.numel() < R * C:
        buf = torch.empty(R * C, dtype=ref.dtype, device=ref.device)
        _scratch[key] = buf
    return buf[:R * C].view(R, C)


class Sparse24Linear(nn.Module):
    """Inference-only linear layer on a compressed 2:4 weight: buffers `values` [R, C/2], `meta` [R, C/16] (int16 holding
    the uint16 index words) and optional `bias` [R]."""

    def __init__(self, values, meta, in_features, bias=None):
        super().__init__()
        native._sparse24_operands(values, meta, in_features)
        self.in_features = int(in_features)
        self.out_features = values.shape[0]
        self.register_buffer("values", values)
        self.register_buffer("meta", meta)
        self.register_buffer("bias", bias)

    @classmethod
    def from_linear(cls, linear):
        """Compresses linear.weight (raises ValueError if it is not 2:4)."""
        values, meta = native.sparse24_compress(linear.weight.detach())
        bias = None if linear.bias is None else linear.bias.detach().to(values.dtype).clone()
        return cls(values, meta, linear.in_features, bias)

    def to_dense(self):
        """An nn.Linear holding the expanded weight (+0 at pruned positions)."""
        lin = nn.Linear(self.in_features, self.out_features, bias=self.bias is not None,
                        device=self.values.device, dtype=self.values.dtype)
        with torch.no_grad():
            native.sparse24_decompress(self.values, self.meta, self.in_features, out=lin.weight.data)
            if self.bias is not None:
                lin.bias.copy_(self.bias)
        return lin

    def forward(self, x):
        if x.requires_grad and torch.is_grad_enabled():
            raise RuntimeError("Sparse24Linear is inference-only: run it under torch.no_grad() / inference_mode(), or "
                               "train on the dense layer (to_dense())")
        if x.dtype != self.values.dtype or x.shape[-1] != self.in_features:
            raise ValueError(f"Sparse24Linear takes [..., {self.in_features}] inputs in {self.values.dtype}, got "
                             f"{list(x.shape)} in {x.dtype}")
        tokens = x.numel() // self.in_features if self.in_features else 0
        if tokens < DENSE_EXPAND_MIN_TOKENS:
            return native.sparse24_linear(x, self.values, self.meta, self.in_features, self.bias)
        W = native.sparse24_decompress(self.values, self.meta, self.in_features,
                                       out=_dense_scratch(self.values, self.out_features, self.in_features))
        return F.linear(x, W, self.bias)

    def extra_repr(self):
        return f"in_features={self.in_features}, out_features={self.out_features}, bias={self.bias is not None}, 2:4"


def compress_model(model):
    """Replaces, in place, every nn.Linear of `model` whose weight is fp16 / bf16 on a CUDA device, 2:4 sparse and has
    in_features % 16 == 0 by a Sparse24Linear; every other linear stays dense (fp32 ViT linears, unpruned heads, LoRA
    layers).  Returns (replaced names, skipped names)."""
    replaced, skipped = [], []
    for name, mod in list(model.named_modules()):
        if not isinstance(mod, nn.Linear):
            continue
        w = mod.weight
        if (type(mod) is not nn.Linear or w.dtype not in (torch.float16, torch.bfloat16) or not w.is_cuda or
                mod.in_features % 16):
            skipped.append(name)
            continue
        try:
            new = Sparse24Linear.from_linear(mod)
        except ValueError:
            skipped.append(name)
            continue
        parent_name, _, child = name.rpartition(".")
        setattr(model.get_submodule(parent_name) if parent_name else model, child, new)
        replaced.append(name)
    return replaced, skipped
