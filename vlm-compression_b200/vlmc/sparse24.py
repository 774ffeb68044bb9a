"""Inference on compressed 2:4 weights (format: include/vlmc.h, "Compressed 2:4 weights").

A model pruned to 2:4 (Wanda / SparseGPT / DSnoT with prune_n = 2, prune_m = 4) still holds dense weights with explicit
zeros.  `compress_model` swaps its 2:4 fp16 / bf16 `nn.Linear`s for `Sparse24Linear`, which keeps half the values and
one bit of index per weight (0.5625x the bytes) resident, and multiplies from that form:
  - below DENSE_EXPAND_MIN_TOKENS tokens: K26 reads the compressed weight and expands it on chip;
  - from DENSE_EXPAND_MIN_TOKENS tokens on: K25 expands the weight into a scratch buffer shared by all layers on the
    stream, then the library GEMM runs on it.
Both give y = F.linear(x, W, bias) of the dense pruned weight W within the library GEMM's error; the second bit for bit.
With sparse_mma=True (opt-in), calls of SPARSE_MMA_MIN_TOKENS <= tokens < SPARSE_MMA_MAX_TOKENS whose in_features is a
multiple of 32 go to K31 instead, which multiplies values and meta as stored on the sparse tensor cores: no dense scratch buffer, and only
the positions meta names take part (an inf / NaN of x at a pruned position does not reach y; include/vlmc.h).

SparseLoRA recovery fine-tuning after 2:4 pruning (prune(lora_model=True) -> train the adapters -> merge + re-mask ->
save) runs on the same format: `Sparse24LoRALinear` holds the frozen weight as values + meta compressed from the layer's
mask (K27), builds the masked training weight from them (K28), gets the LoRA gradients with the mask read from meta
(K29) and merges in place (K30) - 1.125 B per frozen weight resident instead of the dense weight and bool mask's 3 B.
"""
import math

import torch
import torch.nn as nn
import torch.nn.functional as F

from vlmc import native
from vlmc.peft import lora as peft_lora

# Token count from which expand + library GEMM is faster than K26 on a Vicuna-7B block.  Measured on a B200 (1000 W
# limit), fp16 and bf16, T = 1 .. 8192 (profiles/r03_sparse24_probe.log): expand wins at every T (graph replay, T = 1:
# 0.26 against 0.34 ms per block; T = 16: 0.23 against 0.75 ms), so K26 takes no call here until it beats it.
DENSE_EXPAND_MIN_TOKENS = 1

# Token window in which layers built with sparse_mma=True take K31 (sparse tensor cores) instead of expand + GEMM.
# Measured on a B200 (1000 W limit), Vicuna-7B block, graph replay (profiles/r05_sparse24_sp_probe.log): K31 beats expand
# at T = 1 .. 512 (1.44x at T = 1, 1.09x at T = 512) and loses from T = 2048 (0.97x; 0.86x at T = 16384).
SPARSE_MMA_MIN_TOKENS = 1
SPARSE_MMA_MAX_TOKENS = 2048

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

    def __init__(self, values, meta, in_features, bias=None, sparse_mma=False):
        super().__init__()
        native._sparse24_operands(values, meta, in_features)
        self.in_features = int(in_features)
        self.out_features = values.shape[0]
        self.sparse_mma = bool(sparse_mma)          # a routing choice, not state: state_dict() does not hold it
        self.register_buffer("values", values)
        self.register_buffer("meta", meta)
        self.register_buffer("bias", bias)

    @classmethod
    def from_linear(cls, linear, sparse_mma=False):
        """Compresses linear.weight (raises ValueError if it is not 2:4)."""
        values, meta = native.sparse24_compress(linear.weight.detach())
        bias = None if linear.bias is None else linear.bias.detach().to(values.dtype).clone()
        return cls(values, meta, linear.in_features, bias, sparse_mma)

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
        if (self.sparse_mma and SPARSE_MMA_MIN_TOKENS <= tokens < SPARSE_MMA_MAX_TOKENS and
                native.sparse24_linear_sp_supported(x, self.values, self.meta, self.in_features)):
            return native.sparse24_linear_sp(x, self.values, self.meta, self.in_features, self.bias)
        if tokens < DENSE_EXPAND_MIN_TOKENS:
            return native.sparse24_linear(x, self.values, self.meta, self.in_features, self.bias)
        W = native.sparse24_decompress(self.values, self.meta, self.in_features,
                                       out=_dense_scratch(self.values, self.out_features, self.in_features))
        return F.linear(x, W, self.bias)

    def extra_repr(self):
        return (f"in_features={self.in_features}, out_features={self.out_features}, bias={self.bias is not None}, 2:4, "
                f"sparse_mma={self.sparse_mma}")


class _Sparse24WeightSource:
    """vlmc.peft.lora._MaskedLoRALinear's weight source for a mask-driven compressed weight: (values, meta) in place of
    (W, mask).  W_eff goes to the per-stream scratch buffer: it is dead once the GEMM that reads it has run."""
    fused = False

    def __init__(self, in_features):
        self.in_features = in_features

    def effective_weight(self, values, meta, A, B, scaling, sparse):
        out = _dense_scratch(values, values.shape[0], self.in_features)
        return native.sparse24_lora_effective_weight(values, meta, self.in_features, A, B, scaling, sparse, out=out)

    def lora_grads(self, G, meta, A, B, scaling, sparse):
        return native.sparse24_lora_grads(G, meta, A, B, scaling, sparse)


def _dense_only(what):
    return NotImplementedError(f"Sparse24LoRALinear cannot {what}: that path uses the unmasked dense weight, which the "
                               "compressed layer does not keep.  Convert it back with to_lora_linear() first")


class Sparse24LoRALinear(nn.Module):
    """A SparseLoRA linear (vlmc.peft.lora.Linear) whose frozen weight is stored compressed: buffers `values` [R, C/2],
    `meta` [R, C/16] (int16 holding the uint16 index words; the kept set of meta is the layer's mask) and optional
    `bias` [R]; fp32 parameters `lora_A`, `lora_B` as in the dense layer.

    The masked training forward, its backward and merge() give the dense layer's results bit for bit (same kernels on the
    same operands, same library GEMMs).  What the compressed form cannot express raises and names to_lora_linear():
    forward(dense=True), disable_adapters, fan_in_fan_out, fp32 weights, and the dense-delta merge of sparse=False.
    The one divergence from vlmc.peft.lora.Linear: train(False) does not fold the unmasked delta s*B@A into the weight
    (lora.py:340-353), because a dense delta is not 2:4.  It only flips the training flags, and forward stays the masked
    one - which computes the same function the dense layer computes before that fold."""

    def __init__(self, values, meta, in_features, r, lora_alpha=1, sparse=True, bias=None, merge_weights=True):
        super().__init__()
        native._sparse24_operands(values, meta, in_features)
        if not 1 <= int(r) <= 16:
            raise ValueError(f"Sparse24LoRALinear takes ranks 1..16, got r = {r}")
        self.in_features = int(in_features)
        self.out_features = values.shape[0]
        self.register_buffer("values", values)
        self.register_buffer("meta", meta)
        self.register_buffer("bias", bias)
        self.r = int(r)
        self.lora_alpha = lora_alpha
        self.scaling = self.lora_alpha / self.r
        self.sparse = bool(sparse)
        self.merged = False
        self.merge_weights = merge_weights
        self.disable_adapters = False
        self.fan_in_fan_out = False
        self.lora_A = nn.Linear(self.in_features, self.r, bias=False, device=values.device)
        self.lora_B = nn.Linear(self.r, self.out_features, bias=False, device=values.device)
        self.reset_peft()
        self._source = _Sparse24WeightSource(self.in_features)

    @classmethod
    def from_lora_linear(cls, lin):
        """Compresses lin.weight at the positions of lin.mask (K27) and takes over its adapters, bias and flags.  Raises
        ValueError when the mask does not keep exactly two of every four columns."""
        if not isinstance(lin, peft_lora.Linear):
            raise TypeError(f"from_lora_linear takes a vlmc.peft.lora.Linear, got {type(lin).__name__}")
        if lin.fan_in_fan_out:
            raise _dense_only("hold a fan_in_fan_out weight")
        if lin.weight.dtype not in (torch.float16, torch.bfloat16):
            raise TypeError(f"compressed 2:4 weights are float16 / bfloat16, got {lin.weight.dtype}: keep the dense "
                            "vlmc.peft.lora.Linear (Sparse24LoRALinear.to_lora_linear() is the way back for compressed "
                            "layers)")
        if not 1 <= lin.r <= 16:
            raise ValueError(f"Sparse24LoRALinear takes ranks 1..16, got r = {lin.r}")
        if lin.merged:
            raise ValueError("the layer is merged (train(False) folded the unmasked delta into its weight)")
        values, meta = native.sparse24_compress_masked(lin.weight.detach(), lin.mask)
        bias = None if lin.bias is None else lin.bias.detach().clone()
        new = cls(values, meta, lin.in_features, lin.r, lin.lora_alpha, lin.sparse, bias, lin.merge_weights)
        with torch.no_grad():
            new.lora_A.weight.copy_(lin.lora_A.weight)
            new.lora_B.weight.copy_(lin.lora_B.weight)
        new.lora_A.weight.requires_grad_(lin.lora_A.weight.requires_grad)
        new.lora_B.weight.requires_grad_(lin.lora_B.weight.requires_grad)
        new.train(lin.training)
        return new

    def reset_peft(self):
        nn.init.kaiming_uniform_(self.lora_A.weight, a=math.sqrt(5))
        nn.init.zeros_(self.lora_B.weight)

    def train(self, mode=True):
        """Flips the training flags only (see the class docstring: no unmasked fold)."""
        return nn.Module.train(self, mode)

    def _dense_weight(self):
        return native.sparse24_decompress(self.values, self.meta, self.in_features,
                                          out=_dense_scratch(self.values, self.out_features, self.in_features))

    def forward(self, x, dense=False):
        if dense:
            raise _dense_only("run forward(dense=True)")
        if self.disable_adapters:
            raise _dense_only("run with disable_adapters")
        if self.fan_in_fan_out:
            raise _dense_only("hold a fan_in_fan_out weight")
        previous_dtype = self.values.dtype
        if self.merged:
            result = F.linear(x, self._dense_weight(), bias=self.bias)
        else:
            if x.dtype != previous_dtype and not torch.is_autocast_enabled():
                x = x.to(previous_dtype)
            result = peft_lora._MaskedLoRALinear.apply(x, self.values, self.lora_A.weight, self.lora_B.weight, self.bias,
                                                       self.meta, float(self.scaling), bool(self.sparse), self._source)
        if result.dtype != previous_dtype:
            result = result.to(previous_dtype)
        return result

    def merge(self, remask=True):
        """lora.py:384-394 + train.py:634-637 in place on the values (K30), then reset_peft().  The compressed form has no
        pruned weights to keep, so remask=False gives the same layer.  sparse=False raises: its dense-delta merge
        leaves a weight that is not 2:4."""
        if not self.sparse:
            raise _dense_only("merge a sparse=False layer (the dense-delta merge is not 2:4)")
        native.sparse24_lora_merge(self.values, self.meta, self.in_features, self.lora_A.weight.data.float(),
                                   self.lora_B.weight.data.float(), self.scaling)
        self.reset_peft()

    def to_sparse24_linear(self):
        """The inference layer on these values (after merge(): lora_B must be zero, or the adapters would be dropped)."""
        if bool(self.lora_B.weight.detach().ne(0).any()):
            raise ValueError("the adapters are not merged (lora_B is non-zero): call merge() first")
        bias = None if self.bias is None else self.bias.to(self.values.dtype)
        return Sparse24Linear(self.values, self.meta, self.in_features, bias)

    def to_lora_linear(self):
        """A dense vlmc.peft.lora.Linear with the expanded weight (+0 at pruned positions), the mask decoded from meta,
        these adapters, bias and flags."""
        dev, dt = self.values.device, self.values.dtype
        lin = peft_lora.Linear(self.in_features, self.out_features, r=self.r, lora_alpha=self.lora_alpha,
                               merge_weights=self.merge_weights, bias=self.bias is not None, device=dev, dtype=dt)
        lin.lora_A.to(dev)
        lin.lora_B.to(dev)
        with torch.no_grad():
            native.sparse24_decompress(self.values, self.meta, self.in_features, out=lin.weight.data)
            lin.mask.copy_(native.sparse24_decompress(torch.ones_like(self.values), self.meta, self.in_features) != 0)
            if self.bias is not None:
                lin.bias.copy_(self.bias)
            lin.lora_A.weight.copy_(self.lora_A.weight)
            lin.lora_B.weight.copy_(self.lora_B.weight)
        lin.lora_A.weight.requires_grad_(self.lora_A.weight.requires_grad)
        lin.lora_B.weight.requires_grad_(self.lora_B.weight.requires_grad)
        lin.sparse = self.sparse
        nn.Module.train(lin, self.training)          # flags only: Linear.train(False) would fold the delta
        return lin

    def extra_repr(self):
        return (f"in_features={self.in_features}, out_features={self.out_features}, bias={self.bias is not None}, "
                f"r={self.r}, sparse={self.sparse}, 2:4")


def _lora_swappable(mod):
    w = mod.weight
    return (w.dtype in (torch.float16, torch.bfloat16) and w.is_cuda and mod.in_features % 16 == 0 and
            1 <= mod.r <= 16 and not mod.merged and not mod.fan_in_fan_out and not mod.disable_adapters)


def compress_model(model, lora=False, sparse_mma=False):
    """Replaces, in place, every nn.Linear of `model` whose weight is fp16 / bf16 on a CUDA device, 2:4 sparse and has
    in_features % 16 == 0 by a Sparse24Linear; every other linear stays dense (fp32 ViT linears, unpruned heads, LoRA
    layers).  With lora=True every vlmc.peft.lora.Linear that is fp16 / bf16 on CUDA, has in_features % 16 == 0 and
    1 <= r <= 16, is not merged and whose mask keeps exactly two of every four columns becomes a Sparse24LoRALinear
    (its lora_A / lora_B go with it and are not listed).  sparse_mma is passed to every Sparse24Linear (see the module
    docstring).  Returns (replaced names, skipped names)."""
    replaced, skipped = [], []
    moved = []                                      # prefixes of swapped LoRA layers: their children went with them
    for name, mod in list(model.named_modules()):
        if not isinstance(mod, nn.Linear):
            continue
        if any(name.startswith(p) for p in moved):
            continue
        if lora and isinstance(mod, peft_lora.Linear):
            new = None
            if _lora_swappable(mod):
                try:
                    new = Sparse24LoRALinear.from_lora_linear(mod)
                except ValueError:
                    new = None
            if new is None:
                skipped.append(name)
                continue
            parent_name, _, child = name.rpartition(".")
            setattr(model.get_submodule(parent_name) if parent_name else model, child, new)
            replaced.append(name)
            moved.append(name + ".")
            continue
        w = mod.weight
        if (type(mod) is not nn.Linear or w.dtype not in (torch.float16, torch.bfloat16) or not w.is_cuda or
                mod.in_features % 16):
            skipped.append(name)
            continue
        try:
            new = Sparse24Linear.from_linear(mod, sparse_mma)
        except ValueError:
            skipped.append(name)
            continue
        parent_name, _, child = name.rpartition(".")
        setattr(model.get_submodule(parent_name) if parent_name else model, child, new)
        replaced.append(name)
    return replaced, skipped
