"""SparseLoRA linear layer: the slice of lavis/peft/src/peft/tuners/lora.py (:265-394) on the hot path.

Kept verbatim from the reference interface: `mask` (registered bool buffer, True = kept), `sparse`,
`scaling`, `lora_A`, `lora_B`, `fan_in_fan_out`, `merge()`, `forward(x, dense=False)`.
merge() + the re-mask of train.py:634-637 run as ONE kernel (vlmc_sparselora_merge, K14).
The masked training forward (lora.py:359-382, SURVEY 8f-2) builds its weight with ONE kernel per step
(vlmc_sparselora_effective_weight, K15) instead of ~5 elementwise passes over [R, C], and its backward gets the LoRA
gradients from vlmc_sparselora_lora_grads (K16); the two dense GEMMs of a step stay library GEMMs.  With
VLMC_LORA_FUSED=1 the forward is ONE kernel (vlmc_sparselora_linear_forward, K23: the effective weight is built on chip in
front of tcgen05 and never written to HBM) - measured slower than K15 + cuBLAS on a B200, hence opt-in.
"""
import math
import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from vlmc import native


def transpose(weight, fan_in_fan_out):
    return weight.T if fan_in_fan_out else weight


def _use_fused(x, W, mask, rank):
    """K23 (one fused kernel) or K15 + library GEMM (default).  VLMC_LORA_FUSED=1 selects K23 when the layer is 16-bit
    and its pitches are TMA-compatible.  It is opt-in: on a B200 the fused kernel measured 1.2-2.7x SLOWER than K15 +
    cuBLAS at every SparseLoRA shape (DESIGN.md K23: re-deriving the effective weight in front of the tensor core costs
    one K15 pass per 512 tokens, and the 128 x 128 single-CTA MMA shape is shared-memory bound)."""
    if os.environ.get("VLMC_LORA_FUSED", "0") != "1" or not native.sparselora_linear_forward_supported(x, W, mask, rank):
        return False
    if torch.is_autocast_enabled() and torch.get_autocast_dtype("cuda") != W.dtype:
        return False                       # F.linear would run in the autocast dtype: keep the reference's behaviour
    return True


class DenseWeightSource:
    """Where _MaskedLoRALinear gets W_eff and the LoRA gradients for a dense frozen weight W and a bool mask M:
    K15 and K16.  vlmc.sparse24 has the compressed 2:4 source (K28 / K29), which takes (values, meta) in their place."""
    fused = True                           # K23 (VLMC_LORA_FUSED=1) reads this form

    @staticmethod
    def effective_weight(W, mask, A, B, scaling, sparse):
        return native.sparselora_effective_weight(W, A, B, scaling, mask, sparse)

    @staticmethod
    def lora_grads(G, mask, A, B, scaling, sparse):
        return native.sparselora_lora_grads(G, A, B, scaling, mask, sparse)


class _MaskedLoRALinear(torch.autograd.Function):
    """y = F.linear(x, W_eff, bias) with W_eff = (W + s*BA) * M (sparse) or W * M + s*BA (lora.py:364-375).
    W_eff is rebuilt in backward (one K15 pass) instead of being kept alive between forward and backward.  `source`
    (DenseWeightSource or a compressed one) says how W and mask are stored."""

    # custom_fwd / custom_bwd: backward runs under the autocast state of forward, so with fp32 LoRA'd weights under
    # maybe_autocast(), or fp16 weights under bf16 autocast, gy (autocast dtype) meets w_eff (weight dtype) inside an
    # autocast region exactly like the reference's plain-autograd F.linear does
    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda")
    def forward(ctx, x, W, A, B, bias, mask, scaling, sparse, source):
        Af, Bf = A.detach().float(), B.detach().float()
        ctx.save_for_backward(x, W, A, B, mask)
        ctx.scaling, ctx.sparse, ctx.has_bias, ctx.source = scaling, sparse, bias is not None, source
        ctx.bias_dtype = bias.dtype if bias is not None else None
        if source.fused and _use_fused(x, W, mask, Af.shape[0]):
            # K23: the effective weight is built on chip, slice by slice, in front of the tensor core - nothing dense is
            # written to HBM.  Same operand bits as K15 (test_lora_linear_fused_operand_is_k15_bit_exact).
            return native.sparselora_linear_forward(x, W.detach(), Af, Bf, scaling, mask, sparse, bias=bias)
        w_eff = source.effective_weight(W.detach(), mask, Af, Bf, scaling, sparse)
        return F.linear(x, w_eff, bias)

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, gy):
        x, W, A, B, mask = ctx.saved_tensors
        Af, Bf = A.detach().float(), B.detach().float()
        gx = dA = dB = gbias = None
        gy2 = gy.reshape(-1, gy.shape[-1])
        if ctx.needs_input_grad[0]:
            w_eff = ctx.source.effective_weight(W.detach(), mask, Af, Bf, ctx.scaling, ctx.sparse)
            gx = (gy2 @ (w_eff if w_eff.dtype == gy2.dtype or torch.is_autocast_enabled() else w_eff.to(gy2.dtype)))
            gx = gx.reshape(x.shape).to(x.dtype)
        if ctx.needs_input_grad[2] or ctx.needs_input_grad[3]:
            G = gy2.t() @ x.reshape(-1, x.shape[-1]).to(gy2.dtype)          # dL/dW_eff, in the layer's dtype like autograd
            if G.dtype != W.dtype:
                G = G.to(W.dtype)
            dA, dB = ctx.source.lora_grads(G.contiguous(), mask, Af, Bf, ctx.scaling, ctx.sparse)
            dA, dB = dA.to(A.dtype), dB.to(B.dtype)
        if ctx.has_bias and ctx.needs_input_grad[4]:
            gbias = gy2.sum(0).to(ctx.bias_dtype)
        return gx, None, dA, dB, gbias, None, None, None, None


class LoraLayer:
    def __init__(self, r, lora_alpha, lora_dropout, merge_weights):
        self.r = r
        self.lora_alpha = lora_alpha
        self.lora_dropout = nn.Dropout(p=lora_dropout) if lora_dropout > 0.0 else (lambda x: x)
        self.merged = False
        self.merge_weights = merge_weights
        self.disable_adapters = False


class Linear(nn.Linear, LoraLayer):
    def __init__(self, in_features, out_features, r=0, lora_alpha=1, lora_dropout=0.0, fan_in_fan_out=False,
                 merge_weights=True, **kwargs):
        nn.Linear.__init__(self, in_features, out_features, **kwargs)
        LoraLayer.__init__(self, r=r, lora_alpha=lora_alpha, lora_dropout=lora_dropout, merge_weights=merge_weights)
        self.fan_in_fan_out = fan_in_fan_out
        if r > 0:
            self.lora_A = nn.Linear(in_features, r, bias=False)
            self.lora_B = nn.Linear(r, out_features, bias=False)
            self.scaling = self.lora_alpha / self.r
            self.weight.requires_grad = False
        self.reset_parameters()
        if fan_in_fan_out:
            self.weight.data = self.weight.data.T
        self.register_buffer("mask", torch.ones_like(self.weight.data).bool())   # lora.py:317
        self.sparse = False

    def reset_parameters(self):
        nn.Linear.reset_parameters(self)
        self.reset_peft()

    def reset_peft(self):
        if hasattr(self, "lora_A"):
            nn.init.kaiming_uniform_(self.lora_A.weight, a=math.sqrt(5))
            nn.init.zeros_(self.lora_B.weight)

    def _merge_dense_delta(self, sign):
        """W += sign * scaling * B@A on the whole matrix (lora.py:340-353: train(False) merges WITHOUT the mask)."""
        if self.fan_in_fan_out:
            raise NotImplementedError("fan_in_fan_out weights are not on the InstructBLIP path")
        native.sparselora_merge(self.weight.data, self.lora_A.weight.data.float(), self.lora_B.weight.data.float(),
                                sign * self.scaling, torch.ones_like(self.mask), remask=False)

    def train(self, mode=True):
        """lora.py:334-353: with merge_weights, train(False) folds B@A into W and marks the layer merged (the plain
        F.linear path then runs), train(True) takes it out again."""
        nn.Linear.train(self, mode)
        if hasattr(self, "lora_A"):
            self.lora_A.train(mode)
            self.lora_B.train(mode)
        if not mode and self.merge_weights and not self.merged:
            if self.r > 0:
                self._merge_dense_delta(+1.0)
            self.merged = True
        elif self.merge_weights and self.merged:
            if self.r > 0:
                self._merge_dense_delta(-1.0)
            self.merged = False
        return self

    def eval(self):
        """lora.py:355-358: only flips the training flags (no merge, unlike train(False))."""
        nn.Linear.train(self, False)
        if hasattr(self, "lora_A"):
            self.lora_A.train(False)
            self.lora_B.train(False)
        return self

    def forward(self, x, dense=False):
        previous_dtype = self.weight.dtype
        if dense or self.disable_adapters or not (self.r > 0 and not self.merged):
            result = F.linear(x, transpose(self.weight, self.fan_in_fan_out), bias=self.bias)
        else:
            # one fused kernel builds the masked, LoRA-corrected weight (K15); K16 serves the backward.  No host path.
            if self.fan_in_fan_out or self.r > 16:
                raise NotImplementedError("fan_in_fan_out layouts and ranks above 16 are not on the InstructBLIP path")
            if not self.weight.is_cuda:
                raise RuntimeError("vlmc has no CPU path: the masked LoRA forward needs CUDA tensors "
                                   f"(got device {self.weight.device})")
            if x.dtype != previous_dtype and not torch.is_autocast_enabled():
                x = x.to(previous_dtype)
            result = _MaskedLoRALinear.apply(x, self.weight,
                                             self.lora_A.weight, self.lora_B.weight, self.bias, self.mask,
                                             float(self.scaling), bool(self.sparse), DenseWeightSource)
        if result.dtype != previous_dtype:
            result = result.to(previous_dtype)
        return result

    def merge(self, remask=False):
        """lora.py:384-394.  sparse: W += (B@A * scaling) * mask, one fused kernel; remask=True also
        applies train.py:634-637 (W[~mask] = 0) in the same pass."""
        if self.fan_in_fan_out:
            raise NotImplementedError("fan_in_fan_out weights are not on the InstructBLIP path")
        if self.sparse:
            native.sparselora_merge(self.weight.data, self.lora_A.weight.data.float(),
                                    self.lora_B.weight.data.float(), self.scaling, self.mask, remask=remask)
        else:
            # dense-delta branch (lora.py:388-391): W[~mask] = 0 ; W += B@A * scaling  -- same kernel run
            # with an all-ones merge mask after the re-mask
            native.sparselora_merge(self.weight.data, self.lora_A.weight.data.float(),
                                    self.lora_B.weight.data.float(), 0.0, self.mask, remask=True)       # W[~mask] = 0
            self._merge_dense_delta(+1.0)
        self.reset_peft()


def merge_all(modules, remask=False):
    """Linear.merge() for many SparseLoRA linears at once (train.py:626-637 loops over the modules): the sparse ones go
    through vlmc_sparselora_merge_batch, 16 per launch and dtype; the rest merge one by one.  Same results as calling
    merge() on each module."""
    batch = {}
    for m in modules:
        if m.sparse and not m.fan_in_fan_out and m.r <= 8 and m.weight.is_cuda:
            batch.setdefault((m.weight.dtype, m.weight.device), []).append(m)
        else:
            m.merge(remask=remask)
    for ms in batch.values():
        native.sparselora_merge_batch([m.weight.data for m in ms], [m.lora_A.weight.data.float() for m in ms],
                                      [m.lora_B.weight.data.float() for m in ms], [m.scaling for m in ms],
                                      [m.mask for m in ms], remask=remask)
        for m in ms:
            m.reset_peft()
