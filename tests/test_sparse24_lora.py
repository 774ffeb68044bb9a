"""SparseLoRA fine-tuning on compressed 2:4 weights (include/vlmc.h, K27-K30; vlmc.sparse24.Sparse24LoRALinear).

CPU: a numpy reference of the mask-driven compression rule (the kept set is the mask, exactly two per group, the values
keep W's bits there).  GPU: K27 against that reference bit for bit; K28 / K29 / K30 against the dense SparseLoRA
kernels K15 / K16 / K14 on the same weight and mask, bit for bit; the compressed layer against vlmc.peft.lora.Linear;
and a toy model fine-tuned compressed and dense side by side, then merged, saved and loaded.
"""
import copy

import numpy as np
import pytest
import torch

from oracle import sparse24 as oracle24

VICUNA = [(4096, 4096), (11008, 4096), (4096, 11008)]
DT = {"f16": torch.float16, "bf16": torch.bfloat16}
NAN = {"f16": 0x7E00, "bf16": 0x7FC0}
INF = {"f16": 0x7C00, "bf16": 0x7F80}


def ref_compress_masked(Wbits, mask):
    """Numpy reference of K27: uint16 bit patterns W [R, C] and a bool mask [R, C] -> (values uint16 [R, C/2], meta uint16
    [R, C/16]).  Every group of 4 columns must keep exactly two; the values are W's bits at the kept positions."""
    W, M = np.asarray(Wbits, np.uint16), np.asarray(mask, bool)
    R, C = W.shape
    assert C % 16 == 0 and M.shape == W.shape
    g, k = W.reshape(R, C // 4, 4), M.reshape(R, C // 4, 4)
    if (k.sum(-1) != 2).any():
        raise ValueError("mask is not 2:4")
    sel = np.sort(np.argsort(~k, axis=-1, kind="stable")[..., :2], axis=-1)
    values = np.take_along_axis(g, sel, -1).reshape(R, C // 2)
    nib = (sel[..., 0] | (sel[..., 1] << 2)).astype(np.uint16).reshape(R, C // 16, 4)
    meta = nib[..., 0] | (nib[..., 1] << 4) | (nib[..., 2] << 8) | (nib[..., 3] << 12)
    return values.astype(np.uint16), meta.astype(np.uint16)


def random_mask(R, C, seed):
    """Exactly two kept per group of 4, at random positions."""
    rng = np.random.default_rng(seed)
    order = np.argsort(rng.random((R, C // 4, 4)), axis=-1)
    keep = np.zeros((R, C // 4, 4), bool)
    np.put_along_axis(keep, order[..., :2], True, -1)
    return keep.reshape(R, C)


def random_bits(R, C, seed, tag, specials=True):
    """Unzeroed weight bits (what prune(lora_model=True) leaves) with +-0, NaN and +-inf sprinkled at random positions."""
    rng = np.random.default_rng(seed)
    w = torch.from_numpy(rng.standard_normal((R, C)).astype(np.float32) * 0.05).to(DT[tag])
    bits = w.view(torch.int16).numpy().view(np.uint16).copy()
    if specials:
        for v in (0, 0x8000, NAN[tag], INF[tag], INF[tag] | 0x8000):
            idx = rng.integers(0, R * C, size=max(1, R * C // 500))
            bits.reshape(-1)[idx] = v
    return bits


# ------------------------------------------------------------------------------------------- CPU: the reference's rules
@pytest.mark.parametrize("tag", ["f16", "bf16"])
@pytest.mark.parametrize("R,C", [(3, 16), (37, 176), (64, 1024)])
def test_ref_masked_round_trip(tag, R, C):
    W = random_bits(R, C, R * C, tag)
    M = random_mask(R, C, R + C)
    # the specials must also sit on kept positions
    W[M & (np.arange(R * C).reshape(R, C) % 7 == 0)] = NAN[tag]
    W[0, np.flatnonzero(M[0])[:2]] = [0x8000, INF[tag]]
    values, meta = ref_compress_masked(W, M)
    assert values.shape == (R, C // 2) and meta.shape == (R, C // 16)
    dense = oracle24.sparse24_decompress(values, meta)
    assert np.array_equal(dense, np.where(M, W, 0).astype(np.uint16))     # original bits on the mask, +0 off it
    nib = ((meta[..., None].astype(np.int64) >> (4 * np.arange(4))) & 15).reshape(R, C // 4)
    assert ((nib & 3) < (nib >> 2)).all()
    kept = np.zeros((R, C // 4, 4), bool)
    np.put_along_axis(kept, (nib & 3)[..., None], True, -1)
    np.put_along_axis(kept, (nib >> 2)[..., None], True, -1)
    assert np.array_equal(kept.reshape(R, C), M)                           # the kept set decoded from meta IS the mask


@pytest.mark.parametrize("count", [0, 1, 3, 4])
def test_ref_rejects_non_two_of_four(count):
    W = random_bits(8, 32, 1, "bf16", specials=False)
    M = random_mask(8, 32, 2)
    M[5, 8:12] = [i < count for i in range(4)]
    with pytest.raises(ValueError):
        ref_compress_masked(W, M)


# ------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def native(built_lib):
    from vlmc import native as n
    n.load()
    assert torch.cuda.is_available()
    return n


def bits_of(t):
    return t.contiguous().view(torch.int16).cpu().numpy().view(np.uint16)


def from_bits(bits, tag):
    return torch.from_numpy(np.ascontiguousarray(bits).view(np.int16)).view(DT[tag]).cuda()


def check_k27(native, W, M, tag):
    values, meta = native.sparse24_compress_masked(W, M)
    vo, mo = ref_compress_masked(bits_of(W), M.cpu().numpy())
    assert np.array_equal(bits_of(values), vo) and np.array_equal(bits_of(meta), mo)
    return values, meta


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["bf16", "f16"])
@pytest.mark.parametrize("R,C", VICUNA + [(328, 176)])
def test_k27_matches_reference(native, tag, R, C):
    W = from_bits(random_bits(R, C, R + C, tag), tag)
    M = torch.from_numpy(random_mask(R, C, 3 * R + C)).cuda()
    check_k27(native, W, M, tag)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["bf16", "f16"])
def test_k27_strided_and_misaligned_views(native, tag):
    R, C = 96, 352
    W = from_bits(random_bits(R, C + 9, 5, tag), tag)[:, 1:C + 1]            # pitch C + 9, base 2 bytes off
    Mbig = torch.zeros(R, C + 16, dtype=torch.bool, device="cuda")
    Mbig[:, 3:C + 3] = torch.from_numpy(random_mask(R, C, 6)).cuda()
    M = Mbig[:, 3:C + 3]                                                        # pitch C + 16, base 3 bytes off
    assert W.stride(0) == C + 9 and W.data_ptr() % 16 != 0 and M.data_ptr() % 16 != 0
    check_k27(native, W, M, tag)
    Wc = from_bits(random_bits(R, 2 * C, 7, tag), tag)[:, :C]                 # aligned, wider pitch
    Mc = torch.from_numpy(random_mask(R, 2 * C, 8)).cuda()[:, :C]
    check_k27(native, Wc, Mc, tag)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["bf16", "f16"])
@pytest.mark.parametrize("R,C", VICUNA)
def test_k27_wanda_lora_model_masks(native, tag, R, C):
    g = torch.Generator(device="cuda").manual_seed(R + C)
    W = (torch.randn(R, C, device="cuda", generator=g) * 0.02).to(DT[tag])
    W0 = W.clone()
    keep, _ = native.wanda_nm(W, torch.rand(C, device="cuda", generator=g) * 10, 2, 4, zero_w=False)
    assert torch.equal(W, W0)                                                   # lora_model=True: weights unzeroed
    values, meta = check_k27(native, W, keep, tag)
    assert torch.equal(native.sparse24_decompress(values, meta, C), W * keep)


@pytest.mark.gpu
@pytest.mark.parametrize("count", [1, 3])
def test_k27_rejects_and_leaves_w(native, count):
    R, C = 64, 128
    W = from_bits(random_bits(R, C, 9, "bf16"), "bf16")
    M = torch.from_numpy(random_mask(R, C, 10)).cuda()
    M[17, 40:44] = torch.tensor([i < count for i in range(4)])
    before = bits_of(W)
    with pytest.raises(ValueError, match="not 2:4"):
        native.sparse24_compress_masked(W, M)
    assert np.array_equal(bits_of(W), before)


_weights = {}


def lora_operands(R, C, rank, tag, seed):
    """W (unzeroed), a 2:4 mask M (one pair per (R, C, dtype), drawn on the GPU) and fresh fp32 A [rank, C], B [R, rank]."""
    if (R, C, tag) not in _weights:
        g = torch.Generator(device="cuda").manual_seed(R * 7 + C)
        W = (torch.randn(R, C, device="cuda", generator=g) * 0.05).to(DT[tag])
        order = torch.rand(R, C // 4, 4, device="cuda", generator=g).argsort(-1)
        M = torch.zeros(R, C // 4, 4, dtype=torch.bool, device="cuda").scatter_(-1, order[..., :2], True).view(R, C)
        _weights[(R, C, tag)] = (W, M)
    W, M = _weights[(R, C, tag)]
    g = torch.Generator(device="cuda").manual_seed(seed)
    A = torch.randn(rank, C, device="cuda", generator=g) * 0.05
    B = torch.randn(R, rank, device="cuda", generator=g) * 0.05
    return W, M, A, B


GRID = [(s, r, tag) for s in (0, 1) for r in (1, 2, 4, 8, 16) for tag in ("f16", "bf16")]


@pytest.mark.gpu
@pytest.mark.parametrize("sparse,rank,tag", GRID)
@pytest.mark.parametrize("R,C", [(11008, 4096), (328, 176)])
def test_k28_equals_k15(native, sparse, rank, tag, R, C):
    W, M, A, B = lora_operands(R, C, rank, tag, R + rank)
    values, meta = native.sparse24_compress_masked(W, M)
    want = native.sparselora_effective_weight(W, A, B, 1.7, M, sparse)
    got = native.sparse24_lora_effective_weight(values, meta, C, A, B, 1.7, sparse)
    assert np.array_equal(bits_of(got), bits_of(want))
    wide = torch.full((R, C + 24), 7.0, dtype=DT[tag], device="cuda")           # wider output pitch
    native.sparse24_lora_effective_weight(values, meta, C, A, B, 1.7, sparse, out=wide[:, :C])
    assert np.array_equal(bits_of(wide[:, :C]), bits_of(want)) and bool((wide[:, C:] == 7).all())


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f16", "bf16"])
def test_k28_zero_b_is_the_decompressed_weight(native, tag):
    # finite non-zero kept values: W + (+0) keeps their bits (a kept -0 would come back +0, a NaN canonicalised)
    R, C = 520, 1024
    W, M, A, B = lora_operands(R, C, 8, tag, 11)
    W = torch.where(W == 0, torch.ones_like(W), W)
    values, meta = native.sparse24_compress_masked(W, M)
    got = native.sparse24_lora_effective_weight(values, meta, C, A, torch.zeros_like(B), 2.0, True)
    assert np.array_equal(bits_of(got), bits_of(native.sparse24_decompress(values, meta, C)))


@pytest.mark.gpu
@pytest.mark.parametrize("sparse,rank,tag", GRID)
@pytest.mark.parametrize("R,C", [(11008, 4096), (328, 176)])
def test_k29_equals_k16(native, sparse, rank, tag, R, C):
    W, M, A, B = lora_operands(R, C, rank, tag, 2 * R + rank)
    _, meta = native.sparse24_compress_masked(W, M)
    G = (torch.randn(R, C, device="cuda") * 0.3).to(DT[tag])
    dA, dB = native.sparselora_lora_grads(G, A, B, 0.9, M, sparse)
    dA2, dB2 = native.sparse24_lora_grads(G, meta, A, B, 0.9, sparse)
    assert np.array_equal(dA.cpu().numpy().view(np.uint32), dA2.cpu().numpy().view(np.uint32))
    assert np.array_equal(dB.cpu().numpy().view(np.uint32), dB2.cpu().numpy().view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("rank,tag", [(r, t) for r in (1, 2, 4, 8, 16) for t in ("f16", "bf16")])
@pytest.mark.parametrize("R,C", [(11008, 4096), (328, 176)])
def test_k30_equals_k14_remask(native, rank, tag, R, C):
    W, M, A, B = lora_operands(R, C, rank, tag, 3 * R + rank)
    values, meta = native.sparse24_compress_masked(W, M)
    native.sparse24_lora_merge(values, meta, C, A, B, 1.3)
    want = native.sparselora_merge(W.clone(), A, B, 1.3, M, remask=True)
    assert np.array_equal(bits_of(native.sparse24_decompress(values, meta, C)), bits_of(want))


# ------------------------------------------------------------------------------------------- the layer
def dense_lora(R, C, r, tag, bias, seed):
    from vlmc import native
    from vlmc.peft.lora import Linear
    torch.manual_seed(seed)
    lin = Linear(C, R, r=r, lora_alpha=16, bias=bias).cuda().to(DT[tag])
    lin.lora_A.float(); lin.lora_B.float()
    lin.lora_B.weight.data.normal_(0, 0.05)
    with torch.no_grad():
        keep, _ = native.wanda_nm(lin.weight, torch.rand(C, device="cuda"), 2, 4, zero_w=False)
    lin.mask = keep
    lin.sparse = True
    return lin


def grads(mod, x):
    x = x.detach().clone().requires_grad_(True)
    for p in (mod.lora_A.weight, mod.lora_B.weight):
        p.grad = None
    y = mod(x)
    (y.float() * torch.linspace(-1, 1, y.shape[-1], device="cuda")).sum().backward()
    return y.detach(), x.grad, mod.lora_A.weight.grad.clone(), mod.lora_B.weight.grad.clone()


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["f16", "bf16"])
@pytest.mark.parametrize("bias", [False, True])
@pytest.mark.parametrize("shape", [(37, 256), (3, 50, 256)])
def test_layer_bit_identical_to_dense(native, tag, bias, shape):
    """Both layers run the same operand bits through the same library GEMMs (F.linear for y, gy @ W_eff for dx,
    gy^T x for G), so y, dx, dA and dB agree bit for bit."""
    from vlmc.sparse24 import Sparse24LoRALinear
    lin = dense_lora(328, 256, 8, tag, bias, 1)
    comp = Sparse24LoRALinear.from_lora_linear(lin)
    x = torch.randn(*shape, device="cuda").to(DT[tag])
    for a, b, nm in zip(grads(lin, x), grads(comp, x), ("y", "dx", "dA", "dB")):
        assert a.dtype == b.dtype and torch.equal(a, b), nm


@pytest.mark.gpu
@pytest.mark.parametrize("wdtype,acdtype", [(torch.float16, torch.bfloat16), (torch.bfloat16, torch.float16)])
def test_layer_under_autocast(native, wdtype, acdtype):
    """Weight dtype != autocast dtype: trains like the reference's plain-autograd expression (the tolerances of the dense
    layer's autocast test) and gives the dense layer's results."""
    from vlmc.sparse24 import Sparse24LoRALinear
    lin = dense_lora(40, 96, 4, "f16" if wdtype == torch.float16 else "bf16", False, 3)
    comp = Sparse24LoRALinear.from_lora_linear(lin)
    x = torch.randn(2, 7, 96, device="cuda", requires_grad=True)
    with torch.autocast("cuda", dtype=acdtype):
        y = comp(x)
        loss = (y.float() ** 2).sum()
    loss.backward()
    got = (y.detach().float(), x.grad.clone(), comp.lora_A.weight.grad.clone(), comp.lora_B.weight.grad.clone())
    x2 = x.detach().clone().requires_grad_(True)
    A, B = lin.lora_A.weight.detach().clone().requires_grad_(True), lin.lora_B.weight.detach().clone().requires_grad_(True)
    with torch.autocast("cuda", dtype=acdtype):
        w_eff = (lin.weight + (B @ A).to(wdtype) * lin.scaling) * lin.mask
        y2 = torch.nn.functional.linear(x2, w_eff, lin.bias)
        if y2.dtype != wdtype:
            y2 = y2.to(wdtype)
        loss2 = (y2.float() ** 2).sum()
    loss2.backward()
    tol = 3e-2 if acdtype == torch.bfloat16 else 5e-3
    for a, b, nm in zip(got, (y2.detach().float(), x2.grad, A.grad, B.grad), ("y", "dx", "dA", "dB")):
        assert a.dtype == b.dtype or nm == "y", nm
        err = float((a.float() - b.float()).abs().max() / b.float().abs().max().clamp_min(1e-6))
        assert err < tol, (nm, err)
    x3 = x.detach().clone().requires_grad_(True)
    with torch.autocast("cuda", dtype=acdtype):
        y3 = lin(x3)
        (y3.float() ** 2).sum().backward()
    assert torch.equal(y3, y) and torch.equal(x3.grad, got[1])


@pytest.mark.gpu
def test_layer_rejections_and_train_false(native):
    from vlmc.peft.lora import Linear
    from vlmc.sparse24 import Sparse24LoRALinear
    lin = dense_lora(64, 128, 4, "bf16", True, 5)
    comp = Sparse24LoRALinear.from_lora_linear(lin)
    x = torch.randn(9, 128, device="cuda").bfloat16()
    with pytest.raises(NotImplementedError, match="to_lora_linear"):
        comp(x, dense=True)
    comp.disable_adapters = True
    with pytest.raises(NotImplementedError, match="to_lora_linear"):
        comp(x)
    comp.disable_adapters = False
    comp.fan_in_fan_out = True
    with pytest.raises(NotImplementedError, match="to_lora_linear"):
        comp(x)
    comp.fan_in_fan_out = False
    fp32 = Linear(128, 64, r=4).cuda()
    fp32.mask = lin.mask.clone()
    with pytest.raises(TypeError, match="to_lora_linear"):
        Sparse24LoRALinear.from_lora_linear(fp32)
    comp.sparse = False
    with pytest.raises(NotImplementedError, match="to_lora_linear"):
        comp.merge()
    comp.sparse = True
    # train(False): the dense layer folds the UNMASKED delta and switches to F.linear; the compressed one only flips the
    # flags and keeps the masked forward - which equals the dense layer's forward before the fold
    w_masked = lin.weight.detach() * lin.mask
    with torch.no_grad():
        y_masked = lin(x)
        values0 = comp.values.clone()
        comp.train(False)
        assert not comp.training and not comp.lora_A.training and not comp.merged
        assert torch.equal(comp.values, values0) and torch.equal(comp(x), y_masked)
        lin.train(False)
        assert lin.merged and not torch.equal(lin(x), y_masked)
        comp.train(True)
        assert comp.training and torch.equal(comp(x), y_masked)
    back = comp.to_lora_linear()
    assert type(back) is Linear and torch.equal(back.mask, lin.mask) and back.sparse and back.r == 4
    assert torch.equal(back.weight, w_masked) and torch.equal(back.bias, lin.bias)
    assert torch.equal(back.lora_B.weight, comp.lora_B.weight) and back.lora_A.weight.dtype == torch.float32
    with pytest.raises(ValueError, match="merge"):
        comp.to_sparse24_linear()


@pytest.mark.gpu
def test_resident_bytes(native):
    from vlmc.sparse24 import Sparse24LoRALinear
    lin = dense_lora(4096, 11008, 8, "f16", False, 7)
    comp = Sparse24LoRALinear.from_lora_linear(lin)
    dense_bytes = lin.weight.numel() * lin.weight.element_size() + lin.mask.numel() * lin.mask.element_size()
    comp_bytes = comp.values.numel() * comp.values.element_size() + comp.meta.numel() * comp.meta.element_size()
    assert comp_bytes * 8 == dense_bytes * 3                                   # 0.375x, exactly


# ------------------------------------------------------------------------------------------- end to end
LLM = [f"llm_model.model.layers.{i}.{n}" for i in range(2) for n in
       ("self_attn.q_proj", "self_attn.k_proj", "self_attn.v_proj", "self_attn.o_proj", "mlp.gate_proj", "mlp.up_proj",
        "mlp.down_proj")]


def lora_toy(native):
    """The toy model with its 14 LLM linears as SparseLoRA layers (r = 8) and Wanda 2:4 masks on unzeroed weights.  The
    masks come from native.wanda_nm(..., zero_w=False) - the selection prune(lora_model=True) makes - on random
    activation norms: the toy pruners' capture path is built for plain nn.Linears."""
    import toy_model
    from vlmc.peft.lora import Linear
    model = toy_model.ToyBlip().cuda()
    g = torch.Generator(device="cuda").manual_seed(21)
    for name in LLM:
        old = model.get_submodule(name)
        lin = Linear(old.in_features, old.out_features, r=8, lora_alpha=16, bias=False).cuda().to(old.weight.dtype)
        lin.lora_A.float(); lin.lora_B.float()
        with torch.no_grad():
            lin.weight.copy_(old.weight)
            keep, _ = native.wanda_nm(lin.weight, torch.rand(old.in_features, device="cuda", generator=g) + 0.1, 2, 4,
                                      zero_w=False)
        lin.mask = keep
        lin.sparse = True
        parent, _, child = name.rpartition(".")
        setattr(model.get_submodule(parent), child, lin)
    for n, p in model.named_parameters():
        p.requires_grad_("lora_" in n)
    return model


def sgd_steps(model, batches, steps=3):
    params = [p for _, p in sorted(model.named_parameters()) if p.requires_grad]
    opt = torch.optim.SGD(params, lr=0.5)
    losses = []
    for i in range(steps):
        opt.zero_grad()
        y = model(batches[i % len(batches)])
        loss = (y.float() ** 2).mean()
        loss.backward()
        opt.step()
        losses.append(loss.detach())
    return torch.stack(losses)


@pytest.mark.gpu
def test_toy_model_finetune_merge_save(native, tmp_path):
    import toy_model
    from vlmc import checkpoint, sparse24
    model = lora_toy(native)
    dense = copy.deepcopy(model)
    replaced, skipped = sparse24.compress_model(model, lora=True)
    assert sorted(replaced) == sorted(LLM)
    assert any(s.startswith("visual_encoder.") for s in skipped) and "bridge" in skipped
    assert not any(".lora_" in s for s in skipped)
    assert all(isinstance(model.get_submodule(n), sparse24.Sparse24LoRALinear) for n in LLM)
    batches = toy_model.toy_batches(3, device="cuda", seed=5)
    losses_c, losses_d = sgd_steps(model, batches), sgd_steps(dense, batches)
    assert torch.equal(losses_c, losses_d), (losses_c, losses_d)
    for name in LLM:
        c, d = model.get_submodule(name), dense.get_submodule(name)
        assert bool(d.lora_B.weight.ne(0).any())
        assert torch.equal(c.lora_A.weight, d.lora_A.weight) and torch.equal(c.lora_B.weight, d.lora_B.weight), name
    for name in LLM:
        model.get_submodule(name).merge()
        dense.get_submodule(name).merge(remask=True)
        parent, _, child = name.rpartition(".")
        setattr(model.get_submodule(parent), child, model.get_submodule(name).to_sparse24_linear())
    path = str(tmp_path / "toy_lora_24.pth")
    checkpoint.save_compressed_checkpoint(model, path)
    fresh = toy_model.ToyBlip().cuda()
    assert sorted(checkpoint.load_compressed_checkpoint(fresh, path, dense=True)) == sorted(LLM)
    for name in LLM:
        w, want = fresh.get_submodule(name).weight, dense.get_submodule(name).weight
        assert type(fresh.get_submodule(name)) is torch.nn.Linear
        assert np.array_equal(bits_of(w), bits_of(want)), name                 # K14 remask writes +0, so does K25


@pytest.mark.gpu
def test_compress_model_default_skips_lora_layers(native):
    from vlmc import sparse24
    from vlmc.peft.lora import Linear
    model = lora_toy(native)
    replaced, skipped = sparse24.compress_model(model)
    assert not any(n in replaced for n in LLM) and all(n in skipped for n in LLM)
    assert all(type(model.get_submodule(n)) is Linear for n in LLM)
