"""Compressed 2:4 weights (include/vlmc.h, K24-K26; vlmc.sparse24; vlmc.checkpoint compressed files).

CPU: the numpy oracle's format rules.  GPU: compress / decompress bit-exact against the oracle, the K26 linear against an
fp64 product of the same operands (bar: at most 2x the error of F.linear on the dense weight), determinism, the
large-T path, and a pruned toy model compressed, saved and loaded.
Pruned zeros: the format keeps no sign for them (decompression writes +0), while a pruner that multiplies by the mask
leaves -0 where the weight was negative, so bit comparisons canonicalise pruned zeros to +0 first.
"""
import numpy as np
import pytest
import torch

from oracle import sparse24 as oracle24

VICUNA = [(4096, 4096), (11008, 4096), (4096, 11008)]
DT = {"f16": torch.float16, "bf16": torch.bfloat16}


def random_24_bits(R, C, seed, tag="bf16", specials=True):
    """uint16 bit patterns of a 2:4 weight: groups with 0, 1 or 2 kept values at random positions, pruned slots +0 or -0,
    NaN among the kept values and an all-zero row."""
    rng = np.random.default_rng(seed)
    w = torch.from_numpy(rng.standard_normal((R, C)).astype(np.float32) * 0.05).to(DT[tag])
    bits = w.view(torch.int16).numpy().view(np.uint16).copy().reshape(R, C // 4, 4)
    bits[(bits & 0x7FFF) == 0] |= 1                                     # every element non-zero before pruning
    nkeep = rng.choice([0, 1, 2, 2, 2], size=(R, C // 4))
    order = np.argsort(rng.random((R, C // 4, 4)), axis=-1)
    keep = np.zeros((R, C // 4, 4), bool)
    for k in range(2):
        np.put_along_axis(keep, order[..., k:k + 1], (nkeep > k)[..., None], -1)
    zeros = np.where(rng.random((R, C // 4, 4)) < 0.5, 0x8000, 0).astype(np.uint16)
    bits = np.where(keep, bits, zeros)
    if specials:
        nan = 0x7FC0 if tag == "bf16" else 0x7E00
        bits[0, 0] = [nan, 0, 0x8000, 0]
        bits[min(1, R - 1)] = 0x8000
    return bits.reshape(R, C).astype(np.uint16)


def canonical(bits):
    bits = np.asarray(bits, np.uint16).copy()
    bits[bits == 0x8000] = 0
    return bits


# ------------------------------------------------------------------------------------------- CPU: the oracle's rules
@pytest.mark.parametrize("R,C", [(3, 16), (37, 176), (64, 1024)])
def test_oracle_round_trip(R, C):
    W = random_24_bits(R, C, R + C)
    values, meta = oracle24.sparse24_compress(W)
    assert values.shape == (R, C // 2) and meta.shape == (R, C // 16)
    assert np.array_equal(oracle24.sparse24_decompress(values, meta), canonical(W))
    nib = ((meta[..., None].astype(np.int64) >> (4 * np.arange(4))) & 15).reshape(R, C // 4)
    assert ((nib & 3) < (nib >> 2)).all()                      # two distinct indices, ascending
    assert not (values == 0x8000).any()                        # padded slots store +0


def test_oracle_padding_rules():
    W = np.zeros((1, 16), np.uint16)
    W[0, :4] = [0, 0x3C00, 0, 0x4000]          # two kept: indices 1, 3
    W[0, 4:8] = [0, 0, 0x8000, 0x3C00]         # one kept at 3: padded with index 0
    W[0, 8:12] = [0x8000, 0, 0, 0]             # none kept (-0 is pruned): indices 0, 1
    W[0, 12:16] = [0x7E00, 0, 0, 0]            # NaN is kept
    values, meta = oracle24.sparse24_compress(W)
    assert values.tolist() == [[0x3C00, 0x4000, 0, 0x3C00, 0, 0, 0x7E00, 0]]
    assert int(meta[0, 0]) == (1 | 3 << 2) | (0 | 3 << 2) << 4 | (0 | 1 << 2) << 8 | (0 | 1 << 2) << 12


def test_oracle_rejects_three_of_four():
    W = random_24_bits(8, 32, 1, specials=False)
    W[5, 8:12] = [0x3C00, 0x3C00, 0, 0x3C00]
    with pytest.raises(ValueError):
        oracle24.sparse24_compress(W)


@pytest.mark.parametrize("R,C", VICUNA + [(64, 176)])
def test_format_byte_counts(R, C):
    values, meta = oracle24.sparse24_compress(np.zeros((R, C), np.uint16))
    assert values.nbytes == R * C and meta.nbytes == R * C // 8
    assert (values.nbytes + meta.nbytes) / (R * C * 2) == 0.5625


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


def check_against_oracle(native, W, tag):
    values, meta = native.sparse24_compress(W)
    vo, mo = oracle24.sparse24_compress(bits_of(W))
    assert np.array_equal(bits_of(values), vo) and np.array_equal(bits_of(meta), mo)
    Wd = native.sparse24_decompress(values, meta, W.shape[1])
    assert np.array_equal(bits_of(Wd), canonical(bits_of(W)))
    return values, meta


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["bf16", "f16"])
@pytest.mark.parametrize("R,C", VICUNA)
def test_compress_wanda_nm_weights(native, tag, R, C):
    g = torch.Generator(device="cuda").manual_seed(R + C)
    W = (torch.randn(R, C, device="cuda", generator=g) * 0.02).to(DT[tag])
    scaler = torch.rand(C, device="cuda", generator=g) * 10
    native.wanda_nm(W, scaler, 2, 4)
    check_against_oracle(native, W, tag)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["bf16", "f16"])
@pytest.mark.parametrize("R,C", VICUNA)
def test_compress_sparsegpt_24_weights(native, tag, R, C):
    from vlmc.compression.pruners.sparsegpt_pruner import SparseGPT
    torch.manual_seed(R + 3 * C)
    lin = torch.nn.Linear(C, R, bias=False, device="cuda").to(DT[tag])
    sg = SparseGPT(lin)
    sg.add_batch((torch.randn(1, 2048, C, device="cuda")).to(DT[tag]), None)
    sg.fasterprune(0.5, prune_n=2, prune_m=4)
    W = lin.weight.data
    assert float((W == 0).float().mean()) >= 0.5
    check_against_oracle(native, W, tag)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["bf16", "f16"])
def test_compress_specials_and_strided_views(native, tag):
    R, C = 37, 176
    bits = random_24_bits(R, C, 5, tag)
    W = from_bits(bits, tag)
    values, meta = check_against_oracle(native, W, tag)
    for off, pad in ((3, 5), (8, 24)):                  # misaligned (element path) and 16-byte aligned (vector path)
        buf = torch.zeros(R, C + pad, dtype=DT[tag], device="cuda")
        view = buf[:, off:off + C]
        view.copy_(W)
        v2, m2 = native.sparse24_compress(view)
        assert torch.equal(v2.view(torch.int16), values.view(torch.int16)) and torch.equal(m2, meta)
        vbuf = torch.zeros(R, C // 2 + pad, dtype=DT[tag], device="cuda")
        vview = vbuf[:, off:off + C // 2]
        vview.copy_(values)
        out = torch.full((R, C + pad), 7.0, dtype=DT[tag], device="cuda")
        native.sparse24_decompress(vview, meta, C, out=out[:, off:off + C])
        assert np.array_equal(bits_of(out[:, off:off + C]), canonical(bits))
        assert bool((out[:, :off] == 7).all()) and bool((out[:, off + C:] == 7).all())


@pytest.mark.gpu
def test_compress_rejects_three_of_four_and_leaves_w(native):
    W = from_bits(random_24_bits(64, 256, 9, specials=False), "bf16")
    W[40, 100] = 1.0                  # the group 100..103 now has three non-zeros at least once in 64 rows
    W[40, 101] = 1.0
    W[40, 102] = 1.0
    W0 = W.clone()
    with pytest.raises(ValueError, match="2:4"):
        native.sparse24_compress(W)
    assert torch.equal(W.view(torch.int16), W0.view(torch.int16))
    with pytest.raises(ValueError):
        native.sparse24_compress(W[:, :40].contiguous())         # C % 16 != 0
    assert native.load().vlmc_status_string(native.NOT_2OF4).decode().startswith("weight is not 2:4")


def pruned_24(R, C, tag, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    W = (torch.randn(R, C, device="cuda", generator=g) * 0.02).to(DT[tag])
    keep = torch.rand(R, C // 4, 4, device="cuda", generator=g).argsort(-1) < 2
    return (W.view(R, C // 4, 4) * keep).view(R, C)


LINEAR_SHAPES = VICUNA + [(328, 176), (200, 1040)]


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["bf16", "f16"])
@pytest.mark.parametrize("R,C", LINEAR_SHAPES)
@pytest.mark.parametrize("T", [1, 7, 16, 64, 128, 1000, 4096])
def test_linear_vs_fp64(native, tag, R, C, T):
    """K26 against the fp64 product of the same rounded operands: max error at most 2x that of F.linear on the dense
    weight, with and without bias; two calls give the same bits."""
    W = pruned_24(R, C, tag, R * 7 + C + T)
    values, meta = native.sparse24_compress(W)
    g = torch.Generator(device="cuda").manual_seed(T)
    x = torch.randn(T, C, device="cuda", generator=g).to(DT[tag])
    bias = (torch.randn(R, device="cuda", generator=g) * 0.1).to(DT[tag])
    for b in (None, bias):
        y = native.sparse24_linear(x, values, meta, C, b)
        ref = x.double() @ W.double().t() + (0 if b is None else b.double())
        err = float((y.double() - ref).abs().max())
        err_lib = float((torch.nn.functional.linear(x, W, b).double() - ref).abs().max())
        assert err <= 2 * err_lib, (err, err_lib)
        assert torch.equal(native.sparse24_linear(x, values, meta, C, b).view(torch.int16), y.view(torch.int16))


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["bf16", "f16"])
@pytest.mark.parametrize("R,C", [(328, 176), (4096, 4096)])
def test_linear_operand_is_the_decompressed_weight(native, tag, R, C):
    """x = identity: every output is one product 1.0 * W[r, c] plus zeros (in the split-K partials too), so y is the
    on-chip operand itself: equal to decompress(values, meta) transposed."""
    W = pruned_24(R, C, tag, 11)
    values, meta = native.sparse24_compress(W)
    x = torch.eye(C, device="cuda", dtype=DT[tag])
    for T in (1, 16, C):
        y = native.sparse24_linear(x[:T], values, meta, C)
        assert torch.equal(y, native.sparse24_decompress(values, meta, C)[:, :T].t())


@pytest.mark.gpu
def test_module_paths_and_rejections(native, monkeypatch):
    from vlmc import sparse24
    lin = torch.nn.Linear(1024, 520, device="cuda").bfloat16()
    with torch.no_grad():
        lin.weight.copy_(pruned_24(520, 1024, "bf16", 3))
    mod = sparse24.Sparse24Linear.from_linear(lin)
    assert torch.equal(mod.to_dense().weight, lin.weight) and torch.equal(mod.to_dense().bias, lin.bias)
    x = torch.randn(3, 300, 1024, device="cuda").bfloat16()
    with torch.no_grad():
        for limit in (10 ** 9, 1):               # fused K26 at every size / expand + library GEMM at every size
            monkeypatch.setattr(sparse24, "DENSE_EXPAND_MIN_TOKENS", limit)
            y = mod(x)
            assert y.shape == (3, 300, 520)
            if limit == 1:
                W = native.sparse24_decompress(mod.values, mod.meta, 1024)
                assert torch.equal(y, torch.nn.functional.linear(x, W, mod.bias))
            else:
                assert torch.equal(y, native.sparse24_linear(x, mod.values, mod.meta, 1024, mod.bias))
    with pytest.raises(RuntimeError, match="inference-only"):
        mod(x.requires_grad_())
    with pytest.raises(ValueError):
        mod(x.detach().half())
    dense = torch.nn.Linear(64, 32, device="cuda").bfloat16()
    with pytest.raises(ValueError):
        sparse24.Sparse24Linear.from_linear(dense)


@pytest.mark.gpu
def test_toy_model_compress_save_load(native, tmp_path, monkeypatch):
    import toy_model
    import vlmc.compression as comp
    from vlmc import checkpoint, sparse24
    model = toy_model.ToyBlip().eval().cuda()
    batches = toy_model.toy_batches(8, device="cuda")
    pruner = comp.load_pruner("blipt5_wanda_pruner", model, batches, cfg=toy_model.pruner_cfg(0.5, 0.5, prune_n=2, prune_m=4))
    model, _ = pruner.prune()
    pruned_state = {k: v.clone() for k, v in model.state_dict().items()}
    batch = toy_model.toy_batches(1, device="cuda", seed=7)[0]
    with torch.no_grad():
        y_dense = model(batch)
        y64 = toy_model.ToyBlip(llm_dtype=torch.float64).double().cuda()
        y64.load_state_dict({k: v.double() if v.is_floating_point() else v for k, v in pruned_state.items()})
        ref = y64({**batch, "image": batch["image"].double()}).double()
    replaced, skipped = sparse24.compress_model(model)
    assert sorted(replaced) == sorted(f"llm_model.model.layers.{i}.{n}" for i in range(2) for n in
                                      ("self_attn.q_proj", "self_attn.k_proj", "self_attn.v_proj", "self_attn.o_proj",
                                       "mlp.gate_proj", "mlp.up_proj", "mlp.down_proj"))
    assert any(s.startswith("visual_encoder.") for s in skipped) and "bridge" in skipped
    with torch.no_grad():
        assert torch.equal(model(batch), y_dense)                 # expand + library GEMM: the dense model's bits
        monkeypatch.setattr(sparse24, "DENSE_EXPAND_MIN_TOKENS", 10 ** 9)     # K26 on every linear from here on
        y = model(batch)
        err, err_dense = float((y.double() - ref).abs().max()), float((y_dense.double() - ref).abs().max())
        assert err <= 2 * err_dense, (err, err_dense)
    path = str(tmp_path / "toy_24.pth")
    checkpoint.save_compressed_checkpoint(model, path)
    fresh = toy_model.ToyBlip().eval().cuda()
    assert len(checkpoint.load_compressed_checkpoint(fresh, path)) == 14
    assert isinstance(fresh.llm_model.model.layers[1].mlp.down_proj, sparse24.Sparse24Linear)
    with torch.no_grad():
        assert torch.equal(fresh(batch), y)
    dense = toy_model.ToyBlip().eval().cuda()
    checkpoint.load_compressed_checkpoint(dense, path, dense=True)
    assert type(dense.llm_model.model.layers[0].self_attn.q_proj) is torch.nn.Linear
    state = dense.state_dict()
    assert sorted(state) == sorted(pruned_state)
    for k, v in state.items():
        assert torch.equal(v, pruned_state[k]), k                  # -0 and +0 compare equal
