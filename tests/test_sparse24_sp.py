"""K31: the 2:4 linear on the sparse tensor cores (include/vlmc.h; native.sparse24_linear_sp; Sparse24Linear(sparse_mma)).

CPU: the fp64 reference that sums only the positions meta names (linear_named below), and the support check.
GPU: x = identity pins how the kernel reads values and meta (each output is one product 1.0 * w plus exact zeros); the
fp64 accuracy bar of K26 (at most 2x the error of F.linear on the dense weight); strided inputs; the non-finite rule; the
opt-in module path, its checkpoint and a CUDA graph of a compressed toy model.
"""
import numpy as np
import pytest
import torch

from oracle import sparse24 as oracle24

VICUNA = [(4096, 4096), (11008, 4096), (4096, 11008)]
DT = {"f16": torch.float16, "bf16": torch.bfloat16}


def linear_named(values, meta, x, bias=None):
    """fp64 y [T, R] = x [T, C] . W^T (+ bias) summing ONLY the positions meta names (the sparse tensor cores' product):
    an inf / NaN of x at an unnamed position never meets a weight.  values / bias: float arrays (the fp16 / bf16 values
    as numbers), meta: uint16 words [R, C/16], x: float [T, C]."""
    values = np.asarray(values, np.float64)
    meta = np.asarray(meta, np.uint16)
    x = np.asarray(x, np.float64)
    R, H = values.shape
    C = 2 * H
    nib = ((meta[..., None].astype(np.int64) >> (4 * np.arange(4))) & 15).reshape(R, C // 4)
    base = 4 * np.arange(C // 4)
    cols = np.stack([base + (nib & 3), base + (nib >> 2)], -1).reshape(R, H)      # column of every stored value
    y = np.einsum("rk,trk->tr", values, x[:, cols])
    if bias is not None:
        y = y + np.asarray(bias, np.float64)
    return y


def random_pruned(R, C, seed):
    """A float64 [R, C] weight with two non-zeros in every group of four, plus its numpy (values, meta) by the oracle."""
    rng = np.random.default_rng(seed)
    W = rng.standard_normal((R, C)) * 0.05 + 0.01
    keep = np.argsort(rng.random((R, C // 4, 4)), -1) < 2
    W = (W.reshape(R, C // 4, 4) * keep).reshape(R, C).astype(np.float16)
    values, meta = oracle24.sparse24_compress(W.view(np.uint16))
    return W.astype(np.float64), values.view(np.float16).astype(np.float64), meta


# ------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("R,C,T", [(3, 32, 5), (37, 176, 9), (64, 1024, 4)])
def test_linear_named_equals_dense_product_on_finite_inputs(R, C, T):
    W, values, meta = random_pruned(R, C, R + C)
    rng = np.random.default_rng(T)
    x = rng.standard_normal((T, C))
    bias = rng.standard_normal(R)
    np.testing.assert_allclose(linear_named(values, meta, x), x @ W.T, rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(linear_named(values, meta, x, bias), x @ W.T + bias, rtol=1e-12, atol=1e-12)


def test_linear_named_non_finite_rule():
    R, C = 4, 32
    W, values, meta = random_pruned(R, C, 1)
    W[0, :4] = 0                                     # row 0, group 0: no non-zero, padded with indices 0 and 1
    vbits, meta = oracle24.sparse24_compress(W.astype(np.float16).view(np.uint16))
    values = vbits.view(np.float16).astype(np.float64)
    named = oracle24.sparse24_decompress(np.ones_like(vbits), meta) != 0
    x = np.ones((3, C))
    x[0, 2] = np.inf                                 # unnamed in row 0 (padding named 0 and 1)
    x[1, 0] = np.nan                                 # named in row 0 (padding), stored value +0
    x[2, np.flatnonzero(~named[1])[0]] = np.inf      # unnamed in row 1
    y = linear_named(values, meta, x)
    assert np.isfinite(y[0, 0]) and np.isnan(y[1, 0]) and np.isfinite(y[2, 1])
    assert np.isnan(x[0] @ W[0]) and np.isnan(x[2] @ W[1])          # the dense product: 0 * inf
    keep = np.isfinite(x).all(1)
    np.testing.assert_allclose(y[keep], (x @ W.T)[keep])


def test_sp_supported_rejections():
    """C % 32 != 0, fp32, mismatched dtypes and CPU tensors are not K31's (checked on CUDA tensors when a GPU is there)."""
    from vlmc import native

    def ops(C=64, dt=torch.float16, xdt=None, dev="cpu"):
        return (torch.zeros(2, C, dtype=xdt or dt, device=dev), torch.zeros(8, C // 2, dtype=dt, device=dev),
                torch.zeros(8, C // 16, dtype=torch.int16, device=dev), C)

    assert not native.sparse24_linear_sp_supported(*ops())                                     # CPU tensors
    devs = ["cpu"] + (["cuda"] if torch.cuda.is_available() else [])
    for dev in devs:
        assert not native.sparse24_linear_sp_supported(*ops(C=48, dev=dev))                    # C % 32
        assert not native.sparse24_linear_sp_supported(*ops(dt=torch.float32, dev=dev))        # fp32
        assert not native.sparse24_linear_sp_supported(*ops(xdt=torch.bfloat16, dev=dev))      # dtypes differ
    if torch.cuda.is_available():
        assert native.sparse24_linear_sp_supported(*ops(dev="cuda"))


# ------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def native(built_lib):
    from vlmc import native as n
    n.load()
    assert torch.cuda.is_available()
    return n


def pruned_24(R, C, tag, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    W = (torch.randn(R, C, device="cuda", generator=g) * 0.02).to(DT[tag])
    keep = torch.rand(R, C // 4, 4, device="cuda", generator=g).argsort(-1) < 2
    return (W.view(R, C // 4, 4) * keep).view(R, C)


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["bf16", "f16"])
@pytest.mark.parametrize("R,C", [(328, 192), (4096, 4096)])
def test_operand_identity(native, tag, R, C):
    """x = identity: y[t, r] is the product 1.0 * w[r, t] plus exact zeros, so y is the weight the sparse MMA read: any
    misread code, word or row of meta, or value, shows here."""
    W = pruned_24(R, C, tag, 11)
    values, meta = native.sparse24_compress(W)
    Wd = native.sparse24_decompress(values, meta, C)
    x = torch.eye(C, device="cuda", dtype=DT[tag])
    for T in (1, 16, 256, C):
        T = min(T, C)
        y = native.sparse24_linear_sp(x[:T], values, meta, C)
        assert torch.equal(y, Wd[:, :T].t()), (T, int((y != Wd[:, :T].t()).sum()))


LINEAR_SHAPES = VICUNA + [(328, 192), (200, 1056)]


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["bf16", "f16"])
@pytest.mark.parametrize("R,C", LINEAR_SHAPES)
@pytest.mark.parametrize("T", [1, 7, 16, 128, 1000, 4096])
def test_linear_sp_vs_fp64(native, tag, R, C, T):
    """Against the fp64 product of the same rounded operands: max error at most 2x that of F.linear on the dense weight,
    with and without bias; two calls give the same bits."""
    W = pruned_24(R, C, tag, R * 7 + C + T)
    values, meta = native.sparse24_compress(W)
    g = torch.Generator(device="cuda").manual_seed(T)
    x = torch.randn(T, C, device="cuda", generator=g).to(DT[tag])
    bias = (torch.randn(R, device="cuda", generator=g) * 0.1).to(DT[tag])
    for b in (None, bias):
        y = native.sparse24_linear_sp(x, values, meta, C, b)
        ref = x.double() @ W.double().t() + (0 if b is None else b.double())
        err = float((y.double() - ref).abs().max())
        err_lib = float((torch.nn.functional.linear(x, W, b).double() - ref).abs().max())
        assert err <= 2 * err_lib, (err, err_lib)
        assert torch.equal(native.sparse24_linear_sp(x, values, meta, C, b).view(torch.int16), y.view(torch.int16))


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["bf16", "f16"])
def test_strided_inputs_and_rejections(native, tag):
    R, C, T = 200, 1056, 77
    W = pruned_24(R, C, tag, 5)
    values, meta = native.sparse24_compress(W)
    base = torch.randn(T, 2 * C, device="cuda").to(DT[tag])
    odd = torch.randn(T, C + 1, device="cuda").to(DT[tag])
    for x in (base[:, ::2], odd[:, :C], base[:, 3:3 + C], base[:, :C]):   # strided, odd pitch, unaligned, aligned view
        y = native.sparse24_linear_sp(x, values, meta, C)
        exact = x.double() @ W.double().t()
        bound = 2 * float((torch.nn.functional.linear(x, W).double() - exact).abs().max())
        assert float((y.double() - exact).abs().max()) <= bound
    x = base[:, :C].contiguous()
    assert torch.equal(native.sparse24_linear_sp(x.reshape(7, 11, C), values, meta, C).reshape(T, R),
                       native.sparse24_linear_sp(x, values, meta, C))
    Wo = pruned_24(R, 176, tag, 6)                                     # C % 32 != 0
    vo, mo = native.sparse24_compress(Wo)
    xo = torch.randn(3, 176, device="cuda").to(DT[tag])
    with pytest.raises(ValueError, match="32"):
        native.sparse24_linear_sp(xo, vo, mo, 176)
    y = torch.empty(3, R, device="cuda", dtype=DT[tag])
    assert native.load().vlmc_sparse24_linear_sp_forward(xo.data_ptr(), native._dtype(xo), 3, 176, xo.stride(0),
                                                         vo.data_ptr(), vo.stride(0), mo.data_ptr(), mo.stride(0), R,
                                                         None, y.data_ptr(), y.stride(0), None) < 0


@pytest.mark.gpu
@pytest.mark.parametrize("tag", ["bf16", "f16"])
def test_non_finite_rule(native, tag):
    """inf / NaN of x at positions meta does not name leave y finite and equal to the named-only fp64 sum; at named
    positions they propagate."""
    R, C, T = 136, 256, 40
    W = pruned_24(R, C, tag, 9)
    values, meta = native.sparse24_compress(W)
    named = native.sparse24_decompress(torch.ones_like(values), meta, C) != 0          # [R, C]
    x = torch.randn(T, C, device="cuda").to(DT[tag])
    col_unnamed_r0 = int(torch.nonzero(~named[0])[0])
    x[:8, col_unnamed_r0] = float("inf")
    x[8:16, col_unnamed_r0] = float("nan")
    y = native.sparse24_linear_sp(x, values, meta, C)
    yo = linear_named(values.double().cpu().numpy(), meta.cpu().numpy().view(np.uint16),
                               x.double().cpu().numpy())
    unnamed_rows = ~named[:, col_unnamed_r0]                  # rows whose product never meets the bad column
    assert bool(torch.isfinite(y[:16][:, unnamed_rows]).all())
    yo_t = torch.from_numpy(yo).cuda()
    fin = torch.isfinite(yo_t)
    assert torch.equal(fin, torch.isfinite(y))                # non-finite exactly where the named-only sum is
    err = float((y.double() - yo_t)[fin].abs().max())
    clean = torch.nn.functional.linear(x[16:], native.sparse24_decompress(values, meta, C)).double()
    bound = 2 * float((clean - torch.from_numpy(yo[16:]).cuda()).abs().max())
    assert err <= bound, (err, bound)
    assert bool(torch.isnan(torch.nn.functional.linear(x[:16], native.sparse24_decompress(values, meta, C))).any())


@pytest.mark.gpu
def test_module_routing_and_state(native, monkeypatch):
    from vlmc import sparse24
    lin = torch.nn.Linear(1024, 520, device="cuda").bfloat16()
    with torch.no_grad():
        lin.weight.copy_(pruned_24(520, 1024, "bf16", 3))
    base = sparse24.Sparse24Linear.from_linear(lin)
    sp = sparse24.Sparse24Linear.from_linear(lin, sparse_mma=True)
    assert list(base.state_dict()) == list(sp.state_dict())
    assert "sparse_mma=True" in repr(sp) and "sparse_mma=False" in repr(base)
    Wd = native.sparse24_decompress(sp.values, sp.meta, 1024)
    with torch.no_grad():
        monkeypatch.setattr(sparse24, "SPARSE_MMA_MIN_TOKENS", 100)
        monkeypatch.setattr(sparse24, "SPARSE_MMA_MAX_TOKENS", 400)
        for T in (5, 300, 500):                        # below, inside and above the K31 window
            x = torch.randn(T, 1024, device="cuda").bfloat16()
            expand = torch.nn.functional.linear(x, Wd, sp.bias)
            assert torch.equal(base(x), expand)                                   # the default: today's path
            if 100 <= T < 400:
                assert torch.equal(sp(x), native.sparse24_linear_sp(x, sp.values, sp.meta, 1024, sp.bias))
            else:
                assert torch.equal(sp(x), expand)


@pytest.mark.gpu
def test_toy_model_sparse_mma(native, tmp_path, monkeypatch):
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
    monkeypatch.setattr(sparse24, "SPARSE_MMA_MIN_TOKENS", 1)
    replaced, _ = sparse24.compress_model(model, sparse_mma=True)
    assert len(replaced) == 14
    calls = []
    real_sp = native.sparse24_linear_sp
    monkeypatch.setattr(native, "sparse24_linear_sp", lambda x, v, m, C, b=None: calls.append(C) or real_sp(x, v, m, C, b))
    with torch.no_grad():
        y = model(batch)
    layers = model.llm_model.model.layers
    sp_layers = [getattr(getattr(blk, a), n) for blk in layers for a, n in
                 (("self_attn", "q_proj"), ("self_attn", "k_proj"), ("self_attn", "v_proj"), ("self_attn", "o_proj"),
                  ("mlp", "gate_proj"), ("mlp", "up_proj"))]
    assert all(m.in_features == 64 and m.sparse_mma for m in sp_layers)
    assert all(blk.mlp.down_proj.in_features == 176 for blk in layers)
    assert sorted(calls) == [64] * 12                         # q/k/v/o/gate/up take K31; down_proj (C = 176) does not
    err, err_dense = float((y.double() - ref).abs().max()), float((y_dense.double() - ref).abs().max())
    assert err <= 2 * err_dense, (err, err_dense)
    monkeypatch.setattr(native, "sparse24_linear_sp", real_sp)
    path = str(tmp_path / "toy_24_sp.pth")
    checkpoint.save_compressed_checkpoint(model, path)
    fresh = toy_model.ToyBlip().eval().cuda()
    checkpoint.load_compressed_checkpoint(fresh, path, sparse_mma=True)
    assert fresh.llm_model.model.layers[0].self_attn.q_proj.sparse_mma
    with torch.no_grad():
        assert torch.equal(fresh(batch), y)
    # a CUDA graph of the forward replays to the eager result
    static = {k: v.clone() if torch.is_tensor(v) else v for k, v in batch.items()}
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.no_grad(), torch.cuda.stream(s):
        for _ in range(2):
            model(static)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.no_grad(), torch.cuda.graph(g):
        out = model(static)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, y)
