"""CPU: the reference arm of bench.py (`--impl reference`) runs without a GPU and prints the contract's JSON line; ranks
other than 0 exit 0 without work (the driver launches it under torchrun for N > 1)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra, *args):
    env = dict(os.environ, **env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, env=env, capture_output=True,
                          text=True, timeout=600)


import pytest


@pytest.mark.parametrize("kind", ["reference", "port"])
def test_reference_arm_prints_the_contract_line(kind):
    """kind "reference": the unmodified reference files (here /root/reference, on the GPU box baseline/_ref) run the whole
    block; kind "port": they are absent (VLMC_REFERENCE_ROOT points nowhere) and oracle/cpu_port.py times a bounded sample."""
    sys.path.insert(0, ROOT)
    from oracle import ref_loader
    if kind == "reference" and not ref_loader.available():
        pytest.skip("no reference tree")
    r = _run({} if kind == "reference" else {"VLMC_REFERENCE_ROOT": "/nonexistent"}, "--impl", "reference", "--steps", "1",
             "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["higher_is_better"] is False and line["vs_baseline"] is None
    assert line["metric"] == "s_per_vicuna7b_block_pruned" and line["unit"] == "s/block" and line["value"] > 0
    assert abs(line["ms_per_step"] - 1e3 * line["value"]) < 1e-6 * line["ms_per_step"]
    assert line["steps"] == 1 and line["warmup"] == 0 and line["n_gpus"] == 1 and line["data"] == "synthetic"
    assert "workload" in line["config"] and "model" not in line["config"]
    cb = line["cpu_baseline"]
    assert cb["kind"] == kind and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0


def test_reference_arm_other_ranks_exit_quietly():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--impl", "reference", "--gpus", "2", "--steps", "1",
             "--warmup", "0")
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_sample(monkeypatch):
    """--dump-outputs: float32 copies of the same seeded rows of every linear on every call, masks only when the method
    returns them, at most 64 MB for the benched block; a run without timed steps or on several GPUs is refused up front."""
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch
    import bench
    assert sum(2 * bench.DUMP_ROWS * C * 4 for _, _, C, _ in bench.LINEARS) <= 64 << 20
    monkeypatch.setattr(bench, "LINEARS", [("a", 300, 40, "x"), ("b", 129, 24, "y")])
    g = torch.Generator().manual_seed(0)
    W = {n: torch.randn(R, C, generator=g).half() for n, R, C, _ in bench.LINEARS}
    M = {n: torch.rand(R, C, generator=g) < 0.5 for n, R, C, _ in bench.LINEARS}
    got = bench.sample_outputs(torch, W, M)
    assert sorted(got) == ["a.mask", "a.weight", "b.mask", "b.weight"]
    for n, R, C, _ in bench.LINEARS:
        w, m = got[f"{n}.weight"], got[f"{n}.mask"]
        assert w.dtype == m.dtype == np.float32 and w.shape == m.shape == (bench.DUMP_ROWS, C)
        rows = [r for r in range(R) if any(np.array_equal(W[n][r].float().numpy(), x) for x in w)]
        assert len(rows) == bench.DUMP_ROWS and np.array_equal(m, M[n][rows].float().numpy())
    again = bench.sample_outputs(torch, W, None)
    assert sorted(again) == ["a.weight", "b.weight"] and all(np.array_equal(again[k], got[k]) for k in again)
    for bad in (["--steps", "0"], ["--gpus", "2", "--dump-outputs", "out"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = _run({}, *bad)
        assert r.returncode == 2 and "error" in r.stderr, bad


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_step(tmp_path):
    """bench.py --dump-outputs end to end, Wanda 2:4: the graph replay and the eager pass each dump their last timed step;
    both prune the same weight set, so the files are identical, and every dumped row is a 2:4 mask with the weight zero
    wherever the mask drops it."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    dumps = {}
    for graph in (True, False):
        d = tmp_path / ("graph" if graph else "eager")
        r = _run({}, "--steps", "2", "--warmup", "3", "--no-other-methods", "--no-cpu-baseline", "--no-full-model",
                 "--dump-outputs", str(d), *([] if graph else ["--no-graph"]))
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 2 and line["config"]["dump_outputs"]["pass"] == ("graph" if graph else "eager")
        assert sorted(p.name for p in d.iterdir()) == sorted(f"{n}.{k}.npy" for n, *_ in bench.LINEARS for k in ("weight", "mask"))
        dumps[graph] = {p.name: np.load(p) for p in d.iterdir()}
    for name, _, C, _ in bench.LINEARS:
        w, m = dumps[True][f"{name}.weight.npy"], dumps[True][f"{name}.mask.npy"]
        assert w.dtype == m.dtype == np.float32 and w.shape == m.shape == (bench.DUMP_ROWS, C)
        assert set(np.unique(m)) == {0.0, 1.0} and (m.reshape(bench.DUMP_ROWS, -1, 4).sum(axis=2) == 2).all(), name
        assert (w[m == 0] == 0).all() and (w[m == 1] != 0).mean() > 0.99, name
    for f in dumps[True]:
        assert np.array_equal(dumps[True][f], dumps[False][f]), f


def test_statistics_roofline_is_quoted_on_distinct_bytes_when_batched(monkeypatch):
    """SURVEY 8(d) asks to say which byte count the roofline uses: with the block's statistics as ONE launch the linears fed
    the same activations share them through L2, so `achieved` / `frac` count the four distinct tensors (12.21 of the 18.66 GB)
    and the per-linear figure sits beside them; with one launch per linear, or shared inputs, nothing is rescaled."""
    sys.path.insert(0, ROOT)
    import bench
    pk = {"hbm": 6545.0, "tensor": 1688.0, "tensor_sustained": 1408.0, "source": "test"}

    def res(world=1, calib_batch=bench.N_SEQ, shared=False):
        return {"method": "wanda_nm", "steps": 10, "eager_ms_per_step": 2.05, "shared": shared, "world": world, "calib_batch": calib_batch,
                "kernels": {"sqnorm_accum": {"ms": 18.3, "work": 18.66e9 * 10, "spans": 10},
                            "wanda_select": {"ms": 1.86, "work": 1.012e9 * 10, "spans": 10}}}
    monkeypatch.delenv("VLMC_BENCH_STATS_BATCH", raising=False)
    r = bench.roofline_of(res(), pk)
    distinct = (3 * 4096 + 11008) / (6 * 4096 + 11008)
    assert abs(r["frac_per_linear_bytes"] - 18.66e9 / 1.83e-3 / 1e9 / 6545.0) < 1e-9
    assert abs(r["frac"] - r["frac_per_linear_bytes"] * distinct) < 1e-12 and r["frac"] < 1.1 and "bytes_basis" in r
    assert bench.roofline_of(res(world=2), pk)["frac"] == r["frac"]                       # batched at every N > 1
    for plain in (res(calib_batch=16), res(shared=True)):
        q = bench.roofline_of(plain, pk)
        assert "frac_per_linear_bytes" not in q and abs(q["frac"] - r["frac_per_linear_bytes"]) < 1e-9
    monkeypatch.setenv("VLMC_BENCH_STATS_BATCH", "0")
    assert "frac_per_linear_bytes" not in bench.roofline_of(res(), pk)
