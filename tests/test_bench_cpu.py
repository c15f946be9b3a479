"""The CPU arm of bench.py (`--impl reference`) runs without a GPU and prints the
contract's JSON line."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cora",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["value"] > 0 and line["steps"] == 2
    # the reference's own code when oracle/_ref is staged (or /root/reference is mounted), else the port
    sys.path.insert(0, ROOT)
    from oracle import ref_shim
    want_kind = "reference" if ref_shim.reference_root() is not None else "port"
    assert line["cpu_baseline"]["kind"] == want_kind and line["cpu_baseline"]["cores"] == 1
    split = line["cpu_baseline"]["split_seconds"]
    assert split["total"] > 0 and ("laplacian" in split or "laplacian_and_rescale" in split) and "recurrence" in split
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    # same configuration object as the GPU arm prints: the full named shape, not a sample
    from efficient_gnn_b200 import synth
    cfg = line["config"]
    assert cfg["workload"] == "cora-shape" and cfg["n"] == synth.SHAPES["cora"].n and cfg["k"] == 3 and cfg["f"] == 1
    assert cfg["nnz"] == synth.SHAPES["cora"].nnz + cfg["n"] and line["scaling"] == "strong"


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cora",
                          "--gpus", "2", "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300,
                         cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


import numpy as np  # noqa: E402
import pytest  # noqa: E402
import torch  # noqa: E402


def test_bad_steps_and_dump_outputs_of_the_reference_arm_are_refused(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cora", *extra],
                             capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "", extra
    assert os.listdir(tmp_path) == []


def test_dump_features_bounds_the_size_with_a_fixed_row_sample(tmp_path):
    import bench
    feats = torch.randn(300_000, 60, generator=torch.Generator().manual_seed(0))      # 72 MB of float32
    for d in ("a", "b"):
        bench.dump_features(str(tmp_path / d), feats)
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= bench.DUMP_MAX_BYTES
    rows, got = np.load(tmp_path / "a" / "features_rows.npy"), np.load(tmp_path / "a" / "features.npy")
    assert rows.dtype == np.float64 and got.dtype == np.float32 and np.all(np.diff(rows) > 0)
    np.testing.assert_array_equal(got, feats.numpy()[rows.astype(np.int64)])
    for name in ("features_rows.npy", "features.npy"):                 # the same sample on every run
        np.testing.assert_array_equal(np.load(tmp_path / "b" / name), np.load(tmp_path / "a" / name))
    small = torch.randn(10, 3, dtype=torch.float64)
    bench.dump_features(str(tmp_path / "c"), small)
    assert os.listdir(tmp_path / "c") == ["features.npy"]
    np.testing.assert_array_equal(np.load(tmp_path / "c" / "features.npy"), small.float().numpy())


@pytest.mark.gpu
@pytest.mark.parametrize("f", [1, 8])
def test_gpu_arm_dumps_the_features_of_its_last_step(tmp_path, f):
    """--dump-outputs: what the last timed step returned equals the same call made here on the bench's seeded
    graph and signal, and --steps is the number of timed steps."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "pubmed", "--f", str(f),
                          "--steps", "3", "--warmup", "1", "--no-cpu-baseline", "--no-e2e", "--no-ugca",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 3
    assert os.listdir(tmp_path) == ["features.npy"]
    got = np.load(tmp_path / "features.npy")

    import efficient_gnn_b200 as egnn
    from efficient_gnn_b200 import synth
    rp, ci, n = synth.synth_csr("pubmed", self_loops=True, device="cuda")
    x0 = None
    if f > 1:
        x0 = torch.randn(n, f, device="cuda", generator=torch.Generator(device="cuda").manual_seed(synth.SHAPES["pubmed"].seed))
    graph = egnn.CsrGraph(rp, ci, None, n)
    want = egnn.graph_wavelet_features(graph, k=3, s=0.8, X0=x0).cpu().numpy()
    s = egnn.graph_wavelet_features(graph, k=3, s=0.8, X0=x0, return_parts=True).combined.reshape(n, -1).cpu().numpy()
    sure = np.abs(s) > 1e-4 * np.abs(s).max()         # away from sign flips of S ~ 0 (F = 1: H = sign(S))
    assert got.dtype == np.float32 and got.shape == (n, f)
    np.testing.assert_allclose(got[sure], want[sure], rtol=0, atol=1e-6)


@pytest.mark.gpu
def test_gpu_arm_prints_the_contract_line():
    """The GPU arm on a small shape: one JSON line with the contract's keys, the roofline and the
    end-to-end objects, and a config object identical to the reference arm's."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "pubmed", "--steps", "6",
                          "--warmup", "3"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"):
        assert key in line, key
    assert line["n_gpus"] == 1 and line["steps"] == 6 and line["warmup"] >= 3 and line["value"] > 0
    assert line["scaling"] == "strong" and line["vs_baseline"] is None and line["dtype"] == "f32"
    r = line["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and r["peak"] > 0 and 0 < r["frac"] < 1.2
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    e = line["e2e"]
    assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and 0 < e["value"] < line["value"]
    assert line["gpu_launches"] > 0
    ref = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "pubmed",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert ref.returncode == 0, ref.stderr[-2000:]
    assert json.loads(ref.stdout.strip().splitlines()[-1])["config"] == line["config"]
