"""bench.py contract checks that need no GPU: the reference arm runs on the CPU and prints ONE JSON
line with the keys the driver reads; the B200 arm refuses to run without a CUDA device."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, BENCH, "--impl", "reference", "--workload", "c2", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "utterances/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["vs_baseline"] is None and d["dtype"] == "f32" and d["data"] == "synthetic"
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, BENCH, "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_argument_rejections():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        out = subprocess.run([sys.executable, BENCH] + extra, capture_output=True, text=True, timeout=120)
        assert out.returncode == 2 and "error:" in out.stderr, (extra, out.stderr[-500:])


def test_dump_outputs_files(tmp_path):
    """dump_outputs on small CPU tensors: float32 files, the sampled entries are the gradient's."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    N, T, U, V = 3, 5, 4, 7
    grads = torch.randn(N, T, U, V)
    labels = np.random.default_rng(0).integers(1, V, size=(N, U - 1)).astype(np.int32)
    costs = torch.randn(N)
    bench.dump_outputs(torch, str(tmp_path), costs, grads, labels, costs.sum().reshape(1))
    out = {p.stem: np.load(p) for p in tmp_path.iterdir()}
    assert sorted(out) == ["costs", "grads_blank", "grads_label", "grads_sample", "loss"]
    assert all(a.dtype == np.float32 for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= bench.DUMP_LIMIT_BYTES
    assert np.array_equal(out["costs"], costs.numpy()) and np.isclose(out["loss"][0], costs.sum().item())
    g = grads.numpy()
    assert np.isin(out["grads_blank"], g[..., 0]).all()
    at_labels = np.take_along_axis(g[:, :, :U - 1], labels[:, None, :, None].astype(np.int64), 3)
    assert np.isin(out["grads_label"], at_labels).all()
    assert np.isin(out["grads_sample"], g).all()
    again = tmp_path / "again"
    bench.dump_outputs(torch, str(again), costs, grads, labels, costs.sum().reshape(1))
    assert all(np.array_equal(np.load(again / (k + ".npy")), v) for k, v in out.items())


def test_b200_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, BENCH, "--steps", "1", "--warmup", "1"], capture_output=True,
                         text=True, timeout=300)
    assert out.returncode != 0 and "no CUDA device" in (out.stderr + out.stdout)
