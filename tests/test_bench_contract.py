"""bench.py's reference arm runs on CPU and prints its JSON line; `--dump-outputs` writes the same
arrays on every run."""
import importlib.util
import json
import subprocess
import sys
import zlib
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def _bench():
    spec = importlib.util.spec_from_file_location("bench", ROOT / "bench.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference"
    assert line["metric"].startswith("image-text pairs/sec")
    assert line["unit"] == "pairs/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["ms_per_step"] > 0
    cb = line["cpu_baseline"]
    # the unmodified reference when oracle/_ref is built (build container and GPU box), else the port
    want = "reference" if (ROOT / "oracle" / "_ref" / "x_clip" / "x_clip.py").exists() else "port"
    assert cb["kind"] == want and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0,
                           "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]


def test_gpu_arm_refuses_to_run_without_cuda():
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)


def test_step_outputs_sample_is_fixed_and_bounded():
    import torch
    bench = _bench()
    m = torch.nn.Module()
    m.big = torch.nn.Parameter(torch.randn(3000, 3000))
    m.small = torch.nn.Parameter(torch.randn(700))
    m.unused = torch.nn.Parameter(torch.randn(5))
    loss = (m.big.sin().sum() + m.small.square().sum()) / 1e3
    loss.backward()
    a, b = bench.step_outputs(loss, m), bench.step_outputs(loss, m)
    assert sorted(a) == ["grad.big", "grad.small", "loss"]
    assert all(v.dtype == np.float32 for v in a.values())
    assert a["loss"].shape == () and a["loss"] == np.float32(loss.item())
    assert np.array_equal(a["grad.small"], m.small.grad.numpy())
    assert 4096 <= a["grad.big"].size < m.big.numel()
    assert sum(v.size for v in a.values()) <= bench.DUMP_VALUES + 2 * 4096 + 1
    assert all(np.array_equal(a[k], b[k]) for k in a)
    # the documented positions: sorted, drawn without replacement, generator seeded by crc32 of the name
    gen = torch.Generator().manual_seed(zlib.crc32(b"big"))
    idx = torch.randperm(m.big.numel(), generator=gen)[:a["grad.big"].size].sort().values
    assert np.array_equal(a["grad.big"], m.big.grad.reshape(-1)[idx].numpy())


def test_bench_rejects_bad_arguments(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), *extra], capture_output=True, text=True,
                           timeout=300)
        assert r.returncode == 2 and "error:" in r.stderr, (extra, r.stderr[-500:])
    assert not any(tmp_path.iterdir())


@pytest.mark.gpu
def test_dump_outputs_identical_inputs_across_runs(cuda_device, tmp_path):
    """Two runs with the same arguments dump the same arrays (the README model samples its gradients); the
    dumped loss is the one the JSON line reports for the last timed step, and --steps sets how many steps
    the timed region launches."""
    def bench(steps, dump=None):
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "cfg2", "--batch", "64",
                            "--steps", str(steps), "--warmup", "1", "--no-e2e", "--no-profile", "--no-extras",
                            "--no-cpu-baseline", "--no-eager-baseline"] + (["--dump-outputs", str(dump)] if dump else []),
                           capture_output=True, text=True, timeout=280)
        assert r.returncode == 0, r.stderr[-2000:]
        return json.loads(r.stdout.strip().splitlines()[-1])

    lines, dumps = [], []
    for run in range(2):
        d = tmp_path / f"run{run}"
        lines.append(bench(2, d))
        dumps.append({f.stem: np.load(f) for f in sorted(d.glob("*.npy"))})
    one = bench(1)
    assert lines[0]["gpu_launches"] == lines[1]["gpu_launches"] == 2 * one["gpu_launches"] > 0
    a, b = dumps
    assert sorted(a) == sorted(b) and "loss" in a and len(a) > 50
    assert sum(f.stat().st_size for f in (tmp_path / "run0").iterdir()) <= 64 * 2**20
    for line, dump in zip(lines, dumps):
        assert abs(float(dump["loss"]) - line["config"]["loss"]) <= 1e-5 * max(1.0, abs(line["config"]["loss"]))
    for k in a:
        assert a[k].dtype == np.float32 and a[k].shape == b[k].shape, k
        np.testing.assert_allclose(a[k], b[k], rtol=1e-3, atol=1e-3 * float(np.abs(b[k]).max()) + 1e-12, err_msg=k)
