"""bench.py's output contract on the arm that runs without a GPU: `--impl reference` (the oracle port of the reference's CPU path) prints exactly
ONE line on stdout, a JSON object with the keys a caller reads; everything else (library banners, progress) goes to stderr.
On a GPU: what --dump-outputs writes for the native arm."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--batch", "2", "--points", "256", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "clouds/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "B=2" in d["config"]["workload"]


def test_native_arm_fails_loudly_without_a_gpu():
    import torch

    if torch.cuda.is_available():
        return
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode != 0 and "no CUDA device" in (p.stderr + p.stdout)
    assert p.stdout.strip() == ""                       # nothing that could be mistaken for a result line


def test_dump_outputs_keeps_a_fixed_sample_of_whole_clouds_under_the_cap(tmp_path, monkeypatch):
    import numpy as np
    import torch

    import bench

    monkeypatch.setattr(bench, "DUMP_BYTES", 10_000)
    y = torch.randn(40, 5, 30)                          # 24 000 bytes of float32
    bench.dump_outputs(str(tmp_path / "a"), "logits", y)
    bench.dump_outputs(str(tmp_path / "b"), "logits", y)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 10_000
    idx, got = np.load(tmp_path / "a" / "logits_clouds.npy"), np.load(tmp_path / "a" / "logits.npy")
    assert idx.dtype == np.float64 and got.dtype == np.float32 and len(idx) > 0 and np.all(np.diff(idx) > 0)
    np.testing.assert_array_equal(got, y.numpy()[idx.astype(np.int64)])
    np.testing.assert_array_equal(np.load(tmp_path / "b" / "logits_clouds.npy"), idx)


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["seg", "cls"])
def test_native_arm_dumps_the_logits_of_its_last_timed_step(tmp_path, workload):
    """--dump-outputs writes what the timed (graph-replayed) step computed: the logits of an eager forward of the same
    seeded model, calibrated on the same seeded batch, on the same seeded clouds.  --steps is the number of timed steps."""
    import numpy as np
    import torch

    import bench
    from samble_b200 import models
    from samble_b200.testing import synthetic_clouds

    B, N = 2, 512
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--batch", str(B), "--points", str(N),
                        "--steps", "3", "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 3
    _, model, _ = bench.build_model(workload, N)
    model = model.eval().cuda()
    xc, catc = synthetic_clouds(B, N, seed=1002)
    x, cat = synthetic_clouds(B, N, seed=2)
    with torch.no_grad():
        model(xc.cuda(), catc.cuda()) if workload == "seg" else model(xc.cuda())
        models.freeze_boundaries(model)
        y = model(x.cuda(), cat.cuda()) if workload == "seg" else model(x.cuda())
    got = np.load(tmp_path / "logits.npy")
    assert got.dtype == np.float32 and got.shape == tuple(y.shape)
    np.testing.assert_allclose(got, y.cpu().numpy(), rtol=1e-5, atol=1e-5)
