"""bench.py --dump-outputs on the GPU: the timed forward's outputs land as .npy files, they are what an eager forward of the
bench's seeded model and batch returns, and two runs with the same workload (different step counts) compute the same thing."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["--layers", "50", "--image", "128", "--volume", "32", "--views", "2", "--batch", "2", "--warmup", "1",
         "--no-cpu-baseline", "--no-config5", "--no-torch-gpu"]


def _bench(steps, out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--dump-outputs", str(out_dir)] + SMALL,
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0]), {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_dump_outputs_same_workload_same_outputs(tmp_path):
    line_a, a = _bench(2, tmp_path / "a")
    line_b, b = _bench(3, tmp_path / "b")
    assert line_a["steps"] == 2 and line_b["steps"] == 3
    assert sorted(a) == ["base_points", "coord_volumes", "features", "keypoints_3d", "volumes"]
    assert a["keypoints_3d"].shape == (2, 17, 3) and a["base_points"].shape == (2, 3)
    assert a["features"].shape == (2, 2, 32, 32, 32) and a["coord_volumes"].shape == (2, 32, 32, 32, 3)
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    for name in a:
        assert a[name].dtype == np.float32 and np.isfinite(a[name]).all(), name
        assert a[name].shape == b[name].shape
        scale = max(float(np.abs(a[name]).max()), 1e-30)
        assert float(np.abs(a[name] - b[name]).max()) <= 1e-5 * scale, name
    # the same model and batch as bench.py builds them (seeds, calibration, conv mode), run once without CUDA graphs
    import lt_b200
    from lt_b200 import testing
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    np.random.seed(0)
    model = lt_b200.VolumetricTriangulationNet(testing.make_config(num_layers=50, volume_size=32), device=dev, backend="native",
                                               conv_mode="tc", use_cuda_graph=False)
    testing.randomize_weights(model, seed=0, calib_size=128, calib_views=1)
    model = model.to(dev).eval()
    images, batch = testing.make_batch(2, 2, image_size=128, seed=0)
    with torch.no_grad():
        kp, feats, vols, _, _, coords, base = model(images.to(dev), None, batch)
    eager = {"keypoints_3d": kp, "features": feats, "volumes": vols, "coord_volumes": coords, "base_points": base}
    for name, t in eager.items():
        want = t.float().cpu().numpy()
        scale = max(float(np.abs(want).max()), 1e-30)
        assert a[name].shape == want.shape and float(np.abs(a[name] - want).max()) <= 1e-4 * scale, name
