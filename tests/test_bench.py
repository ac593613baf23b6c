"""bench.py --dump-outputs: the outputs of the timed path, identical from run to run, under 64 MB at 4K."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

W, H, WARMUP = 96, 64, 1


def _bench(out, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(WARMUP), "--width", str(W),
           "--height", str(H), "--tris", "20000", "--no-cpu-baseline", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
def test_dump_outputs_repeat_bit_for_bit(tmp_path):
    runs = {steps: _bench(tmp_path / str(steps), steps) for steps in (2, 3)}
    again = _bench(tmp_path / "again", 2)
    for steps, line in runs.items():
        assert line["steps"] == steps and len(line["step_wall_ms"]) == steps
    out = {d: {n: np.load(tmp_path / d / f"{n}.npy") for n in ("accum", "accum_pixel", "ray_counts")} for d in ("2", "3", "again")}
    for name, a in out["2"].items():
        assert a.dtype in (np.float32, np.float64), name
        assert np.array_equal(a.view(np.uint8), out["again"][name].view(np.uint8)), name
    a = out["2"]
    assert a["accum"].shape == (W * H, 3) and np.array_equal(a["accum_pixel"], np.arange(W * H))
    assert np.isfinite(a["accum"]).all() and a["accum"].max() > 0
    # one more timed step: 8 more samples per pixel, and more rays
    assert (out["3"]["accum"].sum() > a["accum"].sum()) and (out["3"]["ray_counts"] > a["ray_counts"]).all()
    assert a["ray_counts"][0] >= 2 * 8 * W * H   # every timed step traces 8 primary rays per pixel


def test_dump_of_the_default_4k_frame_is_a_fixed_sample_under_64_mb(tmp_path):
    import bench
    h, w = bench.HEIGHT, bench.WIDTH
    img = np.random.default_rng(1).random((h, w, 3), dtype=np.float32)
    d = bench.dump_arrays(img, 5.0, 7.0)
    pix = d["accum_pixel"]
    assert d["accum"].shape == (bench.DUMP_PIXELS, 3) and d["accum"].dtype == np.float32 and pix.dtype == np.float64
    assert np.all(np.diff(pix) > 0) and pix[0] >= 0 and pix[-1] < w * h          # distinct pixels of the frame
    p = pix.astype(np.int64)
    assert np.array_equal(d["accum"], img[p // w, p % w])
    assert d["ray_counts"].tolist() == [5.0, 7.0]
    assert np.array_equal(bench.dump_arrays(img, 5.0, 7.0)["accum_pixel"], pix)   # the same sample every run
    bench.write_dump(tmp_path, d)
    assert sorted(os.listdir(tmp_path)) == ["accum.npy", "accum_pixel.npy", "ray_counts.npy"]
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64e6
