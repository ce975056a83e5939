"""bench.py --dump-outputs: the dumped arrays are the headline's BoxBlur output on its seeded inputs (recomputed here
with the CPU oracle), in float32, within 64 MB; and the arguments that cannot describe a run are refused."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
BENCH = [sys.executable, str(ROOT / "bench.py")]


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_refuses_arguments(argv):
    out = subprocess.run(BENCH + argv, capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and "error:" in out.stderr, out.stderr


@pytest.mark.gpu
def test_dump_outputs_is_the_headline_output(tmp_path):
    import oracle_api as oa
    import vapoursynth_zip_b200 as vz

    out = subprocess.run(BENCH + ["--steps", "2", "--warmup", "1", "--no-configs", "--no-cpu", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-4000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["value"] > 0

    files = sorted(tmp_path.glob("*.npy"))
    assert [f.name for f in files] == ["boxblur_u.npy", "boxblur_v.npy", "boxblur_y.npy", "frame_numbers.npy"]
    assert sum(f.stat().st_size for f in files) <= 64 << 20
    planes = [np.load(tmp_path / f"boxblur_{c}.npy") for c in "yuv"]
    frame_nos = np.load(tmp_path / "frame_numbers.npy")
    assert all(p.dtype == np.float32 for p in planes) and frame_nos.dtype == np.float64
    assert planes[0].shape == (len(frame_nos), 1080, 1920) and planes[1].shape == planes[2].shape == (len(frame_nos), 540, 960)

    src = vz.DeviceClip("YUV420P16", 1920, 1080, 1)
    for k, n in enumerate(frame_nos.astype(int)):
        src.fill_noise(seed=1234, first_frame_no=int(n))
        want = oa.boxblur({"format": "YUV420P16", "planes": src.download(0)}, hradius=13, hpasses=5, vradius=13, vpasses=5)
        for p in range(3):
            assert np.array_equal(planes[p][k], want["planes"][p].astype(np.float32)), (int(n), p)
    src.free()
