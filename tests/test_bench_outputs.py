"""bench.py --dump-outputs: the film of the last timed step, the same for the same workload whatever --steps / --warmup
say, and --steps is the number of steps the counters saw."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, bits


def _bench(out_dir, steps, warmup):
    r = subprocess.run([sys.executable, "bench.py", "--workload", "small", "--steps", str(steps), "--warmup", str(warmup),
                        "--no-cpu-baseline", "--dump-outputs", str(out_dir)],
                       cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, "bench.py", "--steps", "0"], cwd=ROOT, capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and "--steps must be at least 1" in r.stderr


@pytest.mark.gpu
def test_dumped_film_is_independent_of_the_step_count(tmp_path):
    a = _bench(tmp_path / "a", 1, 0)
    b = _bench(tmp_path / "b", 3, 1)
    w, h = a["config"]["resolution"]
    spp = a["config"]["spp"]
    for line, steps in ((a, 1), (b, 3)):
        assert line["steps"] == steps
        assert line["ray_mix_per_step"]["camera"] == w * h * spp, "the counters did not see exactly --steps renders"
    for name, shape in (("image_rgb", (h, w, 3)), ("film_raw", (h, w, 4))):
        x, y = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert x.dtype == np.float32 and x.shape == shape
        assert np.array_equal(bits(x), bits(y)), name
    assert float(np.load(tmp_path / "a" / "image_rgb.npy").max()) > 0, "the dumped image is black"
    assert sorted(os.listdir(tmp_path / "a")) == ["film_raw.npy", "image_rgb.npy"]
