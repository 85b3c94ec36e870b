"""bench.py's command line: --steps is validated, and --dump-outputs writes what the timed path delivered in its last step
(the CPU reference arm on any machine, the GPU arm on a B200)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from oracle import bindings as ob

W, H, L = 1920, 1080, 5  # bench.py's C3 frame
COUNTERS = ("primary", "primary_hit", "shadow", "bounce")


def run_bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=900)


def test_steps_must_be_positive():
    r = run_bench("--steps", "0")
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr


def test_reference_arm_dumps_its_last_frame(oracle, tmp_path):
    r = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    frame = np.load(tmp_path / "frame.npy")
    counts = np.load(tmp_path / "ray_counts.npy")
    # the same frame rendered here by the restatement (bench.py uses the reference's own code where oracle/_ref is built;
    # both are bit-identical on this scene)
    flat, lights = ob.dragon_standin_fixture()
    want, cnt = oracle.scene(flat, lights).bvh().render(ob.default_camera(W, H), W, H, trace_limit=L, duplicate_shading=True)
    assert frame.dtype == np.float32 and np.array_equal(frame.view(np.uint32), want.view(np.uint32))
    assert counts.dtype == np.float64 and counts.tolist() == [cnt[k] for k in COUNTERS]
    # Mrays/s x ms per step = the rays of one frame: the line describes the frame that was dumped
    assert line["value"] * line["ms_per_step"] * 1e3 == pytest.approx(counts[0] + counts[2] + counts[3], rel=1e-9)


@pytest.mark.gpu
def test_timed_frame_dump_is_the_rendered_frame(capi, gpu, tmp_path):
    r = run_bench("--gpus", "1", "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    d = capi.dragon_standin()
    s = capi.Scene(d, lights=d.lights)
    rgb, st = s.render(capi.make_camera(W, H), W, H, trace_limit=L)
    frame = np.load(tmp_path / "frame.npy")
    assert frame.dtype == np.float32 and np.array_equal(frame.view(np.uint32), rgb.view(np.uint32))
    assert np.load(tmp_path / "ray_counts.npy").tolist() == [st[k] for k in COUNTERS]
