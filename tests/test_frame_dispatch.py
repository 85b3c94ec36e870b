"""One of four kernel sets renders each frame (cgrt_render_stats.pipeline): the counting wavefront (CGRT_RENDER_COUNT), the path
pipeline (scenes without a search tree), the round pipeline and k_wave. Forced one at a time, they must render the same frames
with the same ray counts, down to the black frame of trace limit 0."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIMITS = (3, 0, 1)  # trace limit 0 after a deeper frame: its statistics must not read state the previous frame left behind

_WORKER = r"""
import hashlib, json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import __graft_entry__ as ge
from oracle import bindings as ob
capi = ge.load_package().capi
flat, lights = ob.dragon_standin_fixture()
s = capi.Scene(flat, lights=lights, exact_only=sys.argv[2] == "1")
flags = capi.RENDER_COUNT if sys.argv[3] == "1" else 0
W, H = 320, 180
cam = capi.make_camera(W, H)
out = {}
for L in (%s):
    rgb, st = s.render(cam, W, H, trace_limit=L, flags=flags)
    out[L] = dict(sha=hashlib.sha1(np.ascontiguousarray(rgb).tobytes()).hexdigest(),
                  black=int(np.count_nonzero(np.ascontiguousarray(rgb).view(np.uint32))) == 0,
                  rays=[st[k] for k in ("primary", "primary_hit", "shadow", "bounce")],
                  launches=st["kernel_launches"], pipeline=st["pipeline"])
print("RESULT " + json.dumps(out))
""" % ", ".join(str(L) for L in LIMITS)

# name: (CGRT_PIPELINE, exact-only scene, CGRT_RENDER_COUNT, expected cgrt_render_stats.pipeline)
VARIANTS = {
    "count": (None, False, True, 0),
    "paths": (None, True, False, 1),
    "rounds": ("rounds", False, False, 2),
    "wave": ("wave", False, False, 3),
}


@pytest.mark.gpu
def test_every_pipeline_renders_the_same_frame(gpu):
    """The pipeline choice is read once per process, so every pipeline renders in its own subprocess."""
    res = {}
    for name, (pref, exact, count, _) in VARIANTS.items():
        env = dict(os.environ)
        env.pop("CGRT_PIPELINE", None)
        if pref:
            env["CGRT_PIPELINE"] = pref
        r = subprocess.run([sys.executable, "-c", _WORKER, ROOT, "1" if exact else "0", "1" if count else "0"], env=env,
                           capture_output=True, text=True, timeout=600)
        line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
        assert r.returncode == 0 and line, (name, r.stdout[-800:], r.stderr[-2000:])
        res[name] = json.loads(line[0][7:])
    base = res["wave"]
    for name, (_, _, _, pipeline) in VARIANTS.items():
        for L in LIMITS:
            v = res[name][str(L)]
            assert v["pipeline"] == pipeline, (name, L, v["pipeline"])
            if L == 0:
                assert v["black"] and v["launches"] == 0, (name, v)
            assert v["sha"] == base[str(L)]["sha"] and v["rays"] == base[str(L)]["rays"], (name, L, v, base[str(L)])
