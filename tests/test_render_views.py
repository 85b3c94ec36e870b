"""cgrt_render_views: several cameras of one scene rendered as one frame. View v of a batch must be bit for bit the frame
cgrt_render returns for camera v, with the batch's ray statistics the sums of those frames'."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, bits, load_golden, same_bits
from oracle import bindings as ob

RAYS = ("primary", "primary_hit", "shadow", "bounce")
W, H = 320, 180


def cameras(capi, W, H):
    """The preset, two motion-blur look-ats, other Euler angles, another fovy and distance, and view 0 again."""
    return [capi.make_camera(W, H),
            capi.make_camera(W, H, look_at=(0.01, 0.0, 0.0)),
            capi.make_camera(W, H, look_at=(0.15, 0.0, 0.0)),
            capi.make_camera(W, H, euler_deg=(-15.0, 40.0, 5.0)),
            capi.make_camera(W, H, fovy_deg=35.0, dist=4.0),
            capi.make_camera(W, H)]


def check_views(capi, s, cams, W, H, L, ref=None):
    """Batch of `cams` on scene `s` against single renders on `ref` (default: the same scene). Returns the batch's stats."""
    got, st = s.render_views(cams, W, H, trace_limit=L)
    assert got.shape == (len(cams), H, W, 3)
    total = dict.fromkeys(RAYS, 0)
    for v, cam in enumerate(cams):
        want, sv = (ref or s).render(cam, W, H, trace_limit=L)
        assert same_bits(got[v], want), (v, L, float(np.abs(got[v] - want).max()))
        for k in RAYS:
            total[k] += sv[k]
    assert {k: st[k] for k in RAYS} == total, (L, st, total)
    if L == 0:
        assert not bits(got).any() and st["primary"] == 0
    return st


# ---- argument validation (no GPU needed: refused before any CUDA call, valid ones fail on a host-only scene) ---------------
def _call(capi, s, cams, n, p, out, device):
    lib = capi.load_library()
    arr = (capi.Camera * max(len(cams), 1))(*cams)
    ptr = C.c_void_p(out.ctypes.data) if out is not None else None
    if device:
        return lib.cgrt_render_views_device(s.h, arr if cams else None, n, C.byref(p), ptr, None)
    st = capi.RenderStats()
    return lib.cgrt_render_views(s.h, arr if cams else None, n, C.byref(p), ptr, C.byref(st))


@pytest.mark.parametrize("device", [False, True])
def test_views_refuse_bad_arguments(capi, device):
    s = capi.Scene(ob.random_soup(10, seed=1, scale=0.3), host_only=True)
    w, h = 16, 8
    cams = [capi.make_camera(w, h)] * 2
    out = np.zeros((2, h, w, 3), np.float32)
    ok = capi.render_params(w, h)
    bad = [
        (cams, 0, ok, out),                                   # no view
        (cams, 1025, ok, out),                                # more than 1024
        ([], 2, ok, out),                                     # null cams
        (cams, 2, ok, None),                                  # null output
        (cams, 1024, capi.render_params(512, 513), out),      # n_views x W x H > 2^28
        (cams, 1024, capi.render_params(1, 1 << 18), out),    # 2^28 pixels, but 2^31 slots of whole 8 x 8 tiles
        (cams, 2, capi.render_params(w, h, world=2), out),    # a share of a multi-GPU frame
        (cams, 2, capi.render_params(w, h, flags=capi.RENDER_COUNT), out),
        (cams, 2, capi.render_params(w, h, flags=capi.RENDER_SCREEN_LAYOUT), out),
    ]
    for i, (c, n, p, o) in enumerate(bad):
        assert _call(capi, s, c, n, p, o, device) == capi.CGRT_ERR_INVALID, i
    # valid arguments reach the device check: a host-only scene has no device state
    assert _call(capi, s, cams, 2, ok, out, device) == capi.CGRT_ERR_NO_DEVICE
    assert _call(capi, s, cams, 2, capi.render_params(w, h, flags=capi.RENDER_PROFILE_ALL), out, device) == capi.CGRT_ERR_NO_DEVICE
    # the largest batch that is allowed: 1024 views of 512 x 512 = 2^28 pixel slots
    big = [capi.make_camera(512, 512)] * 1024
    assert _call(capi, s, big, 1024, capi.render_params(512, 512), np.zeros(1, np.float32), device) == capi.CGRT_ERR_NO_DEVICE


# ---- GPU ----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dragon(capi, gpu):
    flat, lights = ob.dragon_standin_fixture()
    return capi.Scene(flat, lights=lights)


@pytest.fixture(scope="module")
def cornell(capi, gpu):
    g = load_golden("cornell")
    return capi.Scene(g.flat, lights=g.lights)


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["cornell", "dragon"])
@pytest.mark.parametrize("L", [0, 1, 2, 5])
def test_views_equal_single_frames(capi, request, scene, L):
    s = request.getfixturevalue(scene)
    check_views(capi, s, cameras(capi, W, H), W, H, L)


@pytest.mark.gpu
def test_one_view_is_cgrt_render(capi, dragon):
    cam = capi.make_camera(W, H)
    for L in (1, 2, 5):
        got, st = dragon.render_views([cam], W, H, trace_limit=L)
        want, sw = dragon.render(cam, W, H, trace_limit=L)
        assert same_bits(got[0], want)
        assert [st[k] for k in RAYS + ("pipeline",)] == [sw[k] for k in RAYS + ("pipeline",)], (L, st, sw)


@pytest.mark.gpu
def test_views_with_spherical_lights(capi, gpu):
    """Soft-shadow samples are keyed by the pixel's slot in its own view's frame: batched views equal their single renders."""
    g = load_golden("cornell")
    s = capi.Scene(g.flat, lights=g.lights)
    s.set_spherical_lights(np.array([[0, 0.45, 0, 0.1, 1, 1, 1]], np.float32), seed=7)
    w, h = 160, 120
    st = check_views(capi, s, cameras(capi, w, h), w, h, 2)
    assert st["pipeline"] == 2  # soft shadows are a pass of the round pipeline


@pytest.mark.gpu
def test_views_device_form(capi, dragon):
    import torch
    lib = capi.load_library()
    cams = cameras(capi, W, H)
    L = 5
    want, sw = dragon.render_views(cams, W, H, trace_limit=L)
    n = want.size * 4
    d = C.c_void_p()
    capi.check(lib.cgrt_device_malloc(0, n, C.byref(d)))
    try:
        stream = torch.cuda.Stream()
        dragon.render_views_device(cams, capi.render_params(W, H, L), d.value, stream.cuda_stream)
        st = dragon.collect_stats()
        got = np.zeros_like(want)
        capi.check(lib.cgrt_memcpy_d2h(0, C.c_void_p(got.ctypes.data), d, n))
    finally:
        lib.cgrt_device_free(0, d)
    assert same_bits(got, want)
    assert [st[k] for k in RAYS + ("pipeline", "kernel_launches")] == [sw[k] for k in RAYS + ("pipeline", "kernel_launches")]


@pytest.mark.gpu
def test_views_leave_no_state_behind(capi, gpu):
    """Single frames, batches of different sizes and a frame of another shape, interleaved on one scene: each equals what a
    second scene renders frame by frame (tile cache, primaryPixels and the wave tuner are keyed correctly)."""
    flat, lights = ob.dragon_standin_fixture()
    s, ref = capi.Scene(flat, lights=lights), capi.Scene(flat, lights=lights)
    cams = cameras(capi, W, H)
    L = 3
    for step in range(2):
        one, st1 = s.render(cams[3], W, H, trace_limit=L)
        want, sw = ref.render(cams[3], W, H, trace_limit=L)
        assert same_bits(one, want) and [st1[k] for k in RAYS] == [sw[k] for k in RAYS]
        check_views(capi, s, cams[:3], W, H, L, ref=ref)
        check_views(capi, s, cams, W, H, L, ref=ref)
        w2, h2 = 200, 150
        other, st2 = s.render(capi.make_camera(w2, h2), w2, h2, trace_limit=L)
        want2, sw2 = ref.render(capi.make_camera(w2, h2), w2, h2, trace_limit=L)
        assert same_bits(other, want2) and [st2[k] for k in RAYS] == [sw2[k] for k in RAYS], step
        check_views(capi, s, [capi.make_camera(w2, h2, euler_deg=(20.0, 20.0 + 30 * k, 0.0)) for k in range(4)], w2, h2, L, ref=ref)


@pytest.mark.gpu
def test_views_at_benchmark_size(capi, gpu):
    """8 views of C3 (dragon stand-in, 1920 x 1080, trace limit 5)."""
    flat, lights = ob.dragon_standin_fixture()
    s = capi.Scene(flat, lights=lights)
    w, h = 1920, 1080
    cams = [capi.make_camera(w, h)] + [capi.make_camera(w, h, look_at=(0.02 * k, 0.0, 0.0)) for k in range(1, 5)] + \
           [capi.make_camera(w, h, euler_deg=(20.0, 20.0 + 15 * k, 0.0)) for k in range(1, 4)]
    st = check_views(capi, s, cams, w, h, 5)
    assert st["pipeline"] == 3


# ---- every pipeline, each forced in its own process -----------------------------------------------------------------------
_WORKER = r"""
import hashlib, json, sys
import numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
import __graft_entry__ as ge
from oracle import bindings as ob
from test_render_views import cameras, RAYS
capi = ge.load_package().capi
flat, lights = ob.dragon_standin_fixture()
s = capi.Scene(flat, lights=lights, exact_only=sys.argv[2] == "1")
W, H = 320, 180
cams = cameras(capi, W, H)
out = {}
for L in (3, 0, 1):
    got, st = s.render_views(cams, W, H, trace_limit=L)
    same, rays, pipes = True, [0, 0, 0, 0], set()
    for v, cam in enumerate(cams):
        want, sv = s.render(cam, W, H, trace_limit=L)
        same = same and np.array_equal(got[v].view(np.uint32), want.view(np.uint32))
        rays = [a + sv[k] for a, k in zip(rays, RAYS)]
        pipes.add(sv["pipeline"])
    out[L] = dict(same=bool(same), rays=[st[k] for k in RAYS], single_rays=rays, pipeline=st["pipeline"],
                  single_pipelines=sorted(pipes), black=not got.view(np.uint32).any())
print("RESULT " + json.dumps(out))
"""


@pytest.mark.gpu
@pytest.mark.parametrize("name,pref,exact,pipeline", [("wave", "wave", False, 3), ("rounds", "rounds", False, 2),
                                                      ("paths", None, True, 1)])
def test_views_on_every_pipeline(gpu, name, pref, exact, pipeline):
    env = dict(os.environ)
    env.pop("CGRT_PIPELINE", None)
    if pref:
        env["CGRT_PIPELINE"] = pref
    r = subprocess.run([sys.executable, "-c", _WORKER, ROOT, "1" if exact else "0"], env=env, capture_output=True, text=True,
                       timeout=600)
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
    assert r.returncode == 0 and line, (name, r.stdout[-800:], r.stderr[-2000:])
    for L, v in json.loads(line[0][7:]).items():
        assert v["pipeline"] == pipeline and v["single_pipelines"] == [pipeline], (name, L, v)
        assert v["same"] and v["rays"] == v["single_rays"], (name, L, v)
        if L == "0":
            assert v["black"], (name, v)
