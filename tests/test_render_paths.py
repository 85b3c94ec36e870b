"""cgrt_render_paths: every level of each pixel's mirror path (the ray trace(level) cast, its hit, its shading point) and each
light's shadow factor at each hit. rgb and the statistics equal cgrt_render_views; level 0 equals cgrt_render_aovs; every level's
depth / tri / normal equal cgrt_intersect_closest on that level's ray; levels without a ray are +0 rays with FLT_MAX, -1 and 0;
every buffer equals the restatement's walk of the recursion (orc_render_paths in tests/oracle_paths.cpp)."""
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, bits, load_golden, same_bits
from oracle import bindings as ob
from test_render_aovs import SPHERES, _scene, oracle_camera
from test_render_views import cameras

W, H = 320, 180
KEYS = ("ray", "depth", "tri", "normal", "position", "visibility")
STATS = ("primary", "primary_hit", "shadow", "bounce", "pipeline", "class_launches", "box_tests", "tri_tests")
FLT_MAX = np.float32(np.finfo(np.float32).max)
PIXEL_TOL = 1.0 / 255.0


@pytest.fixture(scope="session")
def paths_oracle(tmp_path_factory):
    """The restatement with its mirror-path walk (tests/oracle_paths.cpp includes oracle/cgrt_oracle.cpp), compiled with the
    oracle's flags (oracle/Makefile) into a temporary directory: a CPU checker with the orc_ surface plus orc_render_paths."""
    so = str(tmp_path_factory.mktemp("oracle_paths") / "liboracle_paths.so")
    r = subprocess.run(["/usr/bin/g++", "-std=gnu++17", "-O2", "-fopenmp", "-ffp-contract=off", "-fPIC", "-fno-fast-math", "-shared",
                        "-o", so, os.path.join(ROOT, "tests", "oracle_paths.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return ob._CpuChecker(so, "orc_")


def oracle_paths(bvh, cam, W, H, L, Lv, n_lights):
    """(rgb[H,W,3], {key: [Lv,H,W,...]}) of the restatement's walk, Screen layout; tri holds canonical ids (-2 - s sphere s)."""
    f = bvh.lib.lib.orc_render_paths
    f.restype = None
    f.argtypes = [C.c_void_p, C.POINTER(ob.CameraDesc), C.c_int, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 7 + [C.c_int]
    rgb = np.zeros((H, W, 3), np.float32)
    o = dict(ray=np.zeros((Lv, H, W), ob.RAY_DTYPE), depth=np.zeros((Lv, H, W), np.float32), tri=np.zeros((Lv, H, W), np.int32),
             normal=np.zeros((Lv, H, W, 3), np.float32), position=np.zeros((Lv, H, W, 3), np.float32),
             visibility=np.zeros((Lv, H, W, n_lights), np.float32))
    f(bvh.h, C.byref(cam), W, H, L, Lv, rgb.ctypes.data, *[o[k].ctypes.data for k in KEYS], 0)
    return rgb, o


def raw(a):
    """the bytes of an array as unsigned integers (bit-exact comparison of floats, rays and ids)"""
    a = np.ascontiguousarray(a)
    return a.view(np.uint32) if a.dtype.itemsize % 4 == 0 else a.view(np.uint8)


def check_paths(capi, s, cams, L, Lv=None, orc=None, canon=None, W=W, H=H):
    """render_paths against render_views, render_aovs (level 0), cgrt_intersect_closest on every level's rays, the no-ray
    convention and (orc: the restatement's BVH of paths_oracle) the restatement's walk. Returns (rgb, paths, stats)."""
    rgb, P, st = s.render_paths(cams, W, H, trace_limit=L, n_levels=Lv)
    Lv = max(L, 1) if Lv is None else Lv
    assert set(P) == set(KEYS) and P["depth"].shape == (Lv, len(cams), H, W)
    want, sw = s.render_views(cams, W, H, trace_limit=L)
    assert same_bits(rgb, want), L
    assert [st[k] for k in STATS] == [sw[k] for k in STATS], (L, st, sw)
    assert st["kernel_launches"] > sw["kernel_launches"]
    _, aov, _ = s.render_aovs(cams, W, H, trace_limit=L, hits=False)
    assert same_bits(P["depth"][0], aov["depth"]) and np.array_equal(P["tri"][0], aov["tri"]) and same_bits(P["normal"][0], aov["normal"])
    ray = raw(P["ray"]).reshape(Lv, len(cams), H, W, 8)
    cast = ray.any(axis=-1)
    hit = P["tri"] != -1
    none = ~cast
    assert np.all(P["depth"][none] == FLT_MAX) and np.all(P["tri"][none] == -1) and not bits(P["normal"][none]).any()
    assert not bits(P["position"][~hit]).any() and not bits(P["visibility"][~hit]).any()
    assert not np.any(hit & none)
    if L == 0:
        assert not cast.any()
    else:
        for v, cam in enumerate(cams):
            assert np.array_equal(ray[0, v], raw(capi.generate_rays(cam, W, H).reshape(H, W)[::-1]).reshape(H, W, 8)), v
    for l in range(Lv):
        if cast[l].any():
            got = s.intersect(np.ascontiguousarray(P["ray"][l][cast[l]]))
            assert same_bits(P["depth"][l][cast[l]], got["t"]) and np.array_equal(P["tri"][l][cast[l]], got["tri"]), l
            assert same_bits(P["normal"][l][cast[l]], got["n"]), l
        if l > 0:
            assert not np.any(cast[l] & ~hit[l - 1]), l  # a level's ray comes off the hit before it
    if orc is not None:
        nl = P["visibility"].shape[-1]
        for v, cam in enumerate(cams):
            orgb, o = oracle_paths(orc, oracle_camera(cam), W, H, L, Lv, nl)
            assert float(np.abs(rgb[v] - orgb).max()) <= PIXEL_TOL, (L, v)  # the frame's own parity bound (pow in double)
            for k in ("ray", "depth", "normal", "position", "visibility"):
                assert np.array_equal(raw(P[k][:, v]), raw(o[k])), (L, v, k)
            t = P["tri"][:, v]
            assert np.array_equal(np.where(t >= 0, canon[np.maximum(t, 0)], t), o["tri"]), (L, v)
    return rgb, P, st


# ---- argument validation (no GPU needed: refused before any CUDA call, valid ones fail on a host-only scene) ---------------
def _call(capi, s, cams, n, p, Lv, nl, out, paths, device):
    lib = capi.load_library()
    arr = (capi.Camera * max(len(cams), 1))(*cams)
    ptr = C.c_void_p(out.ctypes.data) if out is not None else None
    b = C.byref(paths) if paths is not None else None
    if device:
        return lib.cgrt_render_paths_device(s.h, arr if cams else None, n, C.byref(p), Lv, nl, ptr, b, None)
    st = capi.RenderStats()
    return lib.cgrt_render_paths(s.h, arr if cams else None, n, C.byref(p), Lv, nl, ptr, b, C.byref(st))


@pytest.mark.parametrize("device", [False, True])
def test_paths_refuse_bad_arguments(capi, device):
    s = capi.Scene(ob.random_soup(10, seed=1, scale=0.3), host_only=True, lights=np.zeros((2, 6), np.float32))
    s.set_spherical_lights(np.array([[0, 0.4, 0, 0.1, 1, 1, 1]], np.float32), seed=7)
    w, h = 16, 8
    cams = [capi.make_camera(w, h)] * 2
    out = np.zeros((2, h, w, 3), np.float32)
    buf = np.zeros(64, np.float32)
    depth = capi.PathBuffers(None, buf.ctypes.data)
    vis = capi.PathBuffers(None, None, None, None, None, buf.ctypes.data)
    ok = capi.render_params(w, h, 3)
    bad = [
        (cams, 0, ok, 3, 3, out, depth),                                    # no view
        (cams, 1025, ok, 3, 3, out, depth),                                 # more than 1024
        ([], 2, ok, 3, 3, out, depth),                                      # null cams
        (cams, 2, ok, 3, 3, None, depth),                                   # null rgb
        (cams, 1024, capi.render_params(512, 513, 1), 1, 3, out, depth),    # n_views x W x H > 2^28
        (cams, 1024, capi.render_params(1, 1 << 18, 1), 1, 3, out, depth),  # 2^31 slots of whole 8 x 8 tiles
        (cams, 2, capi.render_params(w, h, 3, world=2), 3, 3, out, depth),  # a share of a multi-GPU frame
        (cams, 2, capi.render_params(w, h, 3, flags=capi.RENDER_COUNT), 3, 3, out, depth),
        (cams, 2, capi.render_params(w, h, 3, flags=capi.RENDER_SCREEN_LAYOUT), 3, 3, out, depth),
        (cams, 2, ok, 3, 3, out, None),                                     # null paths
        (cams, 2, ok, 3, 3, out, capi.PathBuffers()),                       # no buffer requested
        (cams, 2, ok, 0, 3, out, depth),                                    # n_levels < 1
        (cams, 2, ok, 4, 3, out, depth),                                    # n_levels > trace_limit
        (cams, 2, capi.render_params(w, h, 0), 2, 3, out, depth),           # n_levels > 1 at trace limit 0
        (cams, 64, capi.render_params(1024, 1024, 5), 5, 3, out, depth),    # 5 x 64 x 2^20 > 2^28 path pixels
        (cams, 32, capi.render_params(1024, 1024, 5), 3, 3, out, vis),      # 3 x 3 x 32 x 2^20 > 2^28 visibility entries
        (cams, 2, ok, 3, 2, out, depth),                                    # n_lights below the scene's
        (cams, 2, ok, 3, 4, out, depth),                                    # n_lights above the scene's
        (cams, 2, ok, 3, -1, out, depth),
    ]
    for i, (c, n, p, Lv, nl, o, b) in enumerate(bad):
        assert _call(capi, s, c, n, p, Lv, nl, o, b, device) == capi.CGRT_ERR_INVALID, i
    # valid arguments reach the device check: a host-only scene has no device state
    for k in range(6):
        one = capi.PathBuffers(*[buf.ctypes.data if j == k else None for j in range(6)])
        assert _call(capi, s, cams, 2, ok, 3, 3, out, one, device) == capi.CGRT_ERR_NO_DEVICE, k
    for p, Lv in ((ok, 1), (capi.render_params(w, h, 0), 1), (capi.render_params(w, h, 3, flags=capi.RENDER_PROFILE_ALL), 2)):
        assert _call(capi, s, cams, 2, p, Lv, 3, out, depth, device) == capi.CGRT_ERR_NO_DEVICE
    # 3 x 32 x 2^20 path pixels fit when visibility is not requested
    assert _call(capi, s, cams, 32, capi.render_params(1024, 1024, 5), 3, 3, out, depth, device) == capi.CGRT_ERR_NO_DEVICE
    # the light count follows set_lights
    s.set_lights(np.zeros((3, 6), np.float32))
    assert _call(capi, s, cams, 2, ok, 3, 3, out, depth, device) == capi.CGRT_ERR_INVALID
    assert _call(capi, s, cams, 2, ok, 3, 4, out, depth, device) == capi.CGRT_ERR_NO_DEVICE
    s.close()


@pytest.mark.parametrize("name", ["cornell", "monkey"])
def test_oracle_paths_are_its_recursion(oracle, paths_oracle, name):
    """The restatement's walk: its frame is orc_render's bit for bit, its level-0 ray is orc_generate_rays', and every level's
    hit is its own intersect on that level's ray."""
    g = load_golden(name)
    b = paths_oracle.scene(g.flat, g.lights).bvh()
    cam = ob.default_camera(g.W, g.H)
    nl = len(g.lights)
    for L in (1, 3):
        rgb, o = oracle_paths(b, cam, g.W, g.H, L, L, nl)
        want, _ = oracle.scene(g.flat, g.lights).bvh().render(cam, g.W, g.H, trace_limit=L)
        assert same_bits(rgb, want), L
        r0 = paths_oracle.generate_rays(cam, g.W, g.H).reshape(g.H, g.W)[::-1]
        assert np.array_equal(raw(o["ray"][0]), raw(r0)), L
        cast = raw(o["ray"]).reshape(L, g.H, g.W, 8).any(axis=-1)
        for l in range(L):
            h = b.intersect(np.ascontiguousarray(o["ray"][l][cast[l]]))
            assert same_bits(o["depth"][l][cast[l]], h["t"]) and np.array_equal(o["tri"][l][cast[l]], h["tri"]), (L, l)
            assert same_bits(o["normal"][l][cast[l]], h["n"]), (L, l)
            assert np.all(o["depth"][l][~cast[l]] == FLT_MAX) and np.all(o["tri"][l][~cast[l]] == -1), (L, l)
        hit = o["tri"] != -1
        assert not bits(o["position"][~hit]).any() and not bits(o["visibility"][~hit]).any()
        assert set(np.unique(o["visibility"])) <= {0.0, 1.0} and o["visibility"][hit].any()
        if L == 3 and name == "cornell":
            assert cast[1].any()  # the Cornell box has a mirror


# ---- GPU ----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", params=["cornell", "dragon", "cornell_spheres"])
def scene(request, capi, gpu, paths_oracle):
    s, orc, canon = _scene(capi, request.param, paths_oracle)
    yield request.param, s, orc, canon
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("L", [0, 1, 2, 5])
def test_paths_equal_intersect_and_oracle(capi, scene, L):
    """Six views and a batch of one, n_levels = the limit and below it (the first levels of the same paths)."""
    name, s, orc, canon = scene
    cams = cameras(capi, W, H)
    _, full, _ = check_paths(capi, s, cams, L, orc=orc, canon=canon)
    check_paths(capi, s, cams[3:4], L, orc=orc, canon=canon)
    if L >= 2:
        _, part, _ = check_paths(capi, s, cams, L, Lv=L - 1)
        for k in KEYS:
            assert np.array_equal(raw(part[k]), raw(full[k][:L - 1])), (L, k)
    if L >= 2 and name != "dragon":
        assert raw(full["ray"][1]).any()  # a mirror reflects
        if name == "cornell_spheres":
            assert (full["tri"][1] <= -2).any() or (full["tri"][0] <= -2).any()


@pytest.mark.gpu
def test_one_buffer_at_a_time(capi, gpu):
    """A buffer that is not requested is not written; each one alone equals the full call's."""
    s, _, _ = _scene(capi, "cornell_spheres")
    cams = cameras(capi, W, H)[:2]
    _, full, _ = s.render_paths(cams, W, H, trace_limit=3)
    for k in KEYS:
        _, one, _ = s.render_paths(cams, W, H, trace_limit=3, **{j: j == k for j in KEYS})
        assert set(one) == {k} and np.array_equal(raw(one[k]), raw(full[k])), k
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("L", [1, 2, 5])
def test_spherical_light_visibility(capi, gpu, paths_oracle, L):
    """Radius 0: the samples all aim at the centre, so each factor is 0 or 1 and equals the restatement's bit for bit. Radius
    > 0: every factor is k/200 in [0, 1] and some are strictly between."""
    g = load_golden("cornell")
    cams = cameras(capi, W, H)[:3]
    s = capi.Scene(g.flat, lights=g.lights)
    sph0 = np.array([[0.1, 0.45, 0.05, 0.0, 0.9, 0.8, 0.6]], np.float32)
    s.set_spherical_lights(sph0, seed=7)
    cs = paths_oracle.scene(g.flat, g.lights)
    cs.set_spherical_lights(sph0, seed=7)
    orc = cs.bvh()
    canon = g.flat.canonical_ids()
    _, P, st = check_paths(capi, s, cams, L, orc=orc, canon=canon)
    assert st["pipeline"] == 2
    nP = len(g.lights)
    hit = P["tri"] != -1
    assert np.any(P["visibility"][..., nP][hit] == 1.0) and np.any(P["visibility"][..., nP][hit] == 0.0)
    s.set_spherical_lights(np.array([[0.1, 0.45, 0.05, 0.15, 0.9, 0.8, 0.6], [-0.3, 0.4, 0.2, 0.1, 0.3, 0.4, 1.0]], np.float32),
                           seed=3)
    _, P, _ = check_paths(capi, s, cams, L)
    v = P["visibility"][..., nP:]
    k = np.rint(v * 200.0)
    assert np.all((k >= 0) & (k <= 200)) and same_bits(v, (k / np.float32(200.0)).astype(np.float32))
    assert np.any((v > 0) & (v < 1))
    s.close()


@pytest.mark.gpu
def test_paths_device_form(capi, gpu):
    """The device form on a non-default stream equals the host form; its statistics come from collect_stats."""
    import torch
    s, _, _ = _scene(capi, "cornell_spheres")
    cams = cameras(capi, W, H)
    L, Lv = 5, 4
    want, wp, sw = s.render_paths(cams, W, H, trace_limit=L, n_levels=Lv)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        d_rgb = torch.full(want.shape, float("nan"), dtype=torch.float32, device="cuda")
        d = {k: torch.full(v.view(np.uint8).shape, 0x7f, dtype=torch.uint8, device="cuda") for k, v in wp.items()}
    s.render_paths_device(cams, capi.render_params(W, H, L), Lv, d_rgb.data_ptr(), {k: v.data_ptr() for k, v in d.items()},
                          stream.cuda_stream)
    st = s.collect_stats()
    stream.synchronize()
    assert same_bits(d_rgb.cpu().numpy(), want)
    for k in KEYS:
        assert np.array_equal(d[k].cpu().numpy(), np.ascontiguousarray(wp[k]).view(np.uint8)), k
    keys = ("primary", "primary_hit", "shadow", "bounce", "pipeline", "kernel_launches")
    assert [st[k] for k in keys] == [sw[k] for k in keys]
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("exact_only", [False, True])
def test_paths_leave_no_state_behind(capi, gpu, exact_only):
    """Calls of other limits, sizes and views interleaved on one scene equal what a second scene renders, and the device form
    overwrites every level of a buffer that holds another frame's deeper paths (exact_only: the path pipeline)."""
    import torch
    g = load_golden("cornell")
    s, ref = [capi.Scene(g.flat, lights=g.lights, exact_only=exact_only) for _ in range(2)]
    s.set_spheres(SPHERES)
    ref.set_spheres(SPHERES)
    cams = cameras(capi, W, H)
    near = [capi.make_camera(W, H, dist=1.2)] * 2   # the box fills the frame
    far = [capi.make_camera(W, H, dist=9.0)] * 2    # the box is small: most pixels miss
    for step in range(2):
        for cs, w, h, L in ((cams[:3], W, H, 3), (cameras(capi, 200, 150), 200, 150, 5), (near, W, H, 4), (far, W, H, 4),
                            (near, W, H, 0)):
            a = s.render_paths(cs, w, h, trace_limit=L)
            b = ref.render_paths(cs, w, h, trace_limit=L)
            assert same_bits(a[0], b[0]) and all(np.array_equal(raw(a[1][k]), raw(b[1][k])) for k in KEYS), (step, w, L)
            assert same_bits(s.render_views(cs, w, h, trace_limit=L)[0], b[0])
    _, deep, _ = s.render_paths(near, W, H, trace_limit=4)
    _, shallow, _ = s.render_paths(far, W, H, trace_limit=4)
    d = {k: torch.from_numpy(np.ascontiguousarray(v).view(np.uint8).copy()).cuda() for k, v in deep.items()}
    d_rgb = torch.zeros((2, H, W, 3), dtype=torch.float32, device="cuda")
    s.render_paths_device(far, capi.render_params(W, H, 4), 4, d_rgb.data_ptr(), {k: v.data_ptr() for k, v in d.items()})
    torch.cuda.synchronize()
    assert raw(deep["ray"][1]).any()
    for k in KEYS:
        assert np.array_equal(d[k].cpu().numpy(), np.ascontiguousarray(shallow[k]).view(np.uint8)), k
    s.close()
    ref.close()


@pytest.mark.gpu
def test_paths_at_benchmark_size(capi, gpu):
    """C3 (dragon stand-in, 1920 x 1080, trace limit 5): one view with every check, and 8 views (depth and tri), whose view 0 is
    the one-view call's."""
    flat, lights = ob.dragon_standin_fixture()
    s = capi.Scene(flat, lights=lights)
    w, h = 1920, 1080
    cams = [capi.make_camera(w, h)] + [capi.make_camera(w, h, look_at=(0.02 * k, 0.0, 0.0)) for k in range(1, 5)] + \
           [capi.make_camera(w, h, euler_deg=(20.0, 20.0 + 15 * k, 0.0)) for k in range(1, 4)]
    _, one, st = check_paths(capi, s, cams[:1], 5, W=w, H=h)
    assert st["pipeline"] == 3
    rgb, P, st = s.render_paths(cams, w, h, trace_limit=5, ray=False, normal=False, position=False, visibility=False)
    want, sw = s.render_views(cams, w, h, trace_limit=5)
    assert same_bits(rgb, want) and [st[k] for k in STATS] == [sw[k] for k in STATS]
    assert same_bits(P["depth"][:, 0], one["depth"][:, 0]) and np.array_equal(P["tri"][:, 0], one["tri"][:, 0])
    _, aov, _ = s.render_aovs(cams, w, h, trace_limit=5, normal=False, hits=False)
    assert same_bits(P["depth"][0], aov["depth"]) and np.array_equal(P["tri"][0], aov["tri"])
    s.close()


# ---- every pipeline, each forced in its own process -----------------------------------------------------------------------
_WORKER = r"""
import hashlib, json, sys
import numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
import __graft_entry__ as ge
from oracle import bindings as ob
from test_render_views import cameras
capi = ge.load_package().capi
flat, lights = ob.dragon_standin_fixture()
s = capi.Scene(flat, lights=lights, exact_only=sys.argv[2] == "1")
W, H = 320, 180
cams = cameras(capi, W, H)
out = {}
for L in (3, 0, 1):
    rgb, P, st = s.render_paths(cams, W, H, trace_limit=L)
    want, sw = s.render_views(cams, W, H, trace_limit=L)
    same = bool(np.array_equal(rgb.view(np.uint32), want.view(np.uint32)))
    sha = hashlib.sha1(b"".join(np.ascontiguousarray(P[k]).tobytes() for k in capi.PATH_KEYS)).hexdigest()
    out[L] = dict(same=same, sha=sha, pipeline=st["pipeline"], views_pipeline=sw["pipeline"],
                  launches=st["kernel_launches"] - sw["kernel_launches"], mirrors=int(np.ascontiguousarray(P["ray"][-1]).view(np.uint32).any()))
print("RESULT " + json.dumps(out))
"""


@pytest.mark.gpu
def test_paths_on_every_pipeline(gpu):
    res = {}
    for name, pref, exact, pipeline in (("wave", "wave", False, 3), ("rounds", "rounds", False, 2), ("paths", None, True, 1)):
        env = dict(os.environ)
        env.pop("CGRT_PIPELINE", None)
        if pref:
            env["CGRT_PIPELINE"] = pref
        r = subprocess.run([sys.executable, "-c", _WORKER, ROOT, "1" if exact else "0"], env=env, capture_output=True, text=True,
                           timeout=600)
        line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
        assert r.returncode == 0 and line, (name, r.stdout[-800:], r.stderr[-2000:])
        res[name] = json.loads(line[0][7:])
        for L, v in res[name].items():
            assert v["pipeline"] == pipeline and v["views_pipeline"] == pipeline and v["same"], (name, L, v)
            # the pass: one kernel, two for the path pipeline's records (every pixel's level 0 and misses, then the paths)
            assert v["launches"] == (2 if pipeline == 1 and L != "0" else 1), (name, L, v)
    assert res["wave"]["3"]["mirrors"]
    for name in ("rounds", "paths"):
        for L in res["wave"]:
            assert res[name][L]["sha"] == res["wave"][L]["sha"], (name, L)
