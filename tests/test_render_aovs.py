"""cgrt_render_aovs: per-pixel depth, triangle id, normal and hit-count buffers with the frame. The frame equals cgrt_render_views;
depth, tri and normal equal cgrt_intersect_closest on the rays of cgrt_generate_rays bit for bit; hits equals the restatement's
count of trace() levels that hit (tests/oracle_aovs.cpp, the restatement with one more export, compiled here)."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, bits, load_golden, same_bits
from oracle import bindings as ob
from test_render_views import cameras

W, H = 320, 180
KEYS = ("depth", "tri", "normal", "hits")
STATS = ("primary", "primary_hit", "shadow", "bounce", "pipeline", "class_launches", "box_tests", "tri_tests")
FLT_MAX = np.float32(np.finfo(np.float32).max)
# two spheres in the Cornell box, one of them a mirror: [centre | radius] [kd | shininess] [ks | transparency]
SPHERES = np.array([[-0.2, -0.25, 0.1, 0.15, 0.8, 0.2, 0.2, 20.0, 0.5, 0.5, 0.5, 1.0],
                    [0.22, -0.3, -0.15, 0.12, 0.2, 0.3, 0.8, 10.0, 0.0, 0.0, 0.0, 1.0]], np.float32)


def intersect_aovs(capi, s, cam, W, H):
    """depth, tri, normal of cgrt_intersect_closest on cgrt_generate_rays(cam), flipped to Screen layout (row H-1-y)."""
    h = s.intersect(capi.generate_rays(cam, W, H)).reshape(H, W)[::-1]
    return dict(depth=h["t"], tri=h["tri"], normal=h["n"])


def oracle_camera(cam):
    return ob.CameraDesc.from_buffer_copy(cam)


@pytest.fixture(scope="session")
def aov_oracle(tmp_path_factory):
    """The restatement with its per-pixel buffers (tests/oracle_aovs.cpp includes oracle/cgrt_oracle.cpp), compiled with the
    oracle's flags (oracle/Makefile) into a temporary directory: a CPU checker with the orc_ surface plus orc_render_aovs."""
    so = str(tmp_path_factory.mktemp("oracle_aovs") / "liboracle_aovs.so")
    r = subprocess.run(["/usr/bin/g++", "-std=gnu++17", "-O2", "-fopenmp", "-ffp-contract=off", "-fPIC", "-fno-fast-math", "-shared",
                        "-o", so, os.path.join(ROOT, "tests", "oracle_aovs.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return ob._CpuChecker(so, "orc_")


def oracle_aovs(bvh, cam, W, H, L):
    """(rgb[H,W,3], {"depth", "tri" (canonical ids, -2 - s for sphere s), "normal", "hits"}) of the restatement, Screen layout;
    `bvh` is a BVH of the aov_oracle checker."""
    f = bvh.lib.lib.orc_render_aovs
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.POINTER(ob.CameraDesc), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                  C.c_void_p, C.c_int]
    rgb = np.zeros((H, W, 3), np.float32)
    aov = dict(depth=np.zeros((H, W), np.float32), tri=np.zeros((H, W), np.int32), normal=np.zeros((H, W, 3), np.float32),
               hits=np.zeros((H, W), np.uint8))
    assert f(bvh.h, C.byref(cam), W, H, L, rgb.ctypes.data, *[aov[k].ctypes.data for k in KEYS], 0) == 0
    return rgb, aov


def check_aovs(capi, s, cams, L, orc=None, canon=None, W=W, H=H):
    """render_aovs against render_views, the intersect oracle and (orc: the restatement's BVH, of aov_oracle) its per-pixel
    buffers."""
    rgb, aov, st = s.render_aovs(cams, W, H, trace_limit=L)
    want, sw = s.render_views(cams, W, H, trace_limit=L)
    assert same_bits(rgb, want), L
    assert [st[k] for k in STATS] == [sw[k] for k in STATS], (L, st, sw)
    assert set(aov) == set(KEYS)
    for v, cam in enumerate(cams):
        if L == 0:  # the frame traces nothing: every pixel is a miss
            assert not aov["hits"][v].any() and np.all(aov["tri"][v] == -1) and np.all(aov["depth"][v] == FLT_MAX)
            assert not bits(aov["normal"][v]).any()
        else:
            g = intersect_aovs(capi, s, cam, W, H)
            assert same_bits(aov["depth"][v], g["depth"]), (L, v)
            assert np.array_equal(aov["tri"][v], g["tri"]), (L, v)
            assert same_bits(aov["normal"][v], g["normal"]), (L, v)
            assert np.array_equal(aov["hits"][v] > 0, aov["tri"][v] != -1), (L, v)
        assert aov["hits"][v].max() <= L
        if orc is not None:
            _, o = oracle_aovs(orc, oracle_camera(cam), W, H, L)
            assert np.array_equal(aov["hits"][v], o["hits"]), (L, v)
            assert same_bits(aov["depth"][v], o["depth"]) and same_bits(aov["normal"][v], o["normal"]), (L, v)
            t = aov["tri"][v]
            assert np.array_equal(np.where(t >= 0, canon[np.maximum(t, 0)], t), o["tri"]), (L, v)
    return rgb, aov, st


# ---- argument validation (no GPU needed: refused before any CUDA call, valid ones fail on a host-only scene) ---------------
def _call(capi, s, cams, n, p, out, aov, device):
    lib = capi.load_library()
    arr = (capi.Camera * max(len(cams), 1))(*cams)
    ptr = C.c_void_p(out.ctypes.data) if out is not None else None
    a = C.byref(aov) if aov is not None else None
    if device:
        return lib.cgrt_render_aovs_device(s.h, arr if cams else None, n, C.byref(p), ptr, a, None)
    st = capi.RenderStats()
    return lib.cgrt_render_aovs(s.h, arr if cams else None, n, C.byref(p), ptr, a, C.byref(st))


@pytest.mark.parametrize("device", [False, True])
def test_aovs_refuse_bad_arguments(capi, device):
    s = capi.Scene(ob.random_soup(10, seed=1, scale=0.3), host_only=True)
    w, h = 16, 8
    cams = [capi.make_camera(w, h)] * 2
    out = np.zeros((2, h, w, 3), np.float32)
    depth = np.zeros((2, h, w), np.float32)
    aov = capi.AovBuffers(depth.ctypes.data, None, None, None)
    ok = capi.render_params(w, h)
    bad = [
        (cams, 0, ok, out, aov),                                   # no view
        (cams, 1025, ok, out, aov),                                # more than 1024
        ([], 2, ok, out, aov),                                     # null cams
        (cams, 2, ok, None, aov),                                  # null rgb
        (cams, 1024, capi.render_params(512, 513), out, aov),      # n_views x W x H > 2^28
        (cams, 1024, capi.render_params(1, 1 << 18), out, aov),    # 2^28 pixels, but 2^31 slots of whole 8 x 8 tiles
        (cams, 2, capi.render_params(w, h, world=2), out, aov),    # a share of a multi-GPU frame
        (cams, 2, capi.render_params(w, h, flags=capi.RENDER_COUNT), out, aov),
        (cams, 2, capi.render_params(w, h, flags=capi.RENDER_SCREEN_LAYOUT), out, aov),
        (cams, 2, ok, out, None),                                  # null aov
        (cams, 2, ok, out, capi.AovBuffers()),                     # no buffer requested
    ]
    for i, (c, n, p, o, a) in enumerate(bad):
        assert _call(capi, s, c, n, p, o, a, device) == capi.CGRT_ERR_INVALID, i
    # valid arguments reach the device check: a host-only scene has no device state
    for k in range(4):
        one = capi.AovBuffers(*[depth.ctypes.data if j == k else None for j in range(4)])
        assert _call(capi, s, cams, 2, ok, out, one, device) == capi.CGRT_ERR_NO_DEVICE, k
    assert _call(capi, s, cams, 2, capi.render_params(w, h, flags=capi.RENDER_PROFILE_ALL), out, aov, device) == capi.CGRT_ERR_NO_DEVICE


@pytest.mark.parametrize("name", ["cornell", "monkey"])
def test_oracle_aovs_are_its_intersect(oracle, aov_oracle, name):
    """The restatement's per-pixel buffers: its own frame (also that of oracle/liboracle.so), and its own intersect on its own
    primary rays, bit for bit."""
    g = load_golden(name)
    b = aov_oracle.scene(g.flat, g.lights).bvh()
    cam = ob.default_camera(g.W, g.H)
    c = g.flat.canonical_ids()
    for L in (1, 3):
        rgb, aov = oracle_aovs(b, cam, g.W, g.H, L)
        want, _ = oracle.scene(g.flat, g.lights).bvh().render(cam, g.W, g.H, trace_limit=L)
        assert same_bits(rgb, want)
        h = b.intersect(aov_oracle.generate_rays(cam, g.W, g.H)).reshape(g.H, g.W)[::-1]
        assert same_bits(aov["depth"], h["t"]) and same_bits(aov["normal"], h["n"])
        assert np.array_equal(aov["tri"], h["tri"]) and np.all(c[aov["tri"][aov["tri"] >= 0]] == aov["tri"][aov["tri"] >= 0])
        assert np.array_equal(aov["hits"] > 0, h["tri"] != -1) and aov["hits"].max() <= L
        assert (aov["hits"] > 0).any()


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def _scene(capi, name, checker=None):
    """(product scene, the restatement's BVH of the same scene (checker: aov_oracle; None: no BVH), canonical ids). Cornell's
    spheres reach the product's scene through set_spheres."""
    if name == "dragon":
        flat, lights = ob.dragon_standin_fixture()
    else:
        g = load_golden("cornell")
        flat, lights = g.flat, g.lights
    s = capi.Scene(flat, lights=lights)
    if name == "cornell_spheres":
        s.set_spheres(SPHERES)
        flat = ob.FlatScene(flat.vcount, flat.tcount, flat.vertices, flat.triangles, flat.materials, SPHERES)
    return s, checker.scene(flat, lights).bvh() if checker else None, flat.canonical_ids()


@pytest.fixture(scope="module", params=["cornell", "dragon", "cornell_spheres"])
def scene(request, capi, gpu, aov_oracle):
    s, orc, canon = _scene(capi, request.param, aov_oracle)
    yield request.param, s, orc, canon
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("L", [0, 1, 2, 5])
def test_aovs_equal_intersect_and_oracle(capi, scene, L):
    name, s, orc, canon = scene
    cams = cameras(capi, W, H)
    _, aov, _ = check_aovs(capi, s, cams, L, orc, canon)
    check_aovs(capi, s, cams[3:4], L, orc, canon)  # a batch of one
    if L > 0:
        assert (aov["hits"] > 0).any()
        if name == "cornell_spheres":
            assert (aov["tri"] <= -2).any()
        if L >= 2 and name != "dragon":
            assert (aov["hits"] >= 2).any()


@pytest.mark.gpu
def test_one_buffer_at_a_time(capi, gpu):
    """A buffer that is not requested is not written: the others keep their sentinel."""
    lib = capi.load_library()
    s, _, _ = _scene(capi, "cornell_spheres")
    cams = cameras(capi, W, H)[:2]
    _, full, _ = s.render_aovs(cams, W, H, trace_limit=3)
    K = len(cams)
    for k in KEYS:
        bufs = dict(depth=np.full((K, H, W), 7.5, np.float32), tri=np.full((K, H, W), 77, np.int32),
                    normal=np.full((K, H, W, 3), 7.5, np.float32), hits=np.full((K, H, W), 77, np.uint8))
        sentinel = {j: v.copy() for j, v in bufs.items()}
        a = capi.AovBuffers(*[bufs[j].ctypes.data if j == k else None for j in KEYS])
        rgb = np.zeros((K, H, W, 3), np.float32)
        arr = (capi.Camera * K)(*cams)
        st = capi.RenderStats()
        capi.check(lib.cgrt_render_aovs(s.h, arr, K, C.byref(capi.render_params(W, H, 3)), C.c_void_p(rgb.ctypes.data),
                                        C.byref(a), C.byref(st)))
        for j in KEYS:
            want = full[j] if j == k else sentinel[j]
            assert np.array_equal(bits(bufs[j]) if bufs[j].dtype == np.float32 else bufs[j],
                                  bits(want) if want.dtype == np.float32 else want), (k, j)
        _, one, _ = s.render_aovs(cams, W, H, trace_limit=3, **{j: j == k for j in KEYS})
        assert set(one) == {k}
    s.close()


@pytest.mark.gpu
def test_aovs_with_spherical_lights(capi, gpu):
    g = load_golden("cornell")
    s = capi.Scene(g.flat, lights=g.lights)
    s.set_spherical_lights(np.array([[0, 0.45, 0, 0.1, 1, 1, 1]], np.float32), seed=7)
    _, _, st = check_aovs(capi, s, cameras(capi, W, H), 2)
    assert st["pipeline"] == 2
    s.close()


@pytest.mark.gpu
def test_aovs_device_form(capi, gpu):
    import torch
    s, _, _ = _scene(capi, "dragon")
    cams = cameras(capi, W, H)
    L = 5
    want, wa, sw = s.render_aovs(cams, W, H, trace_limit=L)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        d_rgb = torch.zeros(want.shape, dtype=torch.float32, device="cuda")
        d = dict(depth=torch.zeros(wa["depth"].shape, dtype=torch.float32, device="cuda"),
                 tri=torch.zeros(wa["tri"].shape, dtype=torch.int32, device="cuda"),
                 normal=torch.zeros(wa["normal"].shape, dtype=torch.float32, device="cuda"),
                 hits=torch.zeros(wa["hits"].shape, dtype=torch.uint8, device="cuda"))
    s.render_aovs_device(cams, capi.render_params(W, H, L), d_rgb.data_ptr(), {k: v.data_ptr() for k, v in d.items()},
                         stream.cuda_stream)
    st = s.collect_stats()
    stream.synchronize()
    assert same_bits(d_rgb.cpu().numpy(), want)
    for k in KEYS:
        got = d[k].cpu().numpy()
        assert np.array_equal(bits(got) if got.dtype == np.float32 else got, bits(wa[k]) if got.dtype == np.float32 else wa[k]), k
    keys = ("primary", "primary_hit", "shadow", "bounce", "pipeline", "kernel_launches")
    assert [st[k] for k in keys] == [sw[k] for k in keys]
    s.close()


@pytest.mark.gpu
def test_aovs_leave_no_state_behind(capi, gpu):
    """render, render_views and render_aovs of other sizes and shapes interleaved on one scene: each result equals what a
    second scene renders."""
    s, _, _ = _scene(capi, "dragon")
    ref, _, _ = _scene(capi, "dragon")
    cams = cameras(capi, W, H)
    L = 3
    for step in range(2):
        one, _ = s.render(cams[3], W, H, trace_limit=L)
        assert same_bits(one, ref.render(cams[3], W, H, trace_limit=L)[0]), step
        for cs in (cams[:3], cams):
            a = s.render_aovs(cs, W, H, trace_limit=L)
            b = ref.render_aovs(cs, W, H, trace_limit=L)
            assert same_bits(a[0], b[0]) and all(np.array_equal(bits(a[1][k]) if a[1][k].dtype == np.float32 else a[1][k],
                                                                bits(b[1][k]) if b[1][k].dtype == np.float32 else b[1][k])
                                                 for k in KEYS), step
        views, _ = s.render_views(cams, W, H, trace_limit=L)
        assert same_bits(views, ref.render_views(cams, W, H, trace_limit=L)[0]), step
        w2, h2 = 200, 150
        c2 = [capi.make_camera(w2, h2, euler_deg=(20.0, 20.0 + 30 * k, 0.0)) for k in range(4)]
        a = s.render_aovs(c2, w2, h2, trace_limit=L + 2)
        b = ref.render_aovs(c2, w2, h2, trace_limit=L + 2)
        assert same_bits(a[0], b[0]) and all(np.array_equal(a[1][k].view(np.uint8), b[1][k].view(np.uint8)) for k in KEYS), step
    s.close()
    ref.close()


@pytest.mark.gpu
def test_aovs_at_benchmark_size(capi, gpu):
    """C3 (dragon stand-in, 1920 x 1080, trace limit 5): one view and 8 views against the intersect oracle."""
    flat, lights = ob.dragon_standin_fixture()
    s = capi.Scene(flat, lights=lights)
    w, h = 1920, 1080
    cams = [capi.make_camera(w, h)] + [capi.make_camera(w, h, look_at=(0.02 * k, 0.0, 0.0)) for k in range(1, 5)] + \
           [capi.make_camera(w, h, euler_deg=(20.0, 20.0 + 15 * k, 0.0)) for k in range(1, 4)]
    _, _, st = check_aovs(capi, s, cams[:1], 5, W=w, H=h)
    assert st["pipeline"] == 3
    check_aovs(capi, s, cams, 5, W=w, H=h)
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
    rgb, aov, st = s.render_aovs(cams, W, H, trace_limit=L)
    want, sw = s.render_views(cams, W, H, trace_limit=L)
    same = bool(np.array_equal(rgb.view(np.uint32), want.view(np.uint32)))
    sha = hashlib.sha1(b"".join(np.ascontiguousarray(aov[k]).tobytes() for k in ("depth", "tri", "normal", "hits"))).hexdigest()
    out[L] = dict(same=same, sha=sha, pipeline=st["pipeline"], views_pipeline=sw["pipeline"],
                  launches=st["kernel_launches"] - sw["kernel_launches"])
print("RESULT " + json.dumps(out))
"""


@pytest.mark.gpu
def test_aovs_on_every_pipeline(gpu):
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
            # the AOV pass: one kernel, two for the path pipeline's records (fill every pixel as a miss, then scatter the paths)
            assert v["launches"] == (2 if pipeline == 1 and L != "0" else 1), (name, L, v)
    for name in ("rounds", "paths"):
        for L in res["wave"]:
            assert res[name][L]["sha"] == res["wave"][L]["sha"], (name, L)
