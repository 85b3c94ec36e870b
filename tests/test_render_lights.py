"""cgrt_render_lights: each light group's share of the frame in its own buffer. rgb and the statistics equal cgrt_render_views;
group g is bit for bit the frame with every light outside g black; a group of every light is rgb; the groups of a partition
sum to rgb up to float reassociation; at trace limit 0 every buffer is +0."""
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
STATS = ("primary", "primary_hit", "shadow", "bounce", "pipeline", "class_launches", "box_tests", "tri_tests")
# two spheres in the Cornell box, one of them a mirror (as tests/test_render_aovs.py)
SPHERES = np.array([[-0.2, -0.25, 0.1, 0.15, 0.8, 0.2, 0.2, 20.0, 0.5, 0.5, 0.5, 1.0],
                    [0.22, -0.3, -0.15, 0.12, 0.2, 0.3, 0.8, 10.0, 0.0, 0.0, 0.0, 1.0]], np.float32)
# four point lights of other colours in the Cornell box: groups {0}, {1, 2}, and the last light in no group
CORNELL_LIGHTS = np.array([[0.0, 0.58, 0.0, 1.0, 1.0, 1.0], [-0.4, 0.5, 0.3, 0.8, 0.3, 0.2],
                           [0.35, 0.2, 0.6, 0.2, 0.5, 0.9], [0.1, 0.4, -0.3, 0.6, 0.6, 0.3]], np.float32)
CORNELL_GROUPS = [0, 1, 1, -1]
SPH_LIGHTS = np.array([[0.2, 0.45, 0.1, 0.1, 0.9, 0.8, 0.6], [-0.3, 0.4, 0.2, 0.1, 0.3, 0.4, 1.0]], np.float32)
# largest |sum of a partition's groups - rgb| over max(1, |rgb|) accepted (float reassociation of a few terms per level)
PARTITION_RTOL = 1e-5


def scene_of(capi, name, exact_only=False):
    """(scene, point lights, its groups); every scene but the monkey has more lights than its fixture."""
    if name == "monkey":
        g = load_golden("monkey")
        return capi.Scene(g.flat, lights=g.lights, exact_only=exact_only), g.lights, [0, 1]
    if name == "dragon":
        flat, lights = ob.dragon_standin_fixture()
        lights = np.concatenate([lights, [[1.0, 1.5, 0.5, 0.6, 0.8, 1.0]]]).astype(np.float32)
        return capi.Scene(flat, lights=lights, exact_only=exact_only), lights, [0, 1]
    g = load_golden("cornell")
    s = capi.Scene(g.flat, lights=CORNELL_LIGHTS, exact_only=exact_only)
    if name == "cornell_spheres":
        s.set_spheres(SPHERES)
    return s, CORNELL_LIGHTS, CORNELL_GROUPS


def zeroed(lights, keep, width):
    """`lights` ([n][width], colour in the last three columns) with the colour of every light not in `keep` set to 0."""
    z = np.array(lights, np.float32).copy()
    for i in range(len(z)):
        if i not in keep:
            z[i, width - 3:] = 0.0
    return z


def check_groups(s, cams, L, lights, groups, sph=None, seed=7, W=W, H=H):
    """render_lights against render_views, and each group against render_views with the other lights black (contract 1).
    Restores the scene's lights. Returns (rgb, light_rgb)."""
    rgb, light_rgb, st = s.render_lights(cams, W, H, trace_limit=L, groups=groups)
    want, sw = s.render_views(cams, W, H, trace_limit=L)
    assert same_bits(rgb, want), L
    assert [st[k] for k in STATS] == [sw[k] for k in STATS], (L, st, sw)
    nP = len(lights)
    for g in range(light_rgb.shape[0]):
        members = {i for i, x in enumerate(groups) if x == g}
        s.set_lights(zeroed(lights, members, 6))
        if sph is not None:
            s.set_spherical_lights(zeroed(sph, {i - nP for i in members}, 7), seed=seed)
        black, _ = s.render_views(cams, W, H, trace_limit=L)
        assert same_bits(light_rgb[g], black), (L, g, float(np.abs(light_rgb[g] - black).max()))
        if L == 0:
            assert not bits(light_rgb[g]).any()
    s.set_lights(lights)
    if sph is not None:
        s.set_spherical_lights(sph, seed=seed)
    return rgb, light_rgb


# ---- argument validation (no GPU needed: refused before any CUDA call, valid ones fail on a host-only scene) ---------------
def _call(capi, s, cams, n, p, out, lg, n_lights, n_groups, groups, device):
    lib = capi.load_library()
    arr = (capi.Camera * max(len(cams), 1))(*cams)
    ptr = C.c_void_p(out.ctypes.data) if out is not None else None
    gptr = C.c_void_p(groups.ctypes.data) if groups is not None else None
    lgp = np.ascontiguousarray(lg, np.int32).ctypes.data_as(C.POINTER(C.c_int32)) if lg is not None else None
    if device:
        return lib.cgrt_render_lights_device(s.h, arr if cams else None, n, C.byref(p), lgp, n_lights, n_groups, ptr, gptr, None)
    st = capi.RenderStats()
    return lib.cgrt_render_lights(s.h, arr if cams else None, n, C.byref(p), lgp, n_lights, n_groups, ptr, gptr, C.byref(st))


@pytest.mark.parametrize("device", [False, True])
def test_lights_refuse_bad_arguments(capi, device):
    s = capi.Scene(ob.random_soup(10, seed=1, scale=0.3), host_only=True, lights=CORNELL_LIGHTS[:3])
    s.set_spherical_lights(SPH_LIGHTS, seed=7)
    w, h = 16, 8
    cams = [capi.make_camera(w, h)] * 2
    out = np.zeros((2, h, w, 3), np.float32)
    grp = np.zeros((2, 2, h, w, 3), np.float32)
    lg = [0, 1, -1, 1, 0]  # three point lights, two spherical lights
    ok = capi.render_params(w, h)
    bad = [
        (cams, 0, ok, out, lg, 5, 2, grp),                                     # no view
        (cams, 1025, ok, out, lg, 5, 2, grp),                                  # more than 1024
        ([], 2, ok, out, lg, 5, 2, grp),                                       # null cams
        (cams, 2, ok, None, lg, 5, 2, grp),                                    # null rgb
        (cams, 1024, capi.render_params(512, 513), out, lg, 5, 1, grp),        # n_views x W x H > 2^28
        (cams, 1024, capi.render_params(1, 1 << 18), out, lg, 5, 1, grp),      # 2^31 slots of whole 8 x 8 tiles
        (cams, 2, capi.render_params(w, h, world=2), out, lg, 5, 2, grp),      # a share of a multi-GPU frame
        (cams, 2, capi.render_params(w, h, flags=capi.RENDER_COUNT), out, lg, 5, 2, grp),
        (cams, 2, capi.render_params(w, h, flags=capi.RENDER_SCREEN_LAYOUT), out, lg, 5, 2, grp),
        (cams, 2, ok, out, None, 5, 2, grp),                                   # null light_group
        (cams, 2, ok, out, lg, 5, 2, None),                                    # null groups
        (cams, 2, ok, out, [0] * 5, 5, 0, grp),                                # n_groups < 1
        (cams, 2, ok, out, [0] * 5, 5, 65, grp),                               # n_groups > 64
        (cams, 64, capi.render_params(2048, 1024), out, [0] * 5, 5, 3, grp),   # 3 x 64 x 2^21 > 2^28 group pixels
        (cams, 2, ok, out, lg[:4], 4, 2, grp),                                 # n_lights below the scene's
        (cams, 2, ok, out, lg + [0], 6, 2, grp),                               # n_lights above the scene's
        (cams, 2, ok, out, [0, 1, -2, 1, 0], 5, 2, grp),                       # entry below -1
        (cams, 2, ok, out, [0, 1, -1, 2, 0], 5, 2, grp),                       # entry n_groups
    ]
    for i, (c, n, p, o, l, nl, ng, g) in enumerate(bad):
        assert _call(capi, s, c, n, p, o, l, nl, ng, g, device) == capi.CGRT_ERR_INVALID, i
    # valid arguments reach the device check: a host-only scene has no device state
    for l, ng in ((lg, 2), ([-1] * 5, 1), ([0, 1, 2, 3, 4], 5), ([0] * 5, 64)):
        assert _call(capi, s, cams, 2, ok, out, l, 5, ng, grp, device) == capi.CGRT_ERR_NO_DEVICE, (l, ng)
    assert _call(capi, s, cams, 2, capi.render_params(w, h, flags=capi.RENDER_PROFILE_ALL), out, lg, 5, 2, grp,
                 device) == capi.CGRT_ERR_NO_DEVICE
    # the light count follows set_lights
    s.set_lights(CORNELL_LIGHTS)
    assert _call(capi, s, cams, 2, ok, out, lg, 5, 2, grp, device) == capi.CGRT_ERR_INVALID
    assert _call(capi, s, cams, 2, ok, out, lg + [0], 6, 2, grp, device) == capi.CGRT_ERR_NO_DEVICE
    s.close()


def test_relight_is_the_gained_sum(capi):
    rng = np.random.default_rng(3)
    light_rgb = rng.random((3, 2, 4, 5, 3), dtype=np.float32)
    gains = rng.random((3, 3), dtype=np.float32)
    want = sum(light_rgb[g] * gains[g] for g in range(3))
    assert np.allclose(capi.relight(light_rgb, gains), want, rtol=1e-6)
    assert np.array_equal(capi.relight(light_rgb, np.ones((3, 3))), light_rgb[0] + light_rgb[1] + light_rgb[2])


# ---- GPU ----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", params=["cornell", "monkey", "dragon", "cornell_spheres"])
def scene(request, capi, gpu):
    s, lights, groups = scene_of(capi, request.param)
    yield request.param, s, lights, groups
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("L", [0, 1, 2, 5])
def test_groups_are_renders_with_the_other_lights_black(capi, scene, L):
    """Contracts 1 and 2, six views and a batch of one."""
    name, s, lights, groups = scene
    cams = cameras(capi, W, H)
    for cs in (cams, cams[3:4]):
        rgb, light_rgb = check_groups(s, cs, L, lights, groups)
        if L > 0:
            assert all(bits(light_rgb[g]).any() for g in range(light_rgb.shape[0])), name
        _, every, _ = s.render_lights(cs, W, H, trace_limit=L, groups=[0] * len(lights))
        assert every.shape[0] == 1 and same_bits(every[0], rgb), L


@pytest.mark.gpu
@pytest.mark.parametrize("L", [1, 2, 5])
def test_partition_sums_to_the_frame(capi, scene, L):
    """Contract 3: one group per light; the sum matches rgb up to float reassociation. An empty group is +0."""
    name, s, lights, _ = scene
    n = len(lights)
    rgb, light_rgb, _ = s.render_lights(cameras(capi, W, H), W, H, trace_limit=L, n_groups=n + 1)
    assert not bits(light_rgb[n]).any()
    total = light_rgb.sum(axis=0, dtype=np.float32)
    err = float((np.abs(total - rgb) / np.maximum(1.0, np.abs(rgb))).max())
    print(f"{name} L={L}: largest |sum of groups - rgb| / max(1, |rgb|) = {err:.3g}")
    assert err <= PARTITION_RTOL, err


@pytest.mark.gpu
@pytest.mark.parametrize("L", [0, 2, 5])
def test_spherical_light_groups(capi, gpu, L):
    """Two spherical lights (radius 0.1, seed 7) and one point light, each in its own group: the round pipeline's soft-shadow
    fractions keyed by each light's unchanged index."""
    g = load_golden("cornell")
    s = capi.Scene(g.flat, lights=g.lights)
    s.set_spherical_lights(SPH_LIGHTS, seed=7)
    cams = cameras(capi, W, H)
    rgb, light_rgb = check_groups(s, cams, L, g.lights, [0, 1, 2], sph=SPH_LIGHTS)
    _, every, st = s.render_lights(cams, W, H, trace_limit=L, groups=[0, 0, 0])
    assert same_bits(every[0], rgb)
    if L > 0:
        assert st["pipeline"] == 2 and all(bits(light_rgb[k]).any() for k in range(3))
    s.close()


@pytest.mark.gpu
def test_groups_match_the_restatement(capi, oracle, gpu):
    """Each group of a small Cornell frame against the CPU restatement with the other lights black (within 1/255)."""
    g = load_golden("cornell")
    w, h = g.W, g.H
    s = capi.Scene(g.flat, lights=CORNELL_LIGHTS)
    cam = ob.default_camera(w, h)
    for L in (1, 3):
        _, light_rgb, _ = s.render_lights([capi.make_camera(w, h)], w, h, trace_limit=L, groups=CORNELL_GROUPS)
        for grp in range(2):
            keep = {i for i, x in enumerate(CORNELL_GROUPS) if x == grp}
            want, _ = oracle.scene(g.flat, zeroed(CORNELL_LIGHTS, keep, 6)).bvh().render(cam, w, h, trace_limit=L)
            d = float(np.abs(light_rgb[grp, 0] - want).max())
            assert d <= 1.0 / 255.0, (L, grp, d)
    s.close()


@pytest.mark.gpu
def test_relight_matches_a_render_with_scaled_colours(capi, gpu):
    """relight() of one group per light against a render whose light colours are scaled by the gains."""
    s, lights, _ = scene_of(capi, "cornell_spheres")
    cams = cameras(capi, W, H)[:3]
    gains = np.array([[0.5, 1.0, 2.0], [1.5, 0.25, 0.75], [0.0, 1.0, 1.0], [1.0, 1.0, 1.0]], np.float32)
    _, light_rgb, _ = s.render_lights(cams, W, H, trace_limit=3)
    relit = capi.relight(light_rgb, gains)
    scaled = lights.copy()
    scaled[:, 3:] *= gains
    s.set_lights(scaled)
    want, _ = s.render_views(cams, W, H, trace_limit=3)
    err = float((np.abs(relit - want) / np.maximum(1.0, np.abs(want))).max())
    print(f"relight: largest |relit - render| / max(1, |render|) = {err:.3g}")
    assert err <= PARTITION_RTOL, err
    s.close()


@pytest.mark.gpu
def test_lights_device_form(capi, gpu):
    import torch
    s, lights, groups = scene_of(capi, "dragon")
    cams = cameras(capi, W, H)
    L = 5
    want, wg, sw = s.render_lights(cams, W, H, trace_limit=L, groups=groups)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        d_rgb = torch.full(want.shape, float("nan"), dtype=torch.float32, device="cuda")
        d_grp = torch.full(wg.shape, float("nan"), dtype=torch.float32, device="cuda")
    s.render_lights_device(cams, capi.render_params(W, H, L), groups, wg.shape[0], d_rgb.data_ptr(), d_grp.data_ptr(),
                           stream.cuda_stream)
    st = s.collect_stats()
    stream.synchronize()
    assert same_bits(d_rgb.cpu().numpy(), want) and same_bits(d_grp.cpu().numpy(), wg)
    keys = ("primary", "primary_hit", "shadow", "bounce", "pipeline", "kernel_launches")
    assert [st[k] for k in keys] == [sw[k] for k in keys]
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("exact_only", [False, True])
def test_lights_leave_no_state_behind(capi, gpu, exact_only):
    """render_views / render_aovs / render_lights of other shapes interleaved on one scene equal what a second scene renders;
    the device form writes +0 into every missed pixel of a buffer full of another frame's colours (exact_only: the path
    pipeline, whose misses have no record)."""
    import torch
    s, lights, groups = scene_of(capi, "cornell_spheres", exact_only)
    ref, _, _ = scene_of(capi, "cornell_spheres", exact_only)
    cams = cameras(capi, W, H)
    near = [capi.make_camera(W, H, dist=1.2)] * 2   # the box fills the frame
    far = [capi.make_camera(W, H, dist=9.0)] * 2    # the box is small: most pixels miss
    for step in range(2):
        for cs, w, h, L in ((cams[:3], W, H, 3), (cameras(capi, 200, 150), 200, 150, 5), (near, W, H, 2), (far, W, H, 2)):
            a = s.render_lights(cs, w, h, trace_limit=L, groups=groups)
            b = ref.render_lights(cs, w, h, trace_limit=L, groups=groups)
            assert same_bits(a[0], b[0]) and same_bits(a[1], b[1]), (step, w, L)
            assert same_bits(s.render_views(cs, w, h, trace_limit=L)[0], ref.render_views(cs, w, h, trace_limit=L)[0])
            assert same_bits(s.render_aovs(cs, w, h, trace_limit=L)[0], b[0])
    _, hit_near, _ = s.render_lights(near, W, H, trace_limit=2, groups=groups)
    _, miss_far, _ = s.render_lights(far, W, H, trace_limit=2, groups=groups)
    d_grp = torch.from_numpy(hit_near).cuda()
    d_rgb = torch.zeros((2, H, W, 3), dtype=torch.float32, device="cuda")
    s.render_lights_device(far, capi.render_params(W, H, 2), groups, hit_near.shape[0], d_rgb.data_ptr(), d_grp.data_ptr())
    torch.cuda.synchronize()
    got = d_grp.cpu().numpy()
    missed = ~s.render_aovs(far, W, H, trace_limit=2, depth=False, tri=False, normal=False)[1]["hits"].astype(bool)
    assert (bits(hit_near)[:, missed].any()) and not bits(got)[:, missed].any()
    assert same_bits(got, miss_far)
    s.close()
    ref.close()


@pytest.mark.gpu
def test_lights_at_benchmark_size(capi, gpu):
    """C3 (dragon stand-in, 1920 x 1080, trace limit 5) with one group of every light: one view and 8 views."""
    flat, lights = ob.dragon_standin_fixture()
    s = capi.Scene(flat, lights=lights)
    w, h = 1920, 1080
    cams = [capi.make_camera(w, h)] + [capi.make_camera(w, h, look_at=(0.02 * k, 0.0, 0.0)) for k in range(1, 5)] + \
           [capi.make_camera(w, h, euler_deg=(20.0, 20.0 + 15 * k, 0.0)) for k in range(1, 4)]
    for cs in (cams[:1], cams):
        rgb, light_rgb, st = s.render_lights(cs, w, h, trace_limit=5, groups=[0])
        want, sw = s.render_views(cs, w, h, trace_limit=5)
        assert same_bits(rgb, want) and same_bits(light_rgb[0], rgb)
        assert [st[k] for k in STATS] == [sw[k] for k in STATS]
    assert st["pipeline"] in (2, 3)
    s.close()


# ---- every pipeline, each forced in its own process -----------------------------------------------------------------------
_WORKER = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[1] + "/tests")
import __graft_entry__ as ge
from test_render_lights import scene_of, zeroed
from test_render_views import cameras
capi = ge.load_package().capi
s, lights, groups = scene_of(capi, "cornell_spheres", exact_only=sys.argv[2] == "1")
W, H = 320, 180
cams = cameras(capi, W, H)
out = {}
for L in (3, 0, 1):
    rgb, light_rgb, st = s.render_lights(cams, W, H, trace_limit=L, groups=groups)
    want, sw = s.render_views(cams, W, H, trace_limit=L)
    same = [bool(np.array_equal(rgb.view(np.uint32), want.view(np.uint32)))]
    for g in range(light_rgb.shape[0]):
        s.set_lights(zeroed(lights, {i for i, x in enumerate(groups) if x == g}, 6))
        same.append(bool(np.array_equal(light_rgb[g].view(np.uint32), s.render_views(cams, W, H, trace_limit=L)[0].view(np.uint32))))
        s.set_lights(lights)
    every = s.render_lights(cams, W, H, trace_limit=L, groups=[0] * len(lights))[1]
    same.append(bool(np.array_equal(every[0].view(np.uint32), rgb.view(np.uint32))))
    out[L] = dict(same=same, pipeline=st["pipeline"], views_pipeline=sw["pipeline"], launches=st["kernel_launches"] - sw["kernel_launches"])
print("RESULT " + json.dumps(out))
"""


@pytest.mark.gpu
def test_lights_on_every_pipeline(gpu):
    for name, pref, exact, pipeline in (("wave", "wave", False, 3), ("rounds", "rounds", False, 2), ("paths", None, True, 1)):
        env = dict(os.environ)
        env.pop("CGRT_PIPELINE", None)
        if pref:
            env["CGRT_PIPELINE"] = pref
        r = subprocess.run([sys.executable, "-c", _WORKER, ROOT, "1" if exact else "0"], env=env, capture_output=True, text=True,
                           timeout=600)
        line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
        assert r.returncode == 0 and line, (name, r.stdout[-800:], r.stderr[-2000:])
        for L, v in json.loads(line[0][7:]).items():
            assert v["pipeline"] == pipeline and v["views_pipeline"] == pipeline and all(v["same"]), (name, L, v)
            # the group pass: one kernel; at trace limit 0 only a clear of the buffers
            assert v["launches"] == (0 if L == "0" else 1), (name, L, v)
