"""cgrt_render_effects_views: anti-aliasing, motion blur and bloom for several cameras in one call, on the caller's stream. View v
must be bit for bit what cgrt_render_effects returns for camera v, with the call's ray statistics the sums of those calls'."""
import ctypes as C

import numpy as np
import pytest

from conftest import load_golden, same_bits
from oracle import bindings as ob
from test_render_views import RAYS, cameras

W, H = 320, 180
AA, BLUR, BLOOM = 1, 2, 4
EFFECTS = {"aa": AA, "blur": BLUR, "bloom": BLOOM, "bloom+blur": BLOOM | BLUR, "blur+aa": BLUR | AA}


def flags(effects):
    return dict(antialias=bool(effects & AA), motion_blur=bool(effects & BLUR), bloom=bool(effects & BLOOM))


def check_effects_views(s, cams, w, h, L, effects, ref=None, want=None):
    """The batch of `cams` against one cgrt_render_effects per camera on `ref` (default: the same scene); `want` = precomputed
    (frames, summed ray counts). Returns the batch's frames and stats."""
    got, st = s.render_effects_views(cams, w, h, trace_limit=L, **flags(effects))
    assert got.shape == (len(cams), h, w, 3)
    if want is None:
        want = single_calls(ref or s, cams, w, h, L, effects)
    frames, total = want
    for v in range(len(cams)):
        assert same_bits(got[v], frames[v]), (v, L, effects, float(np.nanmax(np.abs(got[v] - frames[v]))))
    assert {k: st[k] for k in RAYS} == total, (L, effects, st, total)
    return got, st


def single_calls(s, cams, w, h, L, effects):
    frames, total = [], dict.fromkeys(RAYS, 0)
    for cam in cams:
        f, sv = s.render_effects(cam, w, h, trace_limit=L, **flags(effects))
        frames.append(f)
        for k in RAYS:
            total[k] += sv[k]
    return frames, total


# ---- argument validation (no GPU needed: refused before any CUDA call, valid ones fail on a host-only scene) ---------------
def _call(capi, s, cams, n, p, effects, out, device):
    lib = capi.load_library()
    arr = (capi.Camera * max(len(cams), 1))(*cams)
    ptr = C.c_void_p(out.ctypes.data) if out is not None else None
    if device:
        return lib.cgrt_render_effects_views_device(s.h, arr if cams else None, n, C.byref(p), effects, ptr, None)
    st = capi.RenderStats()
    return lib.cgrt_render_effects_views(s.h, arr if cams else None, n, C.byref(p), effects, ptr, C.byref(st))


@pytest.mark.parametrize("device", [False, True])
def test_effects_views_refuse_bad_arguments(capi, device):
    s = capi.Scene(ob.random_soup(10, seed=1, scale=0.3), host_only=True)
    w, h = 16, 8
    cams = [capi.make_camera(w, h)] * 2
    out = np.zeros((2, h, w, 3), np.float32)
    ok = capi.render_params(w, h)
    bad = [
        (cams, 0, ok, BLUR, out),                                    # no view
        (cams, 1025, ok, BLUR, out),                                 # more than 1024
        ([], 2, ok, BLUR, out),                                      # null cams
        (cams, 2, ok, BLUR, None),                                   # null output
        (cams, 2, capi.render_params(0, h), BLUR, out),              # no pixels
        (cams, 1024, capi.render_params(512, 513), BLUR, out),       # n_views x W x H > 2^28
        (cams, 2, capi.render_params(w, h, world=2), BLUR, out),     # a share of a multi-GPU frame
        (cams, 2, capi.render_params(w, h, flags=capi.RENDER_PROFILE_ALL), BLUR, out),  # no profiling mode
        (cams, 2, capi.render_params(w, h, flags=capi.RENDER_COUNT), BLUR, out),
        (cams, 2, capi.render_params(w, h, flags=capi.RENDER_SCREEN_LAYOUT), BLUR, out),
        (cams, 2, capi.render_params(w, h, flags=capi.RENDER_PROFILE_ALL), 0, out),     # also without effects
        (cams, 2, ok, 8, out),                                       # unknown effect bit
        (cams, 2, ok, BLOOM | AA, out),                              # bloom with anti-aliasing
        (cams, 2, ok, BLOOM | AA | BLUR, out),
        (cams, 1, capi.render_params(16384, 8193), AA, out),         # 4 x W x H > 2^28 for anti-aliasing
    ]
    for i, (c, n, p, e, o) in enumerate(bad):
        assert _call(capi, s, c, n, p, e, o, device) == capi.CGRT_ERR_INVALID, i
    # valid arguments reach the device check: a host-only scene has no device state
    for e in (0, AA, BLUR, BLOOM, BLOOM | BLUR, BLUR | AA):
        assert _call(capi, s, cams, 2, ok, e, out, device) == capi.CGRT_ERR_NO_DEVICE, e
    # motion blur wins over anti-aliasing, so the supersampling limit does not apply to it
    assert _call(capi, s, cams, 1, capi.render_params(16384, 8193), BLUR | AA, out, device) == capi.CGRT_ERR_NO_DEVICE
    big = [capi.make_camera(512, 512)] * 1024
    assert _call(capi, s, big, 1024, capi.render_params(512, 512), BLUR, out, device) == capi.CGRT_ERR_NO_DEVICE


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def bright(lights):
    """test_bloom_against_sequential_restatement's light colour: enough pixels over the bloom threshold r + g + b > 1."""
    b = np.array(lights, np.float32).copy()
    b[:, 3:6] = 2.5
    return b


@pytest.fixture(scope="module")
def dragon(capi, gpu):
    flat, lights = ob.dragon_standin_fixture()
    return capi.Scene(flat, lights=bright(lights))


@pytest.fixture(scope="module")
def cornell(capi, gpu):
    g = load_golden("cornell")
    return capi.Scene(g.flat, lights=bright(g.lights))


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["cornell", "dragon"])
@pytest.mark.parametrize("effects", list(EFFECTS))
@pytest.mark.parametrize("L", [0, 1, 2, 5])
def test_effects_views_equal_single_calls(capi, request, scene, effects, L):
    s = request.getfixturevalue(scene)
    e = EFFECTS[effects]
    cams = cameras(capi, W, H)
    frames, _ = want = single_calls(s, cams, W, H, L, e)
    if e & BLOOM and L > 0:
        assert (s.render(cams[0], W, H, trace_limit=L)[0].sum(axis=2) > 1).sum() > 20, "bloom needs pixels over the threshold"
    for K in (1, 3, 6):
        per = [single_calls(s, [c], W, H, L, e)[1] for c in cams[:K]] if K < len(cams) else None
        total = {k: sum(p[k] for p in per) for k in RAYS} if per else want[1]
        check_effects_views(s, cams[:K], W, H, L, e, want=(frames[:K], total))


@pytest.mark.gpu
def test_bloom_views_against_oracle(capi, oracle, dragon):
    """Bloom of 4 views in one pass is oracle.bloom of each view's frame, bit for bit: sizes wider and narrower than the 21 x 21
    window, non-multiples of the progress granularity, and more rows than one wave of warps."""
    for (w, h, L) in ((200, 150, 3), (37, 29, 2), (13, 450, 1)):
        cams = cameras(capi, w, h)[:4]
        got, _ = dragon.render_effects_views(cams, w, h, trace_limit=L, bloom=True)
        for v, cam in enumerate(cams):
            frame, _ = dragon.render(cam, w, h, trace_limit=L)
            assert same_bits(got[v], oracle.bloom(frame)), (w, h, v)


@pytest.mark.gpu
def test_blur_split_over_batches(capi, cornell):
    """2048 x 1152: 15 x 2.36 M pixel slots > 2^25, so each view's cameras span two renders."""
    w, h = 2048, 1152
    cams = [capi.make_camera(w, h), capi.make_camera(w, h, euler_deg=(-15.0, 40.0, 5.0))]
    check_effects_views(cornell, cams, w, h, 1, BLUR)
    check_effects_views(cornell, cams[:1], w, h, 2, BLOOM | BLUR)


@pytest.mark.gpu
def test_antialiasing_split_over_batches(capi, cornell):
    """1920 x 1600: 12.3 M slots at 2W x 2H, two views per render, so five views take three renders, the last one view."""
    w, h = 1920, 1600
    cams = cameras(capi, w, h)[:5]
    check_effects_views(cornell, cams, w, h, 1, AA)


@pytest.mark.gpu
def test_effects_views_with_spherical_lights(capi, gpu):
    g = load_golden("cornell")
    s = capi.Scene(g.flat, lights=g.lights)
    s.set_spherical_lights(np.array([[0, 0.45, 0, 0.1, 1, 1, 1]], np.float32), seed=7)
    w, h = 160, 120
    cams = cameras(capi, w, h)[:3]
    check_effects_views(s, cams, w, h, 2, BLUR)
    check_effects_views(s, cams, w, h, 2, BLOOM | BLUR)


def _device_call(capi, s, cams, params, effects, shape, stream):
    import torch
    out = torch.full(shape, float("nan"), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    s.render_effects_views_device(cams, params, effects, out.data_ptr(), stream.cuda_stream)
    st = s.collect_stats()
    stream.synchronize()
    return out.cpu().numpy(), st


@pytest.mark.gpu
def test_effects_views_device_form(capi, dragon):
    import torch
    cams = cameras(capi, W, H)[:3]
    stream = torch.cuda.Stream()
    for e in (BLUR, BLOOM | BLUR, AA, BLOOM):
        want, sw = dragon.render_effects_views(cams, W, H, trace_limit=5, **flags(e))
        got, st = _device_call(capi, dragon, cams, capi.render_params(W, H, 5), e, want.shape, stream)
        assert same_bits(got, want), e
        assert [st[k] for k in RAYS + ("kernel_launches",)] == [sw[k] for k in RAYS + ("kernel_launches",)], (e, st, sw)
        assert st["device_ms"] > 0


@pytest.mark.gpu
def test_effects_views_leave_no_state_behind(capi, gpu):
    """Effects-views calls interleaved with single frames, views batches and cgrt_render_effects on one scene, then another
    shape: every result equals what a second scene renders call by call."""
    flat, lights = ob.dragon_standin_fixture()
    s, ref = capi.Scene(flat, lights=bright(lights)), capi.Scene(flat, lights=bright(lights))
    cams = cameras(capi, W, H)
    L = 3
    check_effects_views(s, cams[:4], W, H, L, BLOOM | BLUR, ref=ref)
    one, st1 = s.render(cams[3], W, H, trace_limit=L)
    want, sw = ref.render(cams[3], W, H, trace_limit=L)
    assert same_bits(one, want) and [st1[k] for k in RAYS] == [sw[k] for k in RAYS]
    views, stv = s.render_views(cams, W, H, trace_limit=L)
    wv, swv = ref.render_views(cams, W, H, trace_limit=L)
    assert same_bits(views, wv) and [stv[k] for k in RAYS] == [swv[k] for k in RAYS]
    fx, stf = s.render_effects(cams[1], W, H, trace_limit=L, motion_blur=True)
    wf, swf = ref.render_effects(cams[1], W, H, trace_limit=L, motion_blur=True)
    assert same_bits(fx, wf) and [stf[k] for k in RAYS] == [swf[k] for k in RAYS]
    w2, h2 = 200, 150
    cams2 = [capi.make_camera(w2, h2, euler_deg=(20.0, 20.0 + 30 * k, 0.0)) for k in range(5)]
    check_effects_views(s, cams2, w2, h2, L, AA, ref=ref)
    check_effects_views(s, cams2[:2], w2, h2, L, BLOOM, ref=ref)


@pytest.mark.gpu
def test_parameter_ring_outlasts_64_frames(capi, dragon):
    """80 cgrt_render_device frames of 80 cameras enqueued on one stream without a synchronisation: the per-frame parameter
    blocks go through a ring of 64 pinned slots, and each frame must still render its own camera."""
    import torch
    w, h, L = 640, 480, 5
    cams = [capi.make_camera(w, h, euler_deg=(20.0, 20.0 + 4.5 * k, 0.0)) for k in range(80)]
    out = torch.zeros((80, h, w, 3), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    stream = torch.cuda.Stream()
    p = capi.render_params(w, h, L)
    for k, cam in enumerate(cams):
        dragon.render_device(cam, p, out[k].data_ptr(), stream.cuda_stream)
    stream.synchronize()
    got = out.cpu().numpy()
    for k, cam in enumerate(cams):
        want, _ = dragon.render(cam, w, h, trace_limit=L)
        assert same_bits(got[k], want), k


@pytest.mark.gpu
def test_device_call_of_more_than_64_renders(capi, cornell):
    """65 views of 1024 x 1096 with motion blur: one view's 15 cameras per render (15 x 1.12 M slots), 65 renders in one
    device call, against the host form."""
    import torch
    w, h, L = 1024, 1096, 1
    cams = [capi.make_camera(w, h, euler_deg=(20.0, 20.0 + 5.0 * k, 0.0)) for k in range(65)]
    want, sw = cornell.render_effects_views(cams, w, h, trace_limit=L, motion_blur=True)
    got, st = _device_call(capi, cornell, cams, capi.render_params(w, h, L), BLUR, want.shape, torch.cuda.Stream())
    assert same_bits(got, want)
    assert [st[k] for k in RAYS] == [sw[k] for k in RAYS]
    del want, got
    # and three of those views against cgrt_render_effects
    check_effects_views(cornell, cams[::32], w, h, L, BLUR)


@pytest.mark.gpu
def test_effects_views_at_benchmark_size(capi, dragon):
    """C3's size: 4 views of 1920 x 1080 at trace limit 5, bloom + motion blur."""
    w, h = 1920, 1080
    cams = [capi.make_camera(w, h)] + [capi.make_camera(w, h, euler_deg=(20.0, 20.0 + 15 * k, 0.0)) for k in range(1, 4)]
    check_effects_views(dragon, cams, w, h, 5, BLOOM | BLUR)
