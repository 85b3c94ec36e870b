"""ctypes binding of libcgrt_b200.so (include/cgrt_b200.h) — thin plumbing, no computation.

The library is the product; this module only marshals numpy / raw device pointers into the C ABI. It raises
`CgrtError` loudly when the shared library is missing or when the library reports that no CUDA device is usable:
there is no CPU fallback anywhere in the product path.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CGRT_LIB") or os.path.join(HERE, "libcgrt_b200.so")  # CGRT_LIB: A/B builds for tuning

RAY_DTYPE = np.dtype([("o", "f4", 3), ("t", "f4"), ("d", "f4", 3), ("pad", "f4")])
HIT_DTYPE = np.dtype([("t", "f4"), ("tri", "i4"), ("alpha", "f4"), ("beta", "f4"), ("gamma", "f4"), ("n", "f4", 3)])

CGRT_OK, CGRT_ERR_INVALID, CGRT_ERR_NO_DEVICE, CGRT_ERR_CUDA, CGRT_ERR_OOM = 0, 1, 2, 3, 4


class CgrtError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"cgrt error {code}: {msg}")
        self.code = code


class SceneDesc(C.Structure):
    _fields_ = [
        ("n_meshes", C.c_int32),
        ("mesh_vertex_count", C.POINTER(C.c_int32)),
        ("mesh_triangle_count", C.POINTER(C.c_int32)),
        ("vertices", C.POINTER(C.c_float)),
        ("triangles", C.POINTER(C.c_uint32)),
        ("materials", C.POINTER(C.c_float)),
        ("n_spheres", C.c_int32),
        ("spheres", C.POINTER(C.c_float)),
    ]


class SceneOptions(C.Structure):
    _fields_ = [("device", C.c_int32), ("bvh_max_depth", C.c_int32), ("flags", C.c_int32), ("reserved", C.c_int32 * 5)]


class Camera(C.Structure):
    _fields_ = [("fovy", C.c_float), ("aspect", C.c_float), ("dist", C.c_float),
                ("look_at", C.c_float * 3), ("euler", C.c_float * 3)]


class RenderParams(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("trace_limit", C.c_int32), ("rank", C.c_int32),
                ("world", C.c_int32), ("tile_w", C.c_int32), ("tile_h", C.c_int32), ("flags", C.c_int32),
                ("reserved", C.c_int32 * 4)]


class RenderStats(C.Structure):
    _fields_ = [("primary", C.c_uint64), ("primary_hit", C.c_uint64), ("shadow", C.c_uint64), ("bounce", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("box_tests", C.c_uint64 * 3), ("tri_tests", C.c_uint64 * 3),
                ("device_ms", C.c_float), ("class_ms", C.c_float * 4), ("class_launches", C.c_uint32 * 4),
                ("replayed_closest", C.c_uint32), ("replayed_shadow", C.c_uint32), ("pipeline", C.c_uint32)]

    def as_dict(self):
        return dict(primary=int(self.primary), primary_hit=int(self.primary_hit), shadow=int(self.shadow),
                    bounce=int(self.bounce), kernel_launches=int(self.kernel_launches), device_ms=float(self.device_ms),
                    box_tests=[int(v) for v in self.box_tests], tri_tests=[int(v) for v in self.tri_tests],
                    class_ms=[float(v) for v in self.class_ms], class_launches=[int(v) for v in self.class_launches],
                    replayed_closest=int(self.replayed_closest), replayed_shadow=int(self.replayed_shadow),
                    pipeline=int(self.pipeline))


class AovBuffers(C.Structure):
    """cgrt_aov_buffers: per-pixel buffers of cgrt_render_aovs (host or device pointers; None = not produced)."""
    _fields_ = [("depth", C.c_void_p), ("tri", C.c_void_p), ("normal", C.c_void_p), ("hits", C.c_void_p)]


class PathBuffers(C.Structure):
    """cgrt_path_buffers: every level of each pixel's mirror path (host or device pointers; None = not produced)."""
    _fields_ = [("ray", C.c_void_p), ("depth", C.c_void_p), ("tri", C.c_void_p), ("normal", C.c_void_p), ("position", C.c_void_p),
                ("visibility", C.c_void_p)]


PATH_KEYS = ("ray", "depth", "tri", "normal", "position", "visibility")

EXPORTS = [
    "cgrt_version", "cgrt_last_error", "cgrt_device_count", "cgrt_scene_create", "cgrt_scene_destroy",
    "cgrt_scene_set_lights", "cgrt_scene_set_spheres", "cgrt_bvh_num_levels", "cgrt_bvh_num_nodes",
    "cgrt_scene_num_triangles", "cgrt_bvh_export_nodes", "cgrt_bvh_leaf_triangles", "cgrt_intersect_closest",
    "cgrt_intersect_closest_device", "cgrt_intersect_any", "cgrt_intersect_any_device", "cgrt_intersect_brute",
    "cgrt_ray_aabb", "cgrt_ray_triangle", "cgrt_ray_plane", "cgrt_triangle_plane", "cgrt_point_in_triangle",
    "cgrt_ray_sphere", "cgrt_generate_rays", "cgrt_render", "cgrt_render_device", "cgrt_render_collect_stats",
    "cgrt_tile_buffer_floats", "cgrt_tile_list", "cgrt_assemble_tiles", "cgrt_quantize_rgba8", "cgrt_device_malloc", "cgrt_device_free",
    "cgrt_host_alloc_pinned", "cgrt_host_free_pinned", "cgrt_memcpy_h2d", "cgrt_memcpy_d2h", "cgrt_device_synchronize",
    "cgrt_memset_device", "cgrt_memcpy_d2h_async", "cgrt_peer_export", "cgrt_peer_open", "cgrt_peer_close",
    "cgrt_flag_signal", "cgrt_flag_wait", "cgrt_bvh_fast_tree_stats", "cgrt_render_submit", "cgrt_render_wait",
    "cgrt_render_effects", "cgrt_scene_set_spherical_lights", "cgrt_debug_wave_timeline", "cgrt_debug_wave_tuner",
    "cgrt_render_views", "cgrt_render_views_device", "cgrt_render_aovs", "cgrt_render_aovs_device",
    "cgrt_render_effects_views", "cgrt_render_effects_views_device", "cgrt_render_lights", "cgrt_render_lights_device",
    "cgrt_render_paths", "cgrt_render_paths_device",
]

_lib = None


def load_library(path=None):
    """Load libcgrt_b200.so; fail loudly if it has not been built (python -c 'import __graft_entry__ as g; g.build()')."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise CgrtError(-1, f"{path} not found: build the CUDA library first (__graft_entry__.build()); "
                            "there is no CPU fallback")
    lib = C.CDLL(path)
    vp, i32, u64, sz = C.c_void_p, C.c_int32, C.c_uint64, C.c_size_t
    fptr, u8p, u32p, i32p = C.POINTER(C.c_float), C.POINTER(C.c_uint8), C.POINTER(C.c_uint32), C.POINTER(C.c_int32)
    sig = {
        "cgrt_version": (C.c_int, []),
        "cgrt_last_error": (C.c_char_p, []),
        "cgrt_device_count": (C.c_int, [C.POINTER(C.c_int)]),
        "cgrt_scene_create": (C.c_int, [C.POINTER(SceneDesc), C.POINTER(SceneOptions), C.POINTER(vp)]),
        "cgrt_scene_destroy": (None, [vp]),
        "cgrt_scene_set_lights": (C.c_int, [vp, fptr, i32]),
        "cgrt_scene_set_spheres": (C.c_int, [vp, fptr, i32]),
        "cgrt_scene_set_spherical_lights": (C.c_int, [vp, fptr, i32, C.c_uint32]),
        "cgrt_debug_wave_timeline": (C.c_int, [vp, C.POINTER(C.c_int32), i32]),
        "cgrt_debug_wave_tuner": (C.c_int, [vp, C.POINTER(C.c_float), i32]),
        "cgrt_bvh_num_levels": (C.c_int, [vp]),
        "cgrt_bvh_num_nodes": (C.c_int, [vp]),
        "cgrt_scene_num_triangles": (C.c_int64, [vp]),
        "cgrt_bvh_export_nodes": (C.c_int, [vp, i32p, fptr]),
        "cgrt_bvh_leaf_triangles": (C.c_int, [vp, i32, i32p, i32]),
        "cgrt_intersect_closest": (C.c_int, [vp, vp, sz, vp, u32p]),
        "cgrt_intersect_closest_device": (C.c_int, [vp, vp, sz, vp, vp, vp]),
        "cgrt_intersect_any": (C.c_int, [vp, vp, fptr, C.c_float, sz, u8p]),
        "cgrt_intersect_any_device": (C.c_int, [vp, vp, vp, C.c_float, sz, vp, vp]),
        "cgrt_intersect_brute": (C.c_int, [vp, vp, sz, vp]),
        "cgrt_ray_aabb": (C.c_int, [C.c_int, fptr, vp, sz, u8p, fptr]),
        "cgrt_ray_triangle": (C.c_int, [C.c_int, fptr, vp, sz, vp]),
        "cgrt_ray_plane": (C.c_int, [C.c_int, fptr, vp, sz, u8p, fptr]),
        "cgrt_triangle_plane": (C.c_int, [C.c_int, fptr, sz, fptr]),
        "cgrt_point_in_triangle": (C.c_int, [C.c_int, fptr, sz, u8p]),
        "cgrt_ray_sphere": (C.c_int, [C.c_int, fptr, vp, sz, fptr]),
        "cgrt_generate_rays": (C.c_int, [C.c_int, C.POINTER(Camera), i32, i32, vp]),
        "cgrt_render": (C.c_int, [vp, C.POINTER(Camera), C.POINTER(RenderParams), vp, C.POINTER(RenderStats)]),
        "cgrt_render_device": (C.c_int, [vp, C.POINTER(Camera), C.POINTER(RenderParams), vp, vp]),
        "cgrt_render_views": (C.c_int, [vp, C.POINTER(Camera), i32, C.POINTER(RenderParams), vp, C.POINTER(RenderStats)]),
        "cgrt_render_views_device": (C.c_int, [vp, C.POINTER(Camera), i32, C.POINTER(RenderParams), vp, vp]),
        "cgrt_render_aovs": (C.c_int, [vp, C.POINTER(Camera), i32, C.POINTER(RenderParams), vp, C.POINTER(AovBuffers),
                                        C.POINTER(RenderStats)]),
        "cgrt_render_aovs_device": (C.c_int, [vp, C.POINTER(Camera), i32, C.POINTER(RenderParams), vp, C.POINTER(AovBuffers), vp]),
        "cgrt_render_lights": (C.c_int, [vp, C.POINTER(Camera), i32, C.POINTER(RenderParams), i32p, i32, i32, vp, vp,
                                          C.POINTER(RenderStats)]),
        "cgrt_render_lights_device": (C.c_int, [vp, C.POINTER(Camera), i32, C.POINTER(RenderParams), i32p, i32, i32, vp, vp, vp]),
        "cgrt_render_paths": (C.c_int, [vp, C.POINTER(Camera), i32, C.POINTER(RenderParams), i32, i32, vp, C.POINTER(PathBuffers),
                                         C.POINTER(RenderStats)]),
        "cgrt_render_paths_device": (C.c_int, [vp, C.POINTER(Camera), i32, C.POINTER(RenderParams), i32, i32, vp,
                                                C.POINTER(PathBuffers), vp]),
        "cgrt_render_collect_stats": (C.c_int, [vp, C.POINTER(RenderStats)]),
        "cgrt_tile_buffer_floats": (sz, [C.POINTER(RenderParams)]),
        "cgrt_tile_list": (C.c_int, [C.POINTER(RenderParams), i32, i32p, i32]),
        "cgrt_assemble_tiles": (C.c_int, [C.c_int, C.POINTER(RenderParams), vp, vp, vp]),
        "cgrt_quantize_rgba8": (C.c_int, [C.c_int, vp, sz, vp, vp]),
        "cgrt_device_malloc": (C.c_int, [C.c_int, sz, C.POINTER(vp)]),
        "cgrt_device_free": (C.c_int, [C.c_int, vp]),
        "cgrt_host_alloc_pinned": (C.c_int, [sz, C.POINTER(vp)]),
        "cgrt_host_free_pinned": (C.c_int, [vp]),
        "cgrt_memcpy_h2d": (C.c_int, [C.c_int, vp, vp, sz]),
        "cgrt_memcpy_d2h": (C.c_int, [C.c_int, vp, vp, sz]),
        "cgrt_device_synchronize": (C.c_int, [C.c_int]),
        "cgrt_memset_device": (C.c_int, [C.c_int, vp, C.c_int, sz, vp]),
        "cgrt_memcpy_d2h_async": (C.c_int, [C.c_int, vp, vp, sz, vp]),
        "cgrt_peer_export": (C.c_int, [C.c_int, vp, u8p]),
        "cgrt_peer_open": (C.c_int, [C.c_int, u8p, C.POINTER(vp)]),
        "cgrt_peer_close": (C.c_int, [C.c_int, vp]),
        "cgrt_flag_signal": (C.c_int, [C.c_int, C.POINTER(vp), i32, C.c_uint32, vp]),
        "cgrt_flag_wait": (C.c_int, [C.c_int, vp, i32, C.c_uint32, C.c_uint32, vp, vp]),
        "cgrt_bvh_fast_tree_stats": (C.c_int, [vp, C.POINTER(C.c_int64)]),
        "cgrt_render_submit": (C.c_int, [vp, C.POINTER(Camera), C.POINTER(RenderParams), vp]),
        "cgrt_render_wait": (C.c_int, [vp]),
        "cgrt_render_effects": (C.c_int, [vp, C.POINTER(Camera), C.POINTER(RenderParams), i32, vp, C.POINTER(RenderStats)]),
        "cgrt_render_effects_views": (C.c_int, [vp, C.POINTER(Camera), i32, C.POINTER(RenderParams), i32, vp,
                                                 C.POINTER(RenderStats)]),
        "cgrt_render_effects_views_device": (C.c_int, [vp, C.POINTER(Camera), i32, C.POINTER(RenderParams), i32, vp, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError here = header/library drift
        fn.restype = res
        fn.argtypes = args
    if path == LIB_PATH:
        _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise CgrtError(rc, (load_library().cgrt_last_error() or b"").decode())


def device_count():
    n = C.c_int(0)
    rc = load_library().cgrt_device_count(C.byref(n))
    return n.value if rc == 0 else 0


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _vp(a):
    return C.c_void_p(a.ctypes.data)


def make_camera(W, H, fovy_deg=50.0, dist=3.0, look_at=(0.0, 0.0, 0.0), euler_deg=(20.0, 20.0, 0.0)):
    """Reference camera preset (src/main.cpp:730-731): fovy 50 deg, distance 3, rotations (20, 20, 0) deg; aspect = W/H."""
    k = np.float32(0.01745329251994329576923690768489)  # glm::radians
    c = Camera()
    c.fovy = np.float32(fovy_deg) * k
    c.aspect = np.float32(W) / np.float32(H)
    c.dist = dist
    c.look_at[:] = list(look_at)
    c.euler[:] = [float(np.float32(e) * k) for e in euler_deg]
    return c


K_PRIMARY, K_BOUNCE, K_SHADOW, K_SHADE = 0, 1, 2, 3
# kernels per class of each pipeline, indexed by cgrt_render_stats.pipeline (0 count, 1 paths, 2 rounds, 3 k_wave). Frames of
# scenes with a search tree run k_wave or the round pipeline, chosen per frame (DESIGN 4.4); the path pipeline launches no
# class-1 kernel (k_paths follows each path through its bounces)
KERNEL_CLASS_NAMES = ["k_paths", "k_bounce_closest", "k_shadow_all", "k_shade_paths"]  # path pipeline (scenes without a search tree)
ROUND_CLASS_NAMES = ["k_gen", "k_finish", "k_trace", "k_shade_slots"]                   # round pipeline (large shallow frames)
WAVE_CLASS_NAMES = ["-", "-", "k_wave", "-"]                                             # persistent wavefront (the other frames)
COUNT_CLASS_NAMES = ["k_primary", "k_bounce_closest", "k_shadow", "k_shade"]             # counting wavefront (CGRT_RENDER_COUNT)


def class_names(stats):
    """Kernel names behind cgrt_render_stats.class_ms / class_launches for the pipeline that produced `stats`."""
    return [COUNT_CLASS_NAMES, KERNEL_CLASS_NAMES, ROUND_CLASS_NAMES, WAVE_CLASS_NAMES][stats["pipeline"]]
RENDER_PROFILE_ALL, RENDER_COUNT, RENDER_SCREEN_LAYOUT = 0xF, 0x100, 0x200
IPC_HANDLE_BYTES = 64


EFFECT_ANTIALIAS, EFFECT_MOTION_BLUR, EFFECT_BLOOM = 1, 2, 4


def effects_mask(antialias=False, motion_blur=False, bloom=False):
    """The `effects` bits of cgrt_render_effects / cgrt_render_effects_views."""
    return (EFFECT_ANTIALIAS if antialias else 0) | (EFFECT_MOTION_BLUR if motion_blur else 0) | (EFFECT_BLOOM if bloom else 0)


def render_params(W, H, trace_limit=2, rank=0, world=1, tile_w=0, tile_h=0, flags=0):
    p = RenderParams()
    p.width, p.height, p.trace_limit, p.rank, p.world, p.tile_w, p.tile_h = W, H, trace_limit, rank, world, tile_w, tile_h
    p.flags = flags
    return p


class Scene:
    """Device-resident scene + BVH (cgrt_scene). `flat` needs the attributes of the flat-scene layout /
    host loader output: vcount, tcount, vertices[.,6], triangles[.,3], materials[.,8], spheres[.,12]."""

    def __init__(self, flat, lights=None, device=0, bvh_max_depth=12, host_only=False, no_subtrees=False, exact_only=None):
        self.lib = load_library()
        self.device = device
        self._keep = (np.ascontiguousarray(flat.vcount, np.int32), np.ascontiguousarray(flat.tcount, np.int32),
                      np.ascontiguousarray(flat.vertices, np.float32), np.ascontiguousarray(flat.triangles, np.uint32),
                      np.ascontiguousarray(flat.materials, np.float32), np.ascontiguousarray(flat.spheres, np.float32))
        vc, tc, v, t, m, s = self._keep
        d = SceneDesc()
        d.n_meshes = len(vc)
        d.mesh_vertex_count = vc.ctypes.data_as(C.POINTER(C.c_int32))
        d.mesh_triangle_count = tc.ctypes.data_as(C.POINTER(C.c_int32))
        d.vertices = _fp(v)
        d.triangles = t.ctypes.data_as(C.POINTER(C.c_uint32))
        d.materials = _fp(m)
        d.n_spheres = s.reshape(-1, 12).shape[0]
        d.spheres = _fp(s)
        o = SceneOptions()
        o.device = device
        o.bvh_max_depth = bvh_max_depth
        if exact_only is None:  # CGRT_EXACT_ONLY=1: run everything through the exact traversal (A/B for tests / profiling)
            exact_only = os.environ.get("CGRT_EXACT_ONLY", "0") == "1"
        # CGRT_SCENE_HOST_ONLY | CGRT_SCENE_NO_SUBTREES | CGRT_SCENE_EXACT_ONLY
        o.flags = (1 if host_only else 0) | (2 if no_subtrees else 0) | (4 if exact_only else 0)
        h = C.c_void_p()
        check(self.lib.cgrt_scene_create(C.byref(d), C.byref(o), C.byref(h)))
        self.h = h
        self.n_point_lights = self.n_spherical_lights = 0  # as set_lights / set_spherical_lights gave them (render_lights' groups, render_paths' visibility)
        if lights is not None:
            self.set_lights(lights)

    def close(self):
        if getattr(self, "h", None):
            self.lib.cgrt_scene_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_lights(self, lights):
        l = np.ascontiguousarray(lights, np.float32).reshape(-1, 6)
        check(self.lib.cgrt_scene_set_lights(self.h, _fp(l), l.shape[0]))
        self.n_point_lights = l.shape[0]

    def set_spherical_lights(self, lights, seed=1):
        """Scene::sphericalLight: [n][7] = position, radius, colour (soft shadows of main.cpp:168-218)."""
        l = np.ascontiguousarray(lights, np.float32).reshape(-1, 7)
        check(self.lib.cgrt_scene_set_spherical_lights(self.h, _fp(l), l.shape[0], seed))
        self.n_spherical_lights = l.shape[0]

    def set_spheres(self, spheres):
        s = np.ascontiguousarray(spheres, np.float32).reshape(-1, 12)
        check(self.lib.cgrt_scene_set_spheres(self.h, _fp(s), s.shape[0]))

    # -- BVH introspection
    def num_levels(self):
        return self.lib.cgrt_bvh_num_levels(self.h)

    def num_nodes(self):
        return self.lib.cgrt_bvh_num_nodes(self.h)

    def num_triangles(self):
        return int(self.lib.cgrt_scene_num_triangles(self.h))

    def fast_tree_stats(self):
        out = (C.c_int64 * 8)()
        check(self.lib.cgrt_bvh_fast_tree_stats(self.h, out))
        keys = ("wide_nodes", "triangles_reached", "coverage_errors", "containment_errors", "depth", "chain_errors", "present",
                "always_tested")
        return dict(zip(keys, [int(v) for v in out]))

    def nodes(self):
        n = self.num_nodes()
        meta = np.zeros((n, 5), np.int32)
        aabb = np.zeros((n, 6), np.float32)
        if n:
            check(self.lib.cgrt_bvh_export_nodes(self.h, meta.ctypes.data_as(C.POINTER(C.c_int32)), _fp(aabb)))
        return meta, aabb

    def leaf_triangles(self, node, count):
        out = np.zeros(max(count, 1), np.int32)
        k = self.lib.cgrt_bvh_leaf_triangles(self.h, node, out.ctypes.data_as(C.POINTER(C.c_int32)), count)
        assert k == count, (k, count)
        return out[:count]

    # -- queries (host buffers through the C ABI)
    def intersect(self, rays, counts=False):
        rays = np.ascontiguousarray(rays)
        n = rays.shape[0]
        hits = np.zeros(n, HIT_DTYPE)
        cnt = np.zeros((n, 2), np.uint32) if counts else None
        check(self.lib.cgrt_intersect_closest(self.h, _vp(rays), n, _vp(hits),
                                              cnt.ctypes.data_as(C.POINTER(C.c_uint32)) if counts else None))
        return (hits, cnt) if counts else hits

    def intersect_any(self, rays, max_dist, eps=0.001):
        rays = np.ascontiguousarray(rays)
        md = np.ascontiguousarray(max_dist, np.float32)
        n = rays.shape[0]
        occ = np.zeros(n, np.uint8)
        check(self.lib.cgrt_intersect_any(self.h, _vp(rays), _fp(md), eps, n, occ.ctypes.data_as(C.POINTER(C.c_uint8))))
        return occ.astype(bool)

    def intersect_brute(self, rays):
        rays = np.ascontiguousarray(rays)
        hits = np.zeros(rays.shape[0], HIT_DTYPE)
        check(self.lib.cgrt_intersect_brute(self.h, _vp(rays), rays.shape[0], _vp(hits)))
        return hits

    def render(self, cam, W, H, trace_limit=2, rank=0, world=1, tile=(0, 0), out=None, flags=0):
        """Full C-ABI host path: returns (rgb[H,W,3] in Screen layout, stats dict)."""
        p = render_params(W, H, trace_limit, rank, world, tile[0], tile[1], flags)
        rgb = np.zeros((H, W, 3), np.float32) if out is None else out
        st = RenderStats()
        check(self.lib.cgrt_render(self.h, C.byref(cam), C.byref(p), _vp(rgb), C.byref(st)))
        return rgb, st.as_dict()

    def render_effects(self, cam, W, H, trace_limit=2, antialias=False, motion_blur=False, bloom=False):
        """renderRayTracing's anti-aliasing / motion-blur / bloom passes (cgrt_render_effects): (rgb[H,W,3], stats dict)."""
        p = render_params(W, H, trace_limit)
        rgb = np.zeros((H, W, 3), np.float32)
        st = RenderStats()
        check(self.lib.cgrt_render_effects(self.h, C.byref(cam), C.byref(p), (1 if antialias else 0) | (2 if motion_blur else 0) | (4 if bloom else 0),
                                           _vp(rgb), C.byref(st)))
        return rgb, st.as_dict()

    def render_effects_views(self, cams, W, H, trace_limit=2, antialias=False, motion_blur=False, bloom=False):
        """cgrt_render_effects_views: the effects of render_effects for several cameras in one call: (rgb[K,H,W,3], stats dict
        summed over the renders)."""
        arr = (Camera * len(cams))(*cams)
        p = render_params(W, H, trace_limit)
        rgb = np.zeros((len(cams), H, W, 3), np.float32)
        st = RenderStats()
        check(self.lib.cgrt_render_effects_views(self.h, arr, len(cams), C.byref(p), effects_mask(antialias, motion_blur, bloom),
                                                 _vp(rgb), C.byref(st)))
        return rgb, st.as_dict()

    def render_effects_views_device(self, cams, params, effects, d_out_ptr, stream_ptr=0):
        """Device form: [K][H][W][3] floats into d_out_ptr on the stream; statistics through collect_stats()."""
        arr = (Camera * len(cams))(*cams)
        check(self.lib.cgrt_render_effects_views_device(self.h, arr, len(cams), C.byref(params), effects, C.c_void_p(d_out_ptr),
                                                        C.c_void_p(stream_ptr)))

    def render_submit(self, cam, params, host_ptr):
        """Streaming form: enqueue one frame into page-locked host memory (see cgrt_render_submit)."""
        check(self.lib.cgrt_render_submit(self.h, C.byref(cam), C.byref(params), C.c_void_p(host_ptr)))

    def render_wait(self):
        check(self.lib.cgrt_render_wait(self.h))

    def render_device(self, cam, params, d_out_ptr, stream_ptr=0):
        check(self.lib.cgrt_render_device(self.h, C.byref(cam), C.byref(params), C.c_void_p(d_out_ptr), C.c_void_p(stream_ptr)))

    def render_views(self, cams, W, H, trace_limit=2, flags=0):
        """Several cameras of this scene in one frame (cgrt_render_views): (rgb[K,H,W,3], stats dict summed over the views)."""
        arr = (Camera * len(cams))(*cams)
        p = render_params(W, H, trace_limit, flags=flags)
        rgb = np.zeros((len(cams), H, W, 3), np.float32)
        st = RenderStats()
        check(self.lib.cgrt_render_views(self.h, arr, len(cams), C.byref(p), _vp(rgb), C.byref(st)))
        return rgb, st.as_dict()

    def render_views_device(self, cams, params, d_out_ptr, stream_ptr=0):
        """Device form: [K][H][W][3] floats into d_out_ptr on the stream; statistics through collect_stats()."""
        arr = (Camera * len(cams))(*cams)
        check(self.lib.cgrt_render_views_device(self.h, arr, len(cams), C.byref(params), C.c_void_p(d_out_ptr),
                                                C.c_void_p(stream_ptr)))

    def render_aovs(self, cams, W, H, trace_limit=2, tile=(0, 0), flags=0, depth=True, tri=True, normal=True, hits=True):
        """cgrt_render_aovs: (rgb[K,H,W,3], {"depth": float32[K,H,W], "tri": int32[K,H,W], "normal": float32[K,H,W,3],
        "hits": uint8[K,H,W]} with the requested keys only, stats dict summed over the views). Screen layout, like rgb."""
        K = len(cams)
        arr = (Camera * K)(*cams)
        p = render_params(W, H, trace_limit, tile_w=tile[0], tile_h=tile[1], flags=flags)
        rgb = np.zeros((K, H, W, 3), np.float32)
        want = dict(depth=(depth, (K, H, W), np.float32), tri=(tri, (K, H, W), np.int32),
                    normal=(normal, (K, H, W, 3), np.float32), hits=(hits, (K, H, W), np.uint8))
        out = {k: np.zeros(shp, dt) for k, (on, shp, dt) in want.items() if on}
        a = AovBuffers(*[out[k].ctypes.data if k in out else None for k in ("depth", "tri", "normal", "hits")])
        st = RenderStats()
        check(self.lib.cgrt_render_aovs(self.h, arr, K, C.byref(p), _vp(rgb), C.byref(a), C.byref(st)))
        return rgb, out, st.as_dict()

    def render_aovs_device(self, cams, params, d_rgb_ptr, d_aov_ptrs, stream_ptr=0):
        """Device form: rgb [K][H][W][3] into d_rgb_ptr and the buffers of d_aov_ptrs (dict of device pointers with keys
        depth / tri / normal / hits; a missing key or None = not produced) on the stream; statistics through collect_stats()."""
        arr = (Camera * len(cams))(*cams)
        a = AovBuffers(*[d_aov_ptrs.get(k) for k in ("depth", "tri", "normal", "hits")])
        check(self.lib.cgrt_render_aovs_device(self.h, arr, len(cams), C.byref(params), C.c_void_p(d_rgb_ptr), C.byref(a),
                                               C.c_void_p(stream_ptr)))

    def render_lights(self, cams, W, H, trace_limit=2, groups=None, n_groups=None):
        """cgrt_render_lights: (rgb[K,H,W,3], light_rgb[G,K,H,W,3], stats dict summed over the views), Screen layout.
        groups: each light's group (point lights, then spherical lights; -1 = in no group); default one group per light in
        that order. n_groups: G, default max(groups) + 1. Group g is bit for bit the frame with every light outside g black."""
        n = self.n_point_lights + self.n_spherical_lights
        lg = np.ascontiguousarray(np.arange(n) if groups is None else groups, np.int32)
        G = int(n_groups if n_groups is not None else max(int(lg.max(initial=-1)) + 1, 1))
        K = len(cams)
        arr = (Camera * K)(*cams)
        p = render_params(W, H, trace_limit)
        rgb = np.zeros((K, H, W, 3), np.float32)
        light_rgb = np.zeros((G, K, H, W, 3), np.float32)
        st = RenderStats()
        check(self.lib.cgrt_render_lights(self.h, arr, K, C.byref(p), lg.ctypes.data_as(C.POINTER(C.c_int32)), len(lg), G,
                                          _vp(rgb), _vp(light_rgb), C.byref(st)))
        return rgb, light_rgb, st.as_dict()

    def render_lights_device(self, cams, params, groups, n_groups, d_rgb_ptr, d_groups_ptr, stream_ptr=0):
        """Device form: rgb [K][H][W][3] into d_rgb_ptr and the groups [n_groups][K][H][W][3] into d_groups_ptr on the stream;
        groups is the host list of each light's group. Statistics through collect_stats()."""
        arr = (Camera * len(cams))(*cams)
        lg = np.ascontiguousarray(groups, np.int32)
        check(self.lib.cgrt_render_lights_device(self.h, arr, len(cams), C.byref(params), lg.ctypes.data_as(C.POINTER(C.c_int32)),
                                                 len(lg), n_groups, C.c_void_p(d_rgb_ptr), C.c_void_p(d_groups_ptr),
                                                 C.c_void_p(stream_ptr)))

    def render_paths(self, cams, W, H, trace_limit=2, n_levels=None, ray=True, depth=True, tri=True, normal=True, position=True,
                     visibility=True):
        """cgrt_render_paths: (rgb[K,H,W,3], {"ray": RAY_DTYPE[Lv,K,H,W], "depth": float32[Lv,K,H,W], "tri": int32[Lv,K,H,W],
        "normal" / "position": float32[Lv,K,H,W,3], "visibility": float32[Lv,K,H,W,n_lights]} with the requested keys only,
        stats dict summed over the views). Level l is the ray trace(l) cast and its hit; Screen layout, like rgb. n_levels
        (Lv): default max(trace_limit, 1). Lights: point lights, then spherical lights."""
        K = len(cams)
        Lv = int(n_levels if n_levels is not None else max(trace_limit, 1))
        nl = self.n_point_lights + self.n_spherical_lights
        arr = (Camera * K)(*cams)
        p = render_params(W, H, trace_limit)
        rgb = np.zeros((K, H, W, 3), np.float32)
        want = dict(ray=(ray, (Lv, K, H, W), RAY_DTYPE), depth=(depth, (Lv, K, H, W), np.float32), tri=(tri, (Lv, K, H, W), np.int32),
                    normal=(normal, (Lv, K, H, W, 3), np.float32), position=(position, (Lv, K, H, W, 3), np.float32),
                    visibility=(visibility, (Lv, K, H, W, nl), np.float32))
        out = {k: np.zeros(shp, dt) for k, (on, shp, dt) in want.items() if on}
        b = PathBuffers(*[out[k].ctypes.data if k in out else None for k in PATH_KEYS])
        st = RenderStats()
        check(self.lib.cgrt_render_paths(self.h, arr, K, C.byref(p), Lv, nl, _vp(rgb), C.byref(b), C.byref(st)))
        return rgb, out, st.as_dict()

    def render_paths_device(self, cams, params, n_levels, d_rgb_ptr, d_path_ptrs, stream_ptr=0):
        """Device form: rgb [K][H][W][3] into d_rgb_ptr and the buffers of d_path_ptrs (dict of device pointers with the keys of
        render_paths; a missing key or None = not produced) on the stream; statistics through collect_stats()."""
        arr = (Camera * len(cams))(*cams)
        b = PathBuffers(*[d_path_ptrs.get(k) for k in PATH_KEYS])
        check(self.lib.cgrt_render_paths_device(self.h, arr, len(cams), C.byref(params), n_levels,
                                                self.n_point_lights + self.n_spherical_lights, C.c_void_p(d_rgb_ptr), C.byref(b),
                                                C.c_void_p(stream_ptr)))

    def collect_stats(self):
        st = RenderStats()
        check(self.lib.cgrt_render_collect_stats(self.h, C.byref(st)))
        return st.as_dict()


def relight(light_rgb, gains):
    """sum_g gains[g] * light_rgb[g]: the frame with group g's light colours scaled by gains[g] ([G][3], per channel), from the
    buffers of Scene.render_lights without tracing again. Approximate: it matches a render with the scaled colours only up to
    float rounding (the render scales each light before summing, this scales the group's sum)."""
    light_rgb = np.asarray(light_rgb, np.float32)
    g = np.asarray(gains, np.float32).reshape(light_rgb.shape[0], 1, 1, 1, 3)
    return (light_rgb * g).sum(axis=0, dtype=np.float32)


# -- unit predicates (src/ray_tracing.h:10-20), batched, host buffers ---------------------------------------------------
def ray_aabb(boxes, rays, device=0):
    lib = load_library()
    boxes = np.ascontiguousarray(boxes, np.float32).reshape(-1, 6)
    n = boxes.shape[0]
    hit = np.zeros(n, np.uint8)
    t = np.zeros(n, np.float32)
    check(lib.cgrt_ray_aabb(device, _fp(boxes), _vp(np.ascontiguousarray(rays)), n, hit.ctypes.data_as(C.POINTER(C.c_uint8)), _fp(t)))
    return hit.astype(bool), t


def ray_triangle(tris, rays, device=0):
    lib = load_library()
    tris = np.ascontiguousarray(tris, np.float32).reshape(-1, 18)
    out = np.zeros(tris.shape[0], HIT_DTYPE)
    check(lib.cgrt_ray_triangle(device, _fp(tris), _vp(np.ascontiguousarray(rays)), tris.shape[0], _vp(out)))
    return out


def ray_plane(planes, rays, device=0):
    lib = load_library()
    planes = np.ascontiguousarray(planes, np.float32).reshape(-1, 4)
    n = planes.shape[0]
    hit = np.zeros(n, np.uint8)
    t = np.zeros(n, np.float32)
    check(lib.cgrt_ray_plane(device, _fp(planes), _vp(np.ascontiguousarray(rays)), n, hit.ctypes.data_as(C.POINTER(C.c_uint8)), _fp(t)))
    return hit.astype(bool), t


def triangle_plane(tris, device=0):
    lib = load_library()
    tris = np.ascontiguousarray(tris, np.float32).reshape(-1, 9)
    out = np.zeros((tris.shape[0], 4), np.float32)
    check(lib.cgrt_triangle_plane(device, _fp(tris), tris.shape[0], _fp(out)))
    return out


def point_in_triangle(a, device=0):
    lib = load_library()
    a = np.ascontiguousarray(a, np.float32).reshape(-1, 15)
    out = np.zeros(a.shape[0], np.uint8)
    check(lib.cgrt_point_in_triangle(device, _fp(a), a.shape[0], out.ctypes.data_as(C.POINTER(C.c_uint8))))
    return out.astype(bool)


def ray_sphere(spheres, rays, device=0):
    lib = load_library()
    s = np.ascontiguousarray(spheres, np.float32).reshape(-1, 4)
    out = np.zeros((s.shape[0], 5), np.float32)
    check(lib.cgrt_ray_sphere(device, _fp(s), _vp(np.ascontiguousarray(rays)), s.shape[0], _fp(out)))
    return out[:, 0].copy(), out[:, 1].copy().view(np.int32).astype(bool), out[:, 2:5].copy()


def tile_list(params, rank):
    """Global tile ids owned by `rank` under the interleaved partition (host arithmetic only, no GPU needed)."""
    lib = load_library()
    n = lib.cgrt_tile_list(C.byref(params), rank, None, 0)
    if n < 0:
        raise CgrtError(CGRT_ERR_INVALID, "cgrt_tile_list: bad arguments")
    out = np.zeros(max(n, 1), np.int32)
    lib.cgrt_tile_list(C.byref(params), rank, out.ctypes.data_as(C.POINTER(C.c_int32)), n)
    return out[:n]


def tile_buffer_floats(params):
    return int(load_library().cgrt_tile_buffer_floats(C.byref(params)))


def generate_rays(cam, W, H, device=0):
    lib = load_library()
    rays = np.zeros(W * H, RAY_DTYPE)
    check(lib.cgrt_generate_rays(device, C.byref(cam), W, H, _vp(rays)))
    return rays


# -- host-side data formats (include/cgrt_host_c.h): OBJ/MTL loader, scene presets, BMP writer ----------------------------
HOST_EXPORTS = ["cgrt_host_set_default_device", "cgrt_host_scene_load_preset", "cgrt_host_scene_load_obj",
                "cgrt_host_scene_dragon_standin", "cgrt_host_scene_destroy", "cgrt_host_scene_desc",
                "cgrt_host_scene_counts", "cgrt_host_scene_lights", "cgrt_write_bmp"]


def _host_sigs(lib):
    if getattr(lib, "_cgrt_host_ready", False):
        return lib
    vp = C.c_void_p
    lib.cgrt_host_set_default_device.argtypes = [C.c_int]
    lib.cgrt_host_set_default_device.restype = None
    lib.cgrt_host_scene_load_preset.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(vp)]
    lib.cgrt_host_scene_load_obj.argtypes = [C.c_char_p, C.c_int, C.POINTER(vp)]
    lib.cgrt_host_scene_dragon_standin.argtypes = [C.c_int, C.c_int, C.POINTER(vp)]
    lib.cgrt_host_scene_destroy.argtypes = [vp]
    lib.cgrt_host_scene_destroy.restype = None
    lib.cgrt_host_scene_desc.argtypes = [vp, C.POINTER(SceneDesc)]
    lib.cgrt_host_scene_counts.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.cgrt_host_scene_counts.restype = C.c_int64
    lib.cgrt_host_scene_lights.argtypes = [vp, C.POINTER(C.c_float), C.c_int]
    lib.cgrt_write_bmp.argtypes = [C.c_char_p, C.POINTER(C.c_float), C.c_int, C.c_int]
    lib._cgrt_host_ready = True
    return lib


class HostScene:
    """A Scene produced by the host loader (loadScene / loadMesh / the dragon stand-in), exposed as flat numpy arrays
    with the attribute names Scene() expects (vcount, tcount, vertices, triangles, materials, spheres) plus `lights`."""

    def __init__(self, handle, name):
        lib = _host_sigs(load_library())
        self.name = name
        nv, nt = C.c_int64(0), C.c_int64(0)
        nm = int(lib.cgrt_host_scene_counts(handle, C.byref(nv), C.byref(nt)))
        d = SceneDesc()
        if lib.cgrt_host_scene_desc(handle, C.byref(d)) != 0:
            raise CgrtError(CGRT_ERR_INVALID, "cgrt_host_scene_desc failed")
        def arr(ptr, count, dtype):
            if count == 0:
                return np.zeros(0, dtype)
            return np.ctypeslib.as_array(ptr, shape=(count,)).astype(dtype, copy=True)
        self.vcount = arr(d.mesh_vertex_count, nm, np.int32)
        self.tcount = arr(d.mesh_triangle_count, nm, np.int32)
        self.vertices = arr(d.vertices, nv.value * 6, np.float32).reshape(-1, 6)
        self.triangles = arr(d.triangles, nt.value * 3, np.uint32).reshape(-1, 3)
        self.materials = arr(d.materials, nm * 8, np.float32).reshape(-1, 8)
        self.spheres = arr(d.spheres, d.n_spheres * 12, np.float32).reshape(-1, 12)
        nl = lib.cgrt_host_scene_lights(handle, None, 0)
        self.lights = np.zeros((nl, 6), np.float32)
        if nl:
            lib.cgrt_host_scene_lights(handle, _fp(self.lights), nl)
        lib.cgrt_host_scene_destroy(handle)

    @property
    def n_triangles(self):
        return int(self.tcount.sum())


def load_preset(preset, data_dir):
    lib = _host_sigs(load_library())
    h = C.c_void_p()
    rc = lib.cgrt_host_scene_load_preset(preset.encode(), str(data_dir).encode(), C.byref(h))
    if rc != 0:
        raise CgrtError(rc, f"loadScene({preset}, {data_dir}) failed")
    return HostScene(h, preset)


def load_obj(path, normalize=False):
    lib = _host_sigs(load_library())
    h = C.c_void_p()
    rc = lib.cgrt_host_scene_load_obj(str(path).encode(), int(normalize), C.byref(h))
    if rc != 0:
        raise CgrtError(rc, f"loadMesh({path}) failed")
    return HostScene(h, str(path))


def dragon_standin(segments_u=340, segments_v=128):
    lib = _host_sigs(load_library())
    h = C.c_void_p()
    rc = lib.cgrt_host_scene_dragon_standin(segments_u, segments_v, C.byref(h))
    if rc != 0:
        raise CgrtError(rc, "dragon stand-in failed")
    return HostScene(h, f"dragon-standin-{2 * segments_u * segments_v}tri")


def write_bmp(path, rgb):
    lib = _host_sigs(load_library())
    rgb = np.ascontiguousarray(rgb, np.float32)
    H, W = rgb.shape[:2]
    rc = lib.cgrt_write_bmp(str(path).encode(), _fp(rgb), W, H)
    if rc != 0:
        raise CgrtError(rc, f"write_bmp({path}) failed")
