"""CPU: host logic of the product — C-ABI surface, loud failure without a GPU, the range-based BVH builder (host-only
scenes), the tile partition, the OBJ/MTL loader and the BMP writer. No compute call is made here."""
import ctypes
import os
import re
import struct

import numpy as np
import pytest

from conftest import GOLDEN, REFERENCE_DATA, ROOT, load_golden, same_bits
from oracle import bindings as ob


def declared_functions():
    names = []
    for h in ("cgrt_b200.h", "cgrt_host_c.h"):
        src = open(os.path.join(ROOT, "include", h)).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        names += re.findall(r"\b(cgrt_[a-z0-9_]+)\s*\(", src)
    return sorted(set(names))


def test_library_exports_every_declared_symbol(capi):
    lib = ctypes.CDLL(capi.LIB_PATH)
    names = declared_functions()
    assert len(names) >= 45
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    # and the ctypes binding covers the whole header
    bound = set(capi.EXPORTS) | set(capi.HOST_EXPORTS)
    assert set(names) <= bound, sorted(set(names) - bound)
    assert capi.load_library().cgrt_version() == 100


def test_no_gpu_means_loud_failure(capi):
    if capi.device_count() > 0:
        pytest.skip("a CUDA device is present")
    flat = ob.random_soup(10, seed=1, scale=0.3)
    with pytest.raises(capi.CgrtError) as e:
        capi.Scene(flat)
    assert e.value.code == capi.CGRT_ERR_NO_DEVICE
    with pytest.raises(capi.CgrtError):
        capi.ray_aabb(np.zeros((1, 6), np.float32), np.zeros(1, capi.RAY_DTYPE))
    host = capi.Scene(flat, host_only=True)
    with pytest.raises(capi.CgrtError) as e:
        host.intersect(ob.random_rays(4))
    assert e.value.code == capi.CGRT_ERR_NO_DEVICE
    with pytest.raises(capi.CgrtError):
        host.render(capi.make_camera(8, 8), 8, 8)


def test_product_does_not_reach_into_the_oracle():
    """the product path must never import / link / execute anything under oracle/"""
    pkg = os.path.join(ROOT, "cg-raytracer_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".hpp")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "liboracle" not in text and "libcgrt_ref" not in text and "from oracle" not in text and "import oracle" not in text, f


def test_builder_matches_golden_tree(capi, golden):
    """range-based host builder == the reference CONSTRUCTOR's tree (golden node table), node for node, bit for bit"""
    s = capi.Scene(golden.flat, host_only=True)
    meta, aabb = s.nodes()
    assert np.array_equal(meta, golden.z["node_meta"])
    assert same_bits(aabb, golden.z["node_aabb"])
    assert s.num_levels() == int(golden.z["num_levels"])
    canon = golden.flat.canonical_ids()
    leaves = np.nonzero(meta[:, 0])[0]
    order = np.concatenate([s.leaf_triangles(i, meta[i, 4]) for i in leaves])
    assert np.array_equal(canon[order], golden.z["leaf_tris"])
    assert sorted(order.tolist()) == list(range(golden.flat.n_triangles))  # every triangle in exactly one leaf


@pytest.mark.parametrize("ntri,nmesh,depth", [(1, 1, 12), (2, 1, 12), (5, 5, 12), (3000, 1, 12), (3000, 300, 12), (3000, 1, 1),
                                              (3000, 2, 2), (3000, 1, 20), (40000, 3, 12)])
def test_builder_matches_oracle_builder(capi, oracle, ntri, nmesh, depth):
    flat = ob.random_soup(ntri, seed=ntri + nmesh, scale=0.1, n_meshes=nmesh)
    s = capi.Scene(flat, host_only=True, bvh_max_depth=depth)
    b = oracle.scene(flat).bvh(max_depth=depth)
    m0, a0 = s.nodes()
    m1, a1 = b.nodes()
    assert np.array_equal(m0, m1) and same_bits(a0, a1)
    assert s.num_levels() == b.num_levels() <= depth
    canon = flat.canonical_ids()
    for i in np.nonzero(m0[:, 0])[0][:200]:
        assert np.array_equal(canon[s.leaf_triangles(i, m0[i, 4])], b.leaf_triangles(i, m1[i, 4]))


def test_scene_validation(capi):
    flat = ob.random_soup(10, seed=1, scale=0.3)
    flat.triangles[3, 1] = 10 ** 6
    with pytest.raises(capi.CgrtError) as e:
        capi.Scene(flat, host_only=True)
    assert e.value.code == capi.CGRT_ERR_INVALID
    with pytest.raises(capi.CgrtError):
        capi.Scene(ob.random_soup(10, seed=1), host_only=True, bvh_max_depth=500)
    empty = ob.FlatScene(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 6)), np.zeros((0, 3)), np.zeros((0, 8)))
    s = capi.Scene(empty, host_only=True)
    assert s.num_nodes() == 0 and s.num_triangles() == 0  # empty scene: no nodes (bvh.cpp:52-55)


@pytest.mark.parametrize("W,H,world,tile", [(1920, 1080, 8, (0, 0)), (1920, 1080, 4, (16, 4)), (3840, 2160, 8, (0, 0)),
                                            (100, 60, 3, (0, 0)), (7, 5, 2, (4, 4)), (64, 64, 1, (0, 0)), (33, 17, 6, (8, 2))])
def test_tile_partition(capi, W, H, world, tile):
    tw, th = (tile[0] or 8), (tile[1] or 8)
    tx, ty = -(-W // tw), -(-H // th)
    owned = [capi.tile_list(capi.render_params(W, H, 2, r, world, *tile), r) for r in range(world)]
    allt = np.concatenate(owned)
    assert sorted(allt.tolist()) == list(range(tx * ty))  # disjoint cover
    assert all(np.all(np.diff(o) > 0) for o in owned)  # increasing
    sizes = [len(o) for o in owned]
    assert max(sizes) - min(sizes) <= max(1, ty)  # balanced
    p = capi.render_params(W, H, 2, 0, world, *tile)
    floats = capi.tile_buffer_floats(p)
    assert floats == (W * H * 3 if world == 1 else max(sizes) * tw * th * 3)
    if world > 1 and tx >= world:  # interleaved: neighbours along x belong to different ranks
        owner = np.empty(tx * ty, np.int32)
        for r, o in enumerate(owned):
            owner[o] = r
        owner = owner.reshape(ty, tx)
        assert np.all(owner[:, 1:] != owner[:, :-1])
        if ty > 1:
            assert np.any(owner[1:, :] != owner[:-1, :])  # rows are skewed


def test_tile_partition_rejects_bad_arguments(capi):
    lib = capi.load_library()
    p = capi.render_params(64, 64, 2, 5, 4)
    assert lib.cgrt_tile_list(ctypes.byref(p), 5, None, 0) == -1
    assert capi.tile_buffer_floats(capi.render_params(0, 64, 2, 0, 1)) == 0


@pytest.mark.skipif(not os.path.isdir(REFERENCE_DATA), reason="CGRT_REFERENCE_DATA does not name a CG-RayTracer data/ directory")
@pytest.mark.parametrize("name,preset", [("triangle", "SingleTriangle"), ("cube", "Cube"), ("cornell", "CornellBox"),
                                         ("monkey", "Monkey")])
def test_loader_reproduces_fixture_scenes(capi, name, preset):
    g = load_golden(name)
    hs = capi.load_preset(preset, REFERENCE_DATA)
    assert np.array_equal(hs.vcount, g.flat.vcount) and np.array_equal(hs.tcount, g.flat.tcount)
    assert same_bits(hs.vertices, g.flat.vertices) and np.array_equal(hs.triangles, g.flat.triangles)
    assert same_bits(hs.materials, g.flat.materials) and same_bits(hs.lights, g.lights)


@pytest.mark.skipif(not os.path.isdir(REFERENCE_DATA), reason="CGRT_REFERENCE_DATA does not name a CG-RayTracer data/ directory")
def test_loader_details(capi):
    c = capi.load_preset("CornellBox", REFERENCE_DATA)
    # unit normalisation (mesh.cpp:143-166): farthest vertex at distance 1 from the mean of all (duplicated) vertices
    p = c.vertices[:, :3]
    assert abs(np.linalg.norm(p, axis=1).max() - 1.0) < 1e-6 and np.abs(p.mean(0)).max() < 1e-6
    # the mirror of the Cornell box is the only material with ks.z > 0.01 (shade(), main.cpp:246)
    assert (c.materials[:, 5] > 0.01).sum() >= 1
    assert np.allclose(c.lights, [[0, 0.58, 0, 1, 1, 1]])
    d = capi.load_obj(REFERENCE_DATA + "/dodgeColorTest.obj", True)
    assert len(d.vcount) == 11 and d.n_triangles == 16311 and int(d.vcount.sum()) == 48921
    # objects are visited in reverse file order (mesh.cpp node stack): the last object "Cube" (Material.001) comes first
    assert np.allclose(d.materials[0, :3], [0.64, 0.0, 0.055407], atol=1e-6)
    # no `vn` in that file: flat face normals on every corner, unit length
    n = np.linalg.norm(d.vertices[:, 3:], axis=1)
    assert np.all((np.abs(n - 1.0) < 1e-5) | (n == 0.0))  # NormalizeSafe leaves the 3 collinear faces of the model at zero
    assert (n == 0.0).sum() == 9
    t = capi.load_preset("SingleTriangle", REFERENCE_DATA)
    assert same_bits(t.vertices[:, 3:], np.tile(np.array([-1, 0, 0], np.float32), (3, 1)))  # generated, not the file's vn
    assert np.allclose(t.materials[0], [1, 1, 1, 0, 0, 0, 0, 1])  # kd overridden (scene.cpp:11), assimp default elsewhere
    sp = capi.load_preset("Spheres", REFERENCE_DATA)
    assert sp.spheres.shape == (3, 12) and sp.n_triangles == 0 and np.allclose(sp.lights, [[3, 0, 3, 15, 15, 15]])
    with pytest.raises(capi.CgrtError):
        capi.load_obj(REFERENCE_DATA + "/does-not-exist.obj")


def test_dragon_standin(capi):
    d = capi.dragon_standin()
    assert d.n_triangles == 87040 and len(d.vcount) == 1 and int(d.vcount[0]) == 3 * 87040
    p = d.vertices[:, :3]
    assert abs(np.linalg.norm(p, axis=1).max() - 1.0) < 1e-5
    assert np.allclose(np.linalg.norm(d.vertices[:, 3:], axis=1), 1.0, atol=1e-4)
    assert d.materials[0, 5] > 0.01  # mirror material so that the Whitted configuration bounces
    assert np.allclose(d.lights, [[-1, 1, -1, 1, 1, 1]])
    small = capi.dragon_standin(40, 16)
    assert small.n_triangles == 2 * 40 * 16
    again = capi.dragon_standin()
    assert same_bits(again.vertices, d.vertices)  # deterministic
    s = capi.Scene(d, host_only=True)
    assert s.num_levels() == 12 and s.num_nodes() == 4095  # as the report quotes for the dragon (12 levels)
    # the committed copy the CPU legs of bench.py and the full-size parity tests read (tests/golden/make_dragon_fixture.py)
    flat, lights = ob.dragon_standin_fixture()
    assert same_bits(flat.vertices, d.vertices) and np.array_equal(flat.triangles, d.triangles)
    assert same_bits(flat.materials, d.materials) and same_bits(lights, d.lights)
    assert np.array_equal(flat.vcount, d.vcount) and np.array_equal(flat.tcount, d.tcount)


def test_bmp_writer(capi, tmp_path):
    rng = np.random.default_rng(3)
    img = rng.uniform(-0.5, 1.5, (7, 5, 3)).astype(np.float32)
    img[0, 0] = [0.0, 1.0, 0.999999]
    path = tmp_path / "render.bmp"
    capi.write_bmp(path, img)
    raw = open(path, "rb").read()
    assert raw[:2] == b"BM"
    off, = struct.unpack_from("<I", raw, 10)
    w, h, planes, bpp = struct.unpack_from("<iiHH", raw, 18)
    assert (w, h, bpp) == (5, 7, 32)
    px = np.frombuffer(raw, np.uint8, offset=off).reshape(7, 5, 4)[::-1]  # bottom-up rows
    want = (np.clip(img, 0, 1) * np.float32(255.0)).astype(np.uint8)  # clamp, *255, truncate (screen.cpp:43-44)
    assert np.array_equal(px[..., [2, 1, 0]], want) and np.all(px[..., 3] == 255)


@pytest.mark.parametrize("ntri,nmesh,depth", [(1, 1, 12), (7, 1, 12), (9, 3, 12), (3000, 1, 12), (3000, 300, 12), (3000, 1, 1),
                                              (3000, 1, 20), (40000, 3, 12)])
def test_fast_tree_covers_every_triangle_once(capi, ntri, nmesh, depth):
    """the speculative traversal's tree: every triangle hangs under exactly one leaf, boxes contain their geometry, and every
    triangle's certificate chain (reference leaf -> parent -> ... -> root) is intact"""
    flat = ob.random_soup(ntri, seed=5 * ntri + nmesh, scale=0.1, n_meshes=nmesh)
    st = capi.Scene(flat, host_only=True, bvh_max_depth=depth).fast_tree_stats()
    assert st["present"] == 1
    assert st["triangles_reached"] == ntri and st["coverage_errors"] == 0
    assert st["containment_errors"] == 0 and st["chain_errors"] == 0
    assert st["depth"] <= 40
    assert capi.Scene(flat, host_only=True, exact_only=True).fast_tree_stats()["present"] == 0


def test_fast_tree_on_bundled_scenes(capi, golden):
    st = capi.Scene(golden.flat, host_only=True).fast_tree_stats()
    assert st["present"] == 1 and st["triangles_reached"] == golden.flat.n_triangles
    assert st["coverage_errors"] == 0 and st["containment_errors"] == 0 and st["chain_errors"] == 0


@pytest.mark.parametrize("flavour", ["sah", "ref"])
def test_fast_tree_flavours_are_structurally_sound(capi, golden, monkeypatch, flavour):
    """both fast-tree flavours (independent binned-SAH tree / reference tree collapsed on the leaf sub-trees) cover every
    triangle exactly once with boxes that contain their geometry; slivers and degenerate triangles included"""
    monkeypatch.setenv("CGRT_FAST_TREE", flavour)
    rng = np.random.default_rng(11)
    flat = ob.random_soup(5000, seed=99, scale=0.05, n_meshes=3)
    v = flat.vertices.copy()
    t = flat.triangles
    # make some triangles extreme slivers / degenerate (mesh-local indices: only touch mesh 0's first triangles)
    for k in range(6):
        a, b, c = t[k]
        v[c, :3] = v[a, :3] + (v[b, :3] - v[a, :3]) * np.float32(0.5) + rng.normal(0, 1e-9, 3).astype(np.float32)
    a, b, c = t[6]
    v[b, :3] = v[a, :3]
    flat2 = ob.FlatScene(flat.vcount, flat.tcount, v, t, flat.materials, flat.spheres)
    for f in (flat, flat2, golden.flat):
        st = capi.Scene(f, host_only=True).fast_tree_stats()
        assert st["present"] == 1 and st["triangles_reached"] == f.n_triangles
        assert st["coverage_errors"] == 0 and st["containment_errors"] == 0 and st["chain_errors"] == 0
    assert capi.Scene(flat2, host_only=True).fast_tree_stats()["always_tested"] >= 1
