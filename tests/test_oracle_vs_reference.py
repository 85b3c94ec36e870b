"""CPU: restatement vs the reference's own TUs on fresh seeded inputs, including the reference CONSTRUCTOR (mode 0) and edge
cases (single triangle, two triangles, many meshes per leaf, empty scene, spheres). The reference's outputs for these inputs
are stored in tests/golden/vs_reference.npz (tests/golden/make_golden.py); the restatement and the product's host BVH builder
are checked against them everywhere, and against the reference itself where oracle/_ref is built."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, hits_equal, same_bits
from golden.make_golden import VS_REFERENCE_CASES, VS_REFERENCE_LIGHTS, empty_scene_inputs, vs_reference_inputs
from oracle import bindings as ob

COUNTERS = ("primary", "primary_hit", "shadow", "bounce")


@pytest.fixture(scope="module")
def stored():
    return np.load(os.path.join(GOLDEN, "vs_reference.npz"))


def leaf_order(b, meta):
    return np.concatenate([b.leaf_triangles(i, meta[i, 4]) for i in np.nonzero(meta[:, 0])[0]])


@pytest.mark.parametrize("ntri,nmesh,scale,seed", VS_REFERENCE_CASES)
def test_tree_hits_images(reflib, oracle, capi, stored, ntri, nmesh, scale, seed):
    flat, rays = vs_reference_inputs(ntri, nmesh, scale, seed)
    lights = VS_REFERENCE_LIGHTS
    g = {k.split("_", 1)[1]: stored[k] for k in stored.files if k.startswith(f"s{seed}_")}
    ob_ = oracle.scene(flat, lights).bvh()
    m1, a1 = ob_.nodes()
    assert np.array_equal(m1, g["node_meta"]) and same_bits(a1, g["node_aabb"])
    assert np.array_equal(leaf_order(ob_, m1), g["leaf_tris"])
    host = capi.Scene(flat, host_only=True)  # the product's range-based builder
    m2, a2 = host.nodes()
    assert np.array_equal(m2, g["node_meta"]) and same_bits(a2, g["node_aabb"])
    assert np.array_equal(flat.canonical_ids()[leaf_order(host, m2)], g["leaf_tris"])
    h1, c1 = ob_.intersect(rays, counts=True)
    assert hits_equal(h1, g["hits"]) and np.array_equal(c1, g["counts"])
    cam = ob.default_camera(64, 48)
    i1, k1 = ob_.render(cam, 64, 48, trace_limit=3, duplicate_shading=False)
    assert same_bits(i1, g["img_L3"])
    assert [k1[k] for k in COUNTERS] == g["cnt_L3"].tolist()
    if reflib is None:
        return
    rb = reflib.scene(flat, lights).bvh(mode=0)  # the reference constructor itself
    rf = reflib.scene(flat, lights).bvh(mode=1)  # range-based fill of reference Node structs
    m0, a0 = rb.nodes()
    for other in (rf, ob_):
        m, a = other.nodes()
        assert np.array_equal(m0, m) and same_bits(a0, a)
        for i in np.nonzero(m0[:, 0])[0]:
            assert np.array_equal(rb.leaf_triangles(i, m0[i, 4]), other.leaf_triangles(i, m[i, 4]))
    h0, c0 = rb.intersect(rays, counts=True)
    assert hits_equal(h1, h0) and np.array_equal(c0, c1)
    i0, k0 = rb.render(cam, 64, 48, trace_limit=3, duplicate_shading=True)
    assert same_bits(i0, i1)
    assert all(k0[k] == k1[k] for k in COUNTERS)


def test_empty_scene_and_spheres(reflib, oracle, capi, stored):
    empty, rays = empty_scene_inputs()
    assert oracle.scene(empty).bvh().num_nodes() == 0
    assert capi.Scene(empty, host_only=True).num_nodes() == 0
    h1 = oracle.scene(empty).bvh().intersect(rays)
    assert same_bits(h1["t"], stored["empty_t"]) and same_bits(h1["n"], stored["empty_n"])
    assert (h1["t"] < 1e30).sum() > 50
    if reflib is None:
        return
    assert reflib.scene(empty).bvh().num_nodes() == 0
    h0 = reflib.scene(empty).bvh(mode=0).intersect(rays)
    assert same_bits(h0["t"], h1["t"]) and same_bits(h0["n"], h1["n"])
