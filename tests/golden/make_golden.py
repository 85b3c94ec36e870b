"""Generate the golden fixtures under tests/golden/ from the REFERENCE ITSELF.

Run in the build container (needs /root/reference and oracle/_ref/libcgrt_ref.so, i.e. the reference's own
ray_tracing.cpp + bounding_volume_hierarchy.cpp compiled verbatim):

    python tests/golden/make_golden.py

For every bundled scene the fixture stores
  * the flattened scene the loader produced from /root/reference/data (so that tests on the GPU box, where the reference
    checkout does not exist, consume identical inputs), its preset lights,
  * outputs of the verbatim reference code on it: BVH node table (reference CONSTRUCTOR, mode 0), leaf triangle orders,
    closest-hit records + per-ray box/triangle test counts for a ray set (primary rays of a small frame + random rays),
    rendered frames at trace limits 1, 2 and 5 with ray counters,
and one file of unit-function vectors (random + adversarial) with the verbatim functions' answers, and vs_reference.npz:
the outputs tests/test_oracle_vs_reference.py compares on its seeded soups and on the empty scene with spheres
(`--vs-reference-from-restatement` writes that file from oracle/liboracle.so where the reference is not available;
its `source` entry says which).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

import __graft_entry__ as ge  # noqa: E402
from oracle import bindings as ob  # noqa: E402

DATA = "/root/reference/data"
FMAX = np.float32(np.finfo(np.float32).max)


def adversarial_rays(rng, n):
    """Rays with axis-parallel / zero / inf / NaN direction components, tiny and huge t, origins on box faces."""
    r = ob.random_rays(n, seed=int(rng.integers(1 << 30)))
    k = n // 8
    r["d"][0:k, 0] = 0.0
    r["d"][k:2 * k, 1] = -0.0
    r["d"][2 * k:3 * k] = np.eye(3, dtype=np.float32)[rng.integers(0, 3, k)] * rng.choice([-1.0, 1.0], (k, 1)).astype(np.float32)
    r["d"][3 * k:3 * k + 4, 2] = np.inf
    r["d"][3 * k + 4:3 * k + 8, 0] = np.nan
    r["t"][4 * k:5 * k] = rng.uniform(0, 2, k).astype(np.float32)
    r["t"][5 * k:5 * k + 4] = 0.0
    r["o"][6 * k:7 * k] = np.round(r["o"][6 * k:7 * k] * 4) / 4  # many exact coordinates
    return r


def unit_vectors(R, rng):
    n = 4096
    rays = adversarial_rays(rng, n)
    lo = rng.uniform(-1, 0.5, (n, 3)).astype(np.float32)
    hi = (lo + rng.uniform(0, 1, (n, 3))).astype(np.float32)
    boxes = np.concatenate([lo, hi], 1)
    boxes[:64, 3:] = boxes[:64, :3]  # flat boxes
    rays["o"][64:128] = boxes[64:128, :3]  # origin on a corner
    rays["o"][128:192, 0] = boxes[128:192, 0]  # origin on a face
    ahit, at = R.ray_aabb(boxes, rays)

    tri = rng.uniform(-1, 1, (n, 3, 3)).astype(np.float32)
    nrm = rng.normal(size=(n, 3, 3)).astype(np.float32)
    tri[:32, 1] = tri[:32, 0]  # degenerate (NaN plane)
    tri[32:64, 2] = tri[32:64, 0] + 2 * (tri[32:64, 1] - tri[32:64, 0])  # collinear
    # aim half of the rays at the triangle so that hits are common
    tr = ob.random_rays(n, seed=3)
    tgt = (tri[:, 0] * 0.3 + tri[:, 1] * 0.3 + tri[:, 2] * 0.4)
    d = tgt - tr["o"]
    d /= np.maximum(np.linalg.norm(d, axis=1, keepdims=True), 1e-20)
    tr["d"][: n // 2] = d[: n // 2].astype(np.float32)
    tr["d"][n // 2:n // 2 + 64] = (tri[n // 2:n // 2 + 64, 1] - tr["o"][n // 2:n // 2 + 64])  # through a vertex, unnormalised
    tr["o"][n - 64:] = tri[n - 64:, 0]  # origin on a vertex (in-plane shortcut)
    tris18 = np.concatenate([tri.reshape(n, 9), nrm.reshape(n, 9)], 1)
    thit = R.ray_triangle(tris18, tr)

    planes = R.triangle_plane(tri.reshape(n, 9))
    phit, pt = R.ray_plane(planes, tr)
    pts = (tr["o"] + tr["d"] * np.where(np.isfinite(pt) & (pt < 1e30), pt, 0)[:, None]).astype(np.float32)
    pit_in = np.concatenate([tri.reshape(n, 9), planes[:, :3], pts], 1)
    pit = R.point_in_triangle(pit_in)

    sph = np.concatenate([rng.uniform(-1, 1, (n, 3)), rng.uniform(0.05, 1.0, (n, 1))], 1).astype(np.float32)
    st, sh, sn = R.ray_sphere(sph, rays)
    return dict(aabb_boxes=boxes, aabb_rays=rays, aabb_hit=ahit, aabb_t=at, tri_in=tris18, tri_rays=tr, tri_out=thit,
                planes=planes, plane_hit=phit, plane_t=pt, pit_in=pit_in, pit_out=pit, sph_in=sph, sph_t=st, sph_hit=sh, sph_n=sn)


def scene_fixture(R, capi, name, hs, frame, nrand, rng, lights=None, use_ctor=True):
    flat = ob.FlatScene(hs.vcount, hs.tcount, hs.vertices, hs.triangles, hs.materials, hs.spheres)
    lights = hs.lights if lights is None else np.asarray(lights, np.float32)
    rs = R.scene(flat, lights)
    b = rs.bvh(mode=0 if use_ctor else 1)
    meta, aabb = b.nodes()
    leaf_idx = np.nonzero(meta[:, 0])[0]
    leaf_tris = np.concatenate([b.leaf_triangles(i, meta[i, 4]) for i in leaf_idx]) if len(leaf_idx) else np.zeros(0, np.int32)
    W, H = frame
    cam = ob.default_camera(W, H)
    prim = R.generate_rays(cam, W, H)
    rnd = adversarial_rays(rng, nrand)
    # random rays scaled to the scene extent and half of them aimed at triangle centroids
    pos = flat.global_positions()
    cen = pos.mean(1)
    pick = cen[rng.integers(0, len(cen), nrand // 2)]
    d = pick - rnd["o"][: nrand // 2]
    d /= np.maximum(np.linalg.norm(d, axis=1, keepdims=True), 1e-20)
    rnd["d"][: nrand // 2] = d.astype(np.float32)
    rays = np.concatenate([prim, rnd])
    hits, counts = b.intersect(rays, counts=True)
    out = dict(vcount=flat.vcount, tcount=flat.tcount, vertices=flat.vertices, triangles=flat.triangles,
               materials=flat.materials, spheres=flat.spheres, lights=lights, node_meta=meta, node_aabb=aabb,
               leaf_tris=leaf_tris, num_levels=np.int32(b.num_levels()), frame=np.array([W, H], np.int32), rays=rays,
               hits=hits, counts=counts, builder_mode=np.int32(0 if use_ctor else 1))
    for L in (1, 2, 5):
        img, cnt = b.render(cam, W, H, trace_limit=L, duplicate_shading=True)
        out[f"img_L{L}"] = img
        out[f"cnt_L{L}"] = np.array([cnt[k] for k in ("primary", "primary_hit", "shadow", "bounce", "box_tests", "tri_tests")], np.uint64)
    print(f"  {name}: meshes={len(flat.vcount)} tris={flat.n_triangles} nodes={len(meta)} levels={b.num_levels()} "
          f"hits={(hits['tri'] >= 0).sum()}/{len(rays)} L2={dict(zip(('prim','hit','shadow','bounce'), out['cnt_L2'][:4].tolist()))}")
    return out


VS_REFERENCE_CASES = [(1, 1, 0.5, 4), (2, 1, 0.5, 5), (3, 1, 0.4, 6), (7, 3, 0.5, 7), (500, 1, 0.1, 8), (900, 40, 0.2, 9),
                      (2500, 2, 0.05, 10)]  # (triangles, meshes, scale, seed) of tests/test_oracle_vs_reference.py
VS_REFERENCE_LIGHTS = np.array([[0.0, 0.9, 0.0, 1, 1, 1], [-1, 1, -1, 0.5, 0.5, 0.5]], np.float32)
SPHERES_PRESET = [[3, -2, 10.2, 1, .8, .2, .2, 0, 0, 0, 1, 1], [-2, 2, 4, 2, .6, .8, .2, 0, 0, 0, 1, 1],
                  [0, 0, 6, .75, .2, .2, .8, 0, 0, 0, 1, 1]]  # src/scene.cpp:51-56


def vs_reference_inputs(ntri, nmesh, scale, seed):
    """scene and rays of one case of test_tree_hits_images (generated from seeds, not stored)"""
    flat = ob.random_soup(ntri, seed=seed, scale=scale, n_meshes=nmesh)
    rays = ob.random_rays(5000, seed=seed + 100)
    rays["t"][::7] = np.float32(0.7)
    return flat, rays


def empty_scene_inputs():
    """the Spheres preset without meshes and the rays of test_empty_scene_and_spheres"""
    empty = ob.FlatScene(np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros((0, 6)), np.zeros((0, 3)), np.zeros((0, 8)),
                         spheres=SPHERES_PRESET)
    rays = ob.random_rays(4000, seed=1)
    rays["o"][:, 2] -= 3
    return empty, rays


def vs_reference_vectors(R):
    """What tests/test_oracle_vs_reference.py compares: for every seeded soup the tree of the reference CONSTRUCTOR (mode 0),
    its leaf orders, closest hits + per-ray test counts of 5000 rays, the 64x48 frame at trace limit 3 and its ray counters;
    for the empty scene with the Spheres preset, t and n of 4000 rays."""
    out = {}
    for ntri, nmesh, scale, seed in VS_REFERENCE_CASES:
        flat, rays = vs_reference_inputs(ntri, nmesh, scale, seed)
        b = R.scene(flat, VS_REFERENCE_LIGHTS).bvh(mode=0)
        meta, aabb = b.nodes()
        leaves = np.nonzero(meta[:, 0])[0]
        hits, counts = b.intersect(rays, counts=True)
        img, cnt = b.render(ob.default_camera(64, 48), 64, 48, trace_limit=3, duplicate_shading=True)
        k = f"s{seed}_"
        out.update({k + "node_meta": meta, k + "node_aabb": aabb,
                    k + "leaf_tris": np.concatenate([b.leaf_triangles(i, meta[i, 4]) for i in leaves]),
                    k + "hits": hits, k + "counts": counts, k + "img_L3": img,
                    k + "cnt_L3": np.array([cnt[c] for c in ("primary", "primary_hit", "shadow", "bounce")], np.uint64)})
    empty, rays = empty_scene_inputs()
    h = R.scene(empty).bvh(mode=0).intersect(rays)
    out.update(empty_t=h["t"], empty_n=h["n"])
    return out


def write_vs_reference(R, source):
    np.savez_compressed(os.path.join(HERE, "vs_reference.npz"), source=np.array(source), **vs_reference_vectors(R))
    print(f"vs_reference.npz written ({source}), {os.path.getsize(os.path.join(HERE, 'vs_reference.npz')) / 1e6:.2f} MB")


def main():
    capi = ge.load_package().capi
    R = ob.RefLib()
    write_vs_reference(R, "reference")
    rng = np.random.default_rng(20261018)
    np.savez_compressed(os.path.join(HERE, "units.npz"), **unit_vectors(R, rng))
    print("units.npz written")
    scenes = {
        "triangle": (capi.load_preset("SingleTriangle", DATA), None),
        "cube": (capi.load_preset("Cube", DATA), None),
        "cornell": (capi.load_preset("CornellBox", DATA), None),
        "monkey": (capi.load_preset("Monkey", DATA), None),
        # C5: three lights (SURVEY.md §8(d))
        "dodge": (capi.load_obj(DATA + "/dodgeColorTest.obj", True), [[-1, 1, -1, 1, 1, 1], [1, -1, -1, 1, 1, 1], [1, 1, 1, 1, 1, 1]]),
    }
    for name, (hs, lights) in scenes.items():
        fx = scene_fixture(R, capi, name, hs, (96, 72), 2048, rng, lights)
        np.savez_compressed(os.path.join(HERE, f"scene_{name}.npz"), **fx)
    # a multi-mesh soup with leaves that hold several meshes, overlapping boxes, origins inside boxes
    soup = ob.random_soup(6000, seed=99, scale=0.15, n_meshes=70)
    class HS:  # noqa: E701
        pass
    hs = HS()
    hs.vcount, hs.tcount, hs.vertices, hs.triangles, hs.materials, hs.spheres = soup.vcount, soup.tcount, soup.vertices, soup.triangles, soup.materials, soup.spheres
    hs.lights = np.array([[0, 0.9, 0, 1, 1, 1], [-1, 1, -1, .5, .5, .5]], np.float32)
    fx = scene_fixture(R, capi, "soup70", hs, (64, 48), 4096, rng)
    np.savez_compressed(os.path.join(HERE, "scene_soup70.npz"), **fx)
    sz = sum(os.path.getsize(os.path.join(HERE, f)) for f in os.listdir(HERE) if f.endswith(".npz"))
    print(f"total fixture size {sz / 1e6:.2f} MB")


if __name__ == "__main__":
    if sys.argv[1:] == ["--vs-reference-from-restatement"]:
        # without the reference's sources: the restatement's outputs, which test_oracle_vs_reference checked bit-equal to
        # the reference's own on exactly these inputs while oracle/_ref was built
        write_vs_reference(ob.OracleLib(), "restatement, bit-identical to the reference on these inputs")
    else:
        main()
