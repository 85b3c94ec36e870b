"""Device time of a frame with and without its mirror-path buffers: cgrt_render_views_device against cgrt_render_paths_device with
every buffer (ray, depth, tri, normal, position, visibility) and n_levels = the trace limit, for K = 1 and K = 8 views. Device
events around each call; the two forms alternate, and each result line gives the median and the range over the repetitions, per
frame (one view). Prints the GPU's name and power limit first.

    python tools/path_bench.py [--reps 15] [--out DIR]

Shapes: C1 (Cornell 512x512, 1 light, trace limit 2), C2 (monkey 1920x1080, 2 lights, limit 1), C3 (dragon stand-in 1920x1080,
1 light, limit 5), with turntable cameras (yaw steps of 10 degrees). The pass stores 64 + 4 x lights bytes per pixel and level
(ray 32, depth 4, tri 4, normal 12, position 12, visibility 4 per light); `store_gb_per_frame` is that figure for one view.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))  # golden scenes
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402

import __graft_entry__ as ge  # noqa: E402
from aov_bench import gpu_info, stats_of, timed  # noqa: E402
from conftest import load_golden  # noqa: E402

capi = ge.load_package().capi
KS = (1, 8)
# bytes per pixel and level of each buffer (visibility: per light)
BYTES = dict(ray=32, depth=4, tri=4, normal=12, position=12, visibility=4)


def shape(name, flat, lights, W, H, L, reps, out):
    s = capi.Scene(flat, lights=lights)
    n = len(lights)
    stream = torch.cuda.Stream()
    sp = stream.cuda_stream
    p = capi.render_params(W, H, L)
    for K in KS:
        cams = [capi.make_camera(W, H, euler_deg=(20.0, 20.0 + 10.0 * k, 0.0)) for k in range(K)]
        px = K * W * H
        rgb_v = torch.empty(px * 3, dtype=torch.float32, device="cuda")
        rgb_p = torch.empty(px * 3, dtype=torch.float32, device="cuda")
        bufs = {k: torch.empty(L * px * b * (n if k == "visibility" else 1), dtype=torch.uint8, device="cuda")
                for k, b in BYTES.items()}
        ptrs = {k: v.data_ptr() for k, v in bufs.items()}

        def views():
            s.render_views_device(cams, p, rgb_v.data_ptr(), sp)

        def paths():
            s.render_paths_device(cams, p, L, rgb_p.data_ptr(), ptrs, sp)

        fns = [("views", views), ("paths", paths)]
        for _ in range(3):  # warm-up: allocations, the wave tuner's first frames
            for _, fn in fns:
                timed(fn, stream)
        st = s.collect_stats()
        same = bool(torch.equal(rgb_v.view(torch.int32), rgb_p.view(torch.int32)))
        ts = {c: [] for c, _ in fns}
        for _ in range(reps):
            for c, fn in fns:
                ts[c].append(timed(fn, stream) / K)
        base, m = statistics.median(ts["views"]), statistics.median(ts["paths"])
        store = sum(b * (n if k == "visibility" else 1) for k, b in BYTES.items()) * L * W * H
        rec = dict(config=name, W=W, H=H, trace_limit=L, lights=n, K=K, pipeline=st["pipeline"], same_pixels=same,
                   views_ms_per_frame=stats_of(ts["views"]), paths_ms_per_frame=stats_of(ts["paths"]),
                   cost_ms_per_frame=round(m - base, 4), cost_pct=round(100.0 * (m / base - 1.0), 2),
                   store_gb_per_frame=round(store / 1e9, 4))
        print(json.dumps(rec), flush=True)
        out.append(rec)
        del rgb_v, rgb_p, bufs
    s.close()
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--out", default=None, help="directory for path_bench.json")
    a = ap.parse_args()
    if capi.device_count() < 1:
        raise SystemExit("path_bench: no CUDA device (timings are device timings)")
    info = gpu_info()
    print("gpu:", info, flush=True)
    out = []
    g = load_golden("cornell")
    shape("C1 cornell", g.flat, g.lights, 512, 512, 2, a.reps, out)
    g = load_golden("monkey")
    shape("C2 monkey", g.flat, g.lights, 1920, 1080, 1, a.reps, out)
    d = capi.dragon_standin()
    shape("C3 dragon stand-in", d, d.lights, 1920, 1080, 5, a.reps, out)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "path_bench.json"), "w") as f:
            json.dump(dict(gpu=info, results=out), f, indent=1)


if __name__ == "__main__":
    main()
