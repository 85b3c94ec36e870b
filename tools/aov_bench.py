"""Device time of a frame with and without its per-pixel buffers: cgrt_render_views_device against cgrt_render_aovs_device with
all four buffers (depth, tri, normal, hits), for K = 1 and K = 8 views. Device events around each call; the two forms alternate,
and each result line gives the median and the range over the repetitions, per frame (one view). Prints the GPU's name and power
limit first.

    python tools/aov_bench.py [--reps 15] [--out DIR]

Shapes: C1 (Cornell 512x512, trace limit 2), C2 (monkey 1920x1080, limit 1), C3 (dragon stand-in 1920x1080, limit 5), with
turntable cameras (yaw steps of 10 degrees).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))  # golden scenes
import torch  # noqa: E402

import __graft_entry__ as ge  # noqa: E402
from conftest import load_golden  # noqa: E402

capi = ge.load_package().capi
KS = (1, 8)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def timed(fn, stream):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    fn()
    b.record(stream)
    b.synchronize()
    return a.elapsed_time(b)


def stats_of(ts):
    return dict(median=round(statistics.median(ts), 4), min=round(min(ts), 4), max=round(max(ts), 4))


def shape(name, flat, lights, W, H, L, reps, out):
    s = capi.Scene(flat, lights=lights)
    stream = torch.cuda.Stream()
    sp = stream.cuda_stream
    p = capi.render_params(W, H, L)
    for K in KS:
        cams = [capi.make_camera(W, H, euler_deg=(20.0, 20.0 + 10.0 * k, 0.0)) for k in range(K)]
        px = K * W * H
        rgb_v = torch.empty(px * 3, dtype=torch.float32, device="cuda")
        rgb_a = torch.empty(px * 3, dtype=torch.float32, device="cuda")
        aov = dict(depth=torch.empty(px, dtype=torch.float32, device="cuda"), tri=torch.empty(px, dtype=torch.int32, device="cuda"),
                   normal=torch.empty(px * 3, dtype=torch.float32, device="cuda"),
                   hits=torch.empty(px, dtype=torch.uint8, device="cuda"))
        ptrs = {k: v.data_ptr() for k, v in aov.items()}

        def views():
            s.render_views_device(cams, p, rgb_v.data_ptr(), sp)

        def aovs():
            s.render_aovs_device(cams, p, rgb_a.data_ptr(), ptrs, sp)

        for _ in range(3):  # warm-up: allocations, the wave tuner's first frames
            timed(views, stream)
            timed(aovs, stream)
        st = s.collect_stats()
        same = bool(torch.equal(rgb_v.view(torch.int32), rgb_a.view(torch.int32)))
        tv, ta = [], []
        for _ in range(reps):
            tv.append(timed(views, stream) / K)
            ta.append(timed(aovs, stream) / K)
        rec = dict(config=name, W=W, H=H, trace_limit=L, K=K, pipeline=st["pipeline"], same_pixels=same,
                   views_ms_per_frame=stats_of(tv), aovs_ms_per_frame=stats_of(ta),
                   aov_cost_ms_per_frame=round(statistics.median(ta) - statistics.median(tv), 4),
                   aov_cost_pct=round(100.0 * (statistics.median(ta) / statistics.median(tv) - 1.0), 2))
        print(json.dumps(rec), flush=True)
        out.append(rec)
        del rgb_v, rgb_a, aov
    s.close()
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--out", default=None, help="directory for aov_bench.json")
    a = ap.parse_args()
    if capi.device_count() < 1:
        raise SystemExit("aov_bench: no CUDA device (timings are device timings)")
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
        with open(os.path.join(a.out, "aov_bench.json"), "w") as f:
            json.dump(dict(gpu=info, results=out), f, indent=1)


if __name__ == "__main__":
    main()
