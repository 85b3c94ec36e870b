"""Per-view device time of K camera views of one scene: rendered one by one (cgrt_render_device per view, all on one stream)
against one cgrt_render_views_device call. Device events around each sequence; the two forms alternate, and each result line
gives the median and the range over the repetitions, divided by K. Prints the GPU's name and power limit first.

    python tools/views_bench.py [--reps 7] [--out DIR]

Shapes: C1 (Cornell 512x512, trace limit 2), C2 (monkey 1920x1080, limit 1), C3 (dragon stand-in 1920x1080, limit 5) with
turntable cameras (yaw steps of 10 degrees), and C3 with the 15 motion-blur cameras of cgrt_render_effects (look-at (0.01 k, 0, 0)).
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
KS = (1, 2, 4, 8, 15)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def turntable(W, H, K):
    return [capi.make_camera(W, H, euler_deg=(20.0, 20.0 + 10.0 * k, 0.0)) for k in range(K)]


def blur(W, H, K):
    return [capi.make_camera(W, H, look_at=(0.01 * k, 0.0, 0.0)) for k in range(1, K + 1)]


def timed(fn, stream):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    fn()
    b.record(stream)
    b.synchronize()
    return a.elapsed_time(b)


def shape(name, flat, lights, W, H, L, make_cams, reps, out):
    s = capi.Scene(flat, lights=lights)
    stream = torch.cuda.Stream()
    sp = stream.cuda_stream
    p = capi.render_params(W, H, L)
    px = W * H * 3
    for K in KS:
        cams = make_cams(W, H, K)
        one = torch.empty(K * px, dtype=torch.float32, device="cuda")
        batch = torch.empty(K * px, dtype=torch.float32, device="cuda")

        def one_by_one():
            for v, cam in enumerate(cams):
                s.render_device(cam, p, one.data_ptr() + v * px * 4, sp)

        def together():
            s.render_views_device(cams, p, batch.data_ptr(), sp)

        for _ in range(2):  # warm-up: allocations, the wave tuner's first frames
            timed(one_by_one, stream)
            timed(together, stream)
        st = s.collect_stats()
        same = bool(torch.equal(one.view(torch.int32), batch.view(torch.int32)))
        t1, tb = [], []
        for _ in range(reps):
            t1.append(timed(one_by_one, stream) / K)
            tb.append(timed(together, stream) / K)
        rec = dict(config=name, W=W, H=H, trace_limit=L, K=K, pipeline_batch=st["pipeline"], same_pixels=same,
                   one_by_one_ms_per_view=dict(median=round(statistics.median(t1), 4), min=round(min(t1), 4), max=round(max(t1), 4)),
                   batched_ms_per_view=dict(median=round(statistics.median(tb), 4), min=round(min(tb), 4), max=round(max(tb), 4)),
                   speedup=round(statistics.median(t1) / statistics.median(tb), 3))
        print(json.dumps(rec), flush=True)
        out.append(rec)
        del one, batch
    s.close()
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None, help="directory for views_bench.json")
    a = ap.parse_args()
    if capi.device_count() < 1:
        raise SystemExit("views_bench: no CUDA device (timings are device timings)")
    info = gpu_info()
    print("gpu:", info, flush=True)
    out = []
    g = load_golden("cornell")
    shape("C1 cornell", g.flat, g.lights, 512, 512, 2, turntable, a.reps, out)
    g = load_golden("monkey")
    shape("C2 monkey", g.flat, g.lights, 1920, 1080, 1, turntable, a.reps, out)
    d = capi.dragon_standin()
    shape("C3 dragon stand-in", d, d.lights, 1920, 1080, 5, turntable, a.reps, out)
    shape("C3 motion-blur cameras", d, d.lights, 1920, 1080, 5, blur, a.reps, out)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "views_bench.json"), "w") as f:
            json.dump(dict(gpu=info, results=out), f, indent=1)


if __name__ == "__main__":
    main()
