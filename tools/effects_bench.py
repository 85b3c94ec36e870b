"""Anti-aliasing, motion blur and bloom for K views: K calls of cgrt_render_effects against one cgrt_render_effects_views, for
K = 1, 4 and 8. Both host forms are timed with the host clock around the synchronous call (output arrays allocated once, outside
the timing); the two forms alternate. The device form of the batched call is timed with device events on a stream of its own.
Each result line gives the median and the range over the repetitions, per view. Prints the GPU's name and power limit first.

    python tools/effects_bench.py [--reps 7] [--out DIR]

Shapes: C1 (Cornell 512x512, trace limit 2) and C3 (dragon stand-in 1920x1080, limit 5, light colour 2.5 so that bloom has
pixels over its threshold), with turntable cameras (yaw steps of 10 degrees).
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))  # golden scenes
import torch  # noqa: E402

import __graft_entry__ as ge  # noqa: E402
from conftest import load_golden  # noqa: E402

capi = ge.load_package().capi
KS = (1, 4, 8)
EFFECTS = {"blur": 2, "bloom": 4, "bloom+blur": 6, "aa": 1}


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def stats_of(ts):
    return dict(median=round(statistics.median(ts), 4), min=round(min(ts), 4), max=round(max(ts), 4))


def wall(fn):
    t = time.perf_counter()
    fn()
    return 1e3 * (time.perf_counter() - t)


def shape(name, flat, lights, W, H, L, reps, out):
    s = capi.Scene(flat, lights=lights)
    lib = capi.load_library()
    stream = torch.cuda.Stream()
    p = capi.render_params(W, H, L)
    st = capi.RenderStats()
    for K in KS:
        cams = [capi.make_camera(W, H, euler_deg=(20.0, 20.0 + 10.0 * k, 0.0)) for k in range(K)]
        arr = (capi.Camera * K)(*cams)
        one = np.ones((K, H, W, 3), np.float32)   # (touched: no page faults inside the timing)
        many = np.ones((K, H, W, 3), np.float32)
        dev = torch.empty(K * H * W * 3, dtype=torch.float32, device="cuda")
        for ename, e in EFFECTS.items():
            def singles():
                for v in range(K):
                    capi.check(lib.cgrt_render_effects(s.h, C.byref(cams[v]), C.byref(p), e, many[v].ctypes.data, None))

            def batched():
                capi.check(lib.cgrt_render_effects_views(s.h, arr, K, C.byref(p), e, one.ctypes.data, C.byref(st)))

            def device():
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream)
                capi.check(lib.cgrt_render_effects_views_device(s.h, arr, K, C.byref(p), e, C.c_void_p(dev.data_ptr()),
                                                                C.c_void_p(stream.cuda_stream)))
                b.record(stream)
                b.synchronize()
                return a.elapsed_time(b)

            for _ in range(2):  # warm-up: allocations, the wave tuner's first frames
                singles(), batched(), device()
            same = bool(np.array_equal(one.view(np.uint32), many.view(np.uint32)))
            ts, tb, td = [], [], []
            for _ in range(reps):
                ts.append(wall(singles) / K)
                tb.append(wall(batched) / K)
                td.append(device() / K)
            rec = dict(config=name, W=W, H=H, trace_limit=L, K=K, effects=ename, same_pixels=same, pipeline=int(st.pipeline),
                       launches=int(st.kernel_launches), effects_ms_per_view=stats_of(ts), effects_views_ms_per_view=stats_of(tb),
                       device_form_ms_per_view=stats_of(td))
            print(json.dumps(rec), flush=True)
            out.append(rec)
        del dev
    s.close()
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None, help="directory for effects_bench.json")
    a = ap.parse_args()
    if capi.device_count() < 1:
        raise SystemExit("effects_bench: no CUDA device (timings are GPU timings)")
    info = gpu_info()
    print("gpu:", info, flush=True)
    out = []
    g = load_golden("cornell")
    shape("C1 cornell", g.flat, g.lights, 512, 512, 2, a.reps, out)
    d = capi.dragon_standin()
    bright = np.array(d.lights, np.float32).copy()
    bright[:, 3:6] = 2.5
    shape("C3 dragon stand-in, bright lights", d, bright, 1920, 1080, 5, a.reps, out)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "effects_bench.json"), "w") as f:
            json.dump(dict(gpu=info, results=out), f, indent=1)


if __name__ == "__main__":
    main()
