#!/usr/bin/env python
"""bench.py — Mrays/s (primary + shadow + bounce) of the hot path on BASELINE.json's headline configuration.

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, sm_100a)
    python bench.py --impl reference --steps K --warmup W    # the reference's own CPU code (oracle/_ref) on the host cores

Workload (config.workload): C3 = dragon 1920x1080 Whitted render, 1 point light, 1 shadow ray per hit and light, trace
limit 5 (up to 4 mirror bounces), reference camera preset, reference-rule BVH (depth 12). data/dragon.obj is NOT part of the
reference checkout, so the scene is the named procedural stand-in of the same size (87 040 triangles, mirror material
assigned by the harness so that bounces exist) — said in `data`.

A step = one frame. `value` = logical rays of the frame (all ranks) / device time of the frame with the scene resident in HBM,
timed with CUDA events per step, L2 flushed between steps, max over ranks. `e2e` = the same through the host-buffer API:
camera + lights go host->device and the float framebuffer comes back to pinned host memory inside the timed region, one
synchronous call per frame (the kept renderRayTracing signature); `e2e_streaming` = the pipelined form, two frames in flight.
The line also carries `parity` (the GPU frame against the CPU reference's frame of the same configuration, rendered in this
run) and, for N > 1, `frame_equals_single_gpu`. The CPU legs read the scene from tests/golden/dragon_standin.npz and never
load the product library; their thread count is set explicitly (torchrun exports OMP_NUM_THREADS=1).
With N > 1 the frame is partitioned into interleaved tiles (strong scaling); the timed region includes the exchange: every
rank stores its pixels straight into rank 0's frame over NVLink peer memory and signals arrival with a flag
(CGRT_EXCHANGE=nccl selects the NCCL gather + de-interleave kernel instead).

The benchmark runs what __graft_entry__.build() left in the tree and writes nothing into an up-to-date tree (it may be
read-only); a build older than its sources is redone first where the tree can be written.
`--dump-outputs DIR` writes what the last timed frame delivered (DIR/frame.npy, DIR/ray_counts.npy): the inputs are fixed,
so two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # no __pycache__ next to the sources

import __graft_entry__ as ge  # noqa: E402

METRIC = "Mrays/s (primary+shadow+bounce)"
WIDTH, HEIGHT, TRACE_LIMIT = 1920, 1080, 5
CPU_BUDGET_S = 12.0  # cpu_baseline leg of our arm: the full frame is repeated until about this much CPU time has been spent
B_RAY, B_BOX, B_TRI = 48, 32, 48  # algorithmic bytes: ray in + hit out, per box test, per triangle test (SURVEY.md §8(d))
L2_PEAK_GBS = 20000.0  # order of magnitude of B200's L2 bandwidth (no measured figure in MEASURED_PEAKS.json): context for l2_frac only


# re-exported for tests/test_multirank_gloo.py
def _distributed():
    from importlib import import_module
    ge.load_package()
    return import_module("cg_raytracer_b200.distributed")


def pack_tiles(capi, params, frame):
    return _distributed().pack_tiles(capi, params, frame)


def assemble_on_host(capi, params, buffers):
    return _distributed().assemble_on_host(capi, params, buffers)


def gather_tiles(local, rank, world):
    return _distributed().gather_tiles(local, rank, world)


DATA = "synthetic (procedural dragon stand-in; data/dragon.obj is not in the reference checkout)"


def workload_name(n_tris):
    return (f"C3 dragon stand-in (procedural torus knot, {n_tris} triangles, mirror ks=0.5) {WIDTH}x{HEIGHT} Whitted: "
            f"1 point light, 1 shadow ray/hit/light, trace limit {TRACE_LIMIT} (<=4 mirror bounces), reference camera preset, "
            f"strict arithmetic (-fmad=false); every ray is SEARCHED in an 8-wide binned-SAH tree and CERTIFIED against the "
            f"reference-rule BVH (depth 12), results bit-identical to the reference traversal (config.exact_only_ms = the same "
            f"frame through the exact reference-order traversal alone)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "10"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def cpu_threads():
    """Host threads the CPU legs use: every core this process may run on. Passed explicitly to the renderer, so that
    torchrun's OMP_NUM_THREADS=1 (set for N > 1) does not turn the reference arm into a single-thread run."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def use_build(product=True):
    """Run what build() left: nothing is written into a tree that is up to date. A build older than its sources is redone
    (build_checkers() alone for the CPU legs, which never load the product library) when the tree can be written;
    a read-only tree is used as it is, with a warning."""
    if not ge.stale(product):
        return
    if not os.access(ROOT, os.W_OK):
        sys.stderr.write("bench.py: the built libraries are older than their sources and the tree is read-only: using them as built\n")
    elif product:
        ge.build()  # every rank: serialised by a file lock
    else:
        ge.build_checkers()


def cpu_checker():
    """oracle/_ref (the reference's own compiled TUs) when present, else the restatement. Test infrastructure: this is the
    only place besides tests/ and smoke() where bench.py touches oracle/. Never loads the product library."""
    use_build(product=False)
    from oracle import bindings as ob
    try:
        return ob.RefLib(), "reference", ob
    except (FileNotFoundError, OSError):
        return ob.OracleLib(), "port", ob


def cpu_scene():
    """The C3 stand-in on the CPU side: flat arrays from tests/golden/dragon_standin.npz (the product generator's output,
    committed as a fixture), BVH by range-based fill of the reference's own Node structs (its constructor needs ~25 GB)."""
    lib, kind, ob = cpu_checker()
    flat, lights = ob.dragon_standin_fixture()
    b = lib.scene(flat, lights).bvh(mode=1)
    return lib, kind, ob, flat, lights, b


def cpu_frames(b, ob, steps, warmup, budget_s=None):
    """Render the full WIDTH x HEIGHT frame on the host cores: `warmup` untimed frames, then `steps` timed ones (or, with
    budget_s, as many as fit in that much wall time, at least one). Returns (Mrays/s, threads, rays, seconds, frames, last
    frame, its counters)."""
    nt = cpu_threads()
    cam = ob.default_camera(WIDTH, HEIGHT)
    for _ in range(warmup):
        b.render(cam, WIDTH, HEIGHT, trace_limit=TRACE_LIMIT, duplicate_shading=True, nthreads=nt)
    rays, total, n, rgb, cnt = 0, 0.0, 0, None, None
    while (n < steps) if budget_s is None else (n < 1 or total < budget_s):
        t0 = time.perf_counter()
        rgb, cnt = b.render(cam, WIDTH, HEIGHT, trace_limit=TRACE_LIMIT, duplicate_shading=True, nthreads=nt)
        total += time.perf_counter() - t0
        rays += cnt["primary"] + cnt["shadow"] + cnt["bounce"]
        n += 1
    return rays / total / 1e6, nt, rays, total, n, rgb, cnt


def sample_text(frames):
    return (f"{frames} full {WIDTH}x{HEIGHT} frame(s) of the same scene, camera, lights and trace limit through the reference's own "
            f"code path incl. its duplicated shading() call (main.cpp:284), rays counted once, OpenMP static rows, "
            f"{cpu_threads()} threads set explicitly")


def frame_parity(rgb, counters, ref_rgb, ref_cnt):
    """GPU frame vs the CPU reference's frame of the same configuration (bench line `parity`)."""
    a = np.ascontiguousarray(rgb, np.float32).reshape(HEIGHT, WIDTH, 3)
    b = np.ascontiguousarray(ref_rgb, np.float32).reshape(HEIGHT, WIDTH, 3)
    keys = ("primary", "shadow", "bounce")
    return {"against": "CPU reference frame rendered in this run (cpu_baseline leg), full frame",
            "counters_equal": bool(all(int(counters[k]) == int(ref_cnt[k]) for k in keys)),
            "max_abs": float(np.abs(a - b).max()),
            "bit_equal_frac": float((a.view(np.uint32) == b.view(np.uint32)).all(axis=2).mean()),
            "tolerance": "max_abs <= 1/255, bit_equal_frac >= 0.999 (pow() in the specular term is the only inexact op)"}


def write_outputs(path, arrays):
    """DIR/<name>.npy for each array of the last timed step: `frame` = the float32 [HEIGHT, WIDTH, 3] frame the timed call
    leaves on rank 0 (24.9 MB), `ray_counts` = primary, primary_hit, shadow, bounce rays of that frame over all ranks (float64)."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


def run_reference(args):
    lib, kind, ob, flat, lights, b = cpu_scene()
    v, nt, rays, dt, n, rgb, cnt = cpu_frames(b, ob, args.steps, args.warmup)
    if args.dump_outputs:
        counts = np.array([cnt[k] for k in ("primary", "primary_hit", "shadow", "bounce")], np.float64)
        write_outputs(args.dump_outputs, {"frame": rgb, "ray_counts": counts})
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / max(n, 1) * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": DATA,
        "config": {"workload": workload_name(flat.n_triangles)},
        "cpu_baseline": {"value": v, "unit": "Mrays/s", "cores": nt, "kind": kind, "sample": sample_text(n)},
        "e2e": {"value": v, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed frame's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if rank == 0:  # the CPU arm runs on rank 0 alone; the other ranks exit without work. The product library is not loaded.
            run_reference(args)
        return
    use_build()

    import torch
    import torch.distributed as dist
    pkg = ge.load_package()
    capi = pkg.capi
    distributed = _distributed()

    if capi.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device visible — the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize(dev)

    # ---- scene (host build + upload: outside every timed region, like the reference's BVH construction at scene load)
    d = capi.dragon_standin()
    scene = capi.Scene(d, lights=d.lights, device=local_rank)
    cam = capi.make_camera(WIDTH, HEIGHT)
    R = distributed.TiledRenderer(scene, WIDTH, HEIGHT, TRACE_LIMIT, rank, world, local_rank,
                                  mode=os.environ.get("CGRT_EXCHANGE"))  # p2p (default) | nccl
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    # ---- untimed: warm-up, ray counts, reference test counts (algorithmic bytes), per-class kernel times
    for _ in range(args.warmup):
        R.render_device(cam)
    barrier()
    st_count = R.count_pass(cam)
    R.render_device(cam, flags=capi.RENDER_PROFILE_ALL)
    st_prof = scene.collect_stats()
    rays_local = st_count["primary"] + st_count["shadow"] + st_count["bounce"]
    dominant = int(np.argmax(st_prof["class_ms"]))
    cls_rays = [st_count["primary"], st_count["bounce"], st_count["shadow"]]
    alg_bytes_class = [B_RAY * cls_rays[c] + B_BOX * st_count["box_tests"][c] + B_TRI * st_count["tri_tests"][c] for c in range(3)]
    alg_bytes_frame_local = sum(alg_bytes_class)
    names = capi.class_names(st_prof)
    if names is capi.ROUND_CLASS_NAMES or names is capi.WAVE_CLASS_NAMES:
        # round pipeline: k_trace (class 2) searches every ray of the frame; persistent wavefront: k_wave (class 2) IS the frame
        alg_bytes_class = [0, 0, alg_bytes_frame_local]
    elif st_prof["class_launches"][1] == 0:  # path pipeline: k_paths traces the primary AND the bounce rays
        alg_bytes_class = [alg_bytes_class[0] + alg_bytes_class[1], 0, alg_bytes_class[2]]
    tot = torch.tensor([rays_local, st_count["primary"], st_count["shadow"], st_count["bounce"], alg_bytes_frame_local],
                       dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    rays_frame, n_primary, n_shadow, n_bounce, alg_bytes_frame = [float(x) for x in tot.tolist()]

    # the same frame through the exact reference-order traversal alone (no speculative search): reported next to the headline
    exact_only_ms = None
    if world == 1 and not os.environ.get("CGRT_BENCH_SKIP_EXACT"):
        ex = capi.Scene(d, lights=d.lights, device=local_rank, exact_only=True)
        ems = []
        for _ in range(4):
            _, est = ex.render(cam, WIDTH, HEIGHT, trace_limit=TRACE_LIMIT)
            ems.append(est["device_ms"])
        exact_only_ms = float(min(ems[1:]))
        ex.close()

    # ---- timed: K frames, CUDA events per frame on the launching stream, L2 flushed between frames (outside the events)
    sampler = ClockSampler(local_rank)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    dom_ms, dom_launches = 0.0, 0
    barrier()
    if rank == 0:
        sampler.start()
    for k in range(args.steps):
        flush.zero_()
        ev[k][0].record()
        frame = R.render_device(cam, flags=(1 << dominant))
        ev[k][1].record()
        st = scene.collect_stats()  # synchronises the frame; reads the dominant kernel's event times
        dom_ms += st["class_ms"][dominant]
        dom_launches += st["class_launches"][dominant]
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:  # copied now: the frame buffers are reused by the frames below
        counts = torch.tensor([st[k] for k in ("primary", "primary_hit", "shadow", "bounce")], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(counts, op=dist.ReduceOp.SUM)
        dump = {"frame": frame.cpu().numpy().reshape(HEIGHT, WIDTH, 3), "ray_counts": counts.cpu().numpy()} if rank == 0 else None
    total_ms = sum(a.elapsed_time(b) for a, b in ev)
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    value = rays_frame * args.steps / (total_ms * 1e-3) / 1e6
    launches_per_step = int(st["kernel_launches"]) + R.extra_launches_per_frame()
    timeouts = R.timeouts()

    # ---- end to end: host-buffer API, per-frame H2D of camera + lights, D2H of the float frame to pinned memory.
    # One GPU: the streaming form (cgrt_render_submit / cgrt_render_wait, two frames in flight: the copy of frame k overlaps
    # the kernels of frame k+1; all K frames are delivered before the clock stops). The synchronous call (cgrt_render, one
    # frame at a time) is the line's `e2e`; the streaming number is `e2e_streaming`. N > 1: synchronous frames on rank 0.
    streaming = world == 1 or R.mode == "p2p"
    e2e_mode = "streaming (cgrt_render_submit x K + cgrt_render_wait, 2 frames in flight)" if world == 1 else \
               ("streaming (two frames on rank 0, copy-out of frame k on a second stream while frame k+1 renders)" if streaming
                else "synchronous per frame (render, exchange, D2H, stream sync)")
    for _ in range(2):
        R.render_to_host(cam)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        R.render_to_host(cam)
    barrier()
    e2e_sync_s = time.perf_counter() - t0
    e2e_s = e2e_sync_s
    e2e_frames_equal = None
    if streaming:
        R.stream_to_host(cam, 3)
        barrier()
        t0 = time.perf_counter()
        last = R.stream_to_host(cam, args.steps)
        barrier()
        e2e_s = time.perf_counter() - t0
        last = last.copy() if rank == 0 else None
        ref_frame = R.render_to_host(cam)
        if rank == 0:  # reported, not asserted: a bench line with a failed check is more useful than no line
            e2e_frames_equal = bool(np.array_equal(last, ref_frame))
    t = torch.tensor([e2e_s, e2e_sync_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s, e2e_sync_s = [float(x) for x in t.tolist()]
    e2e_value = rays_frame * args.steps / e2e_s / 1e6
    e2e_sync_value = rays_frame * args.steps / e2e_sync_s / 1e6
    timeouts = max(timeouts, R.timeouts())

    # ---- untimed checks carried in the line: (i) N > 1: the frame the timed mode delivers on rank 0 == the frame rank 0 renders
    # alone on one GPU, bit for bit (SURVEY 8e); (ii) the frame against the CPU reference's frame of the same configuration
    gpu_frame = R.render_to_host(cam)
    gpu_frame = gpu_frame.copy() if rank == 0 else None
    frame_equals_single = None
    if world > 1:
        barrier()
        if rank == 0:
            single, _ = scene.render(cam, WIDTH, HEIGHT, trace_limit=TRACE_LIMIT)
            frame_equals_single = bool(np.array_equal(single.view(np.uint32), gpu_frame.view(np.uint32)))
        barrier()
    h2d = 128 + 32 * len(d.lights)  # FrameParams block + lights (cgrt_capi.cu: CGRT_PARAM_BLOCK_HEADER + 2 float4 per light)
    d2h = WIDTH * HEIGHT * 12

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")
        dom_name = names[dominant]
        dom_avg_s = dom_ms * 1e-3 / max(dom_launches, 1)
        # algorithmic bytes of the rays this rank's launches of the dominant kernel process, averaged per launch
        dom_bytes_per_launch = alg_bytes_class[dominant] / max(st_prof["class_launches"][dominant], 1) if dominant < 3 else 0.0
        achieved = dom_bytes_per_launch / dom_avg_s / 1e9 if dom_avg_s > 0 else 0.0
        traffic, counters = None, {}
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            counters = prof.get(dom_name, {})
            traffic = counters.get("dram_bytes_per_launch")
        except Exception:
            pass
        # what the kernel is really bound by (ncu --set full of this kernel on this frame, profiles/traffic.json): bytes it
        # requested from L2 / L1, the fraction of the issue slots it used, active threads per warp instruction
        sm_clock = (clocks or {}).get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0
        issue_peak = 148 * 4 * sm_clock * 1e6  # warp instructions per second: 148 SMs x 4 schedulers
        extras = {}
        if counters.get("warp_inst_per_launch") and dom_avg_s > 0:
            extras["issue_frac"] = counters["warp_inst_per_launch"] / dom_avg_s / issue_peak
            extras["warp_inst_per_ray"] = counters["warp_inst_per_launch"] / max(rays_frame / max(st_prof["class_launches"][dominant], 1), 1)
        if counters.get("l2_bytes_per_launch") and dom_avg_s > 0:
            extras["requested_bytes_per_launch"] = {"lts__t_bytes": counters["l2_bytes_per_launch"], "l1tex__t_bytes": counters.get("l1_bytes_per_launch")}
            extras["l2_frac"] = counters["l2_bytes_per_launch"] / dom_avg_s / 1e9 / L2_PEAK_GBS
        if counters.get("threads_per_warp_inst"):
            extras["threads_per_warp_inst"] = counters["threads_per_warp_inst"]
        extras["counters_source"] = counters.get("source")
        line = {
            "metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic (procedural dragon stand-in; data/dragon.obj is not in the reference checkout)",
            "config": {"workload": workload_name(d.n_triangles), "l2": "flushed between timed frames (256 MiB memset outside the event pair)",
                       "parallelism": f"tiles{world}" if world > 1 else "single", "tile": "8x8 interleaved, row skew 3, centre-out order",
                       "exchange": {"single": "none", "p2p": "direct stores into rank 0's frame over NVLink peer memory + arrival/consumed flags",
                                    "nccl": "NCCL gather of tile-major buffers + assemble kernel"}[R.mode],
                       "exchange_fallback_reason": R.fallback_reason, "handoff_timeouts": timeouts, "e2e_mode": e2e_mode, "e2e_streamed_frame_equals_synchronous_frame": e2e_frames_equal,
                       "frame_equals_single_gpu": frame_equals_single,
                       "rays_per_frame": {"primary": n_primary, "shadow": n_shadow, "bounce": n_bounce}, "exact_only_ms": exact_only_ms,
                       "pipeline": {0: "counting", 1: "path pipeline", 2: "round pipeline", 3: "persistent wavefront (k_wave)"}.get(st_prof.get("pipeline")),
                       "kernel_ms_per_frame_rank0": dict(zip(names, [round(v, 4) for v in st_prof["class_ms"]])),
                       "kernel_launches_per_frame": dict(zip(names, st_prof["class_launches"])),
                       "frame_roofline": {"algorithmic_bytes_per_frame": alg_bytes_frame, "bytes_per_ray": alg_bytes_frame / rays_frame,
                                          "achieved_GBps": alg_bytes_frame * args.steps / (total_ms * 1e-3) / 1e9,
                                          "frac_of_hbm_peak": alg_bytes_frame * args.steps / (total_ms * 1e-3) / 1e9 / (peak * world)}},
            # e2e = the kept synchronous call (one cgrt_render per frame: what the renderRayTracing shim of INTEGRATION.md makes);
            # e2e_streaming = the pipelined form (two frames in flight) next to it
            "e2e": {"value": e2e_sync_value, "unit": "Mrays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_sync_s / args.steps * 1e3, "mode": "synchronous: render, exchange, D2H to pinned host memory, stream sync per frame"},
            "e2e_streaming": {"value": e2e_value, "unit": "Mrays/s", "ms_per_step": e2e_s / args.steps * 1e3, "mode": e2e_mode},
            "frame_equals_single_gpu": frame_equals_single,
            "gpu_launches": launches_per_step * args.steps,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": dom_bytes_per_launch, "avg_launch_ms": dom_avg_s * 1e3,
                         "launches_timed": dom_launches, "exact_only_ms": exact_only_ms, **extras,
                         "note": "algorithmic bytes = the box / triangle tests the REFERENCE traversal performs for these rays (counting "
                                 "pass, SURVEY 8d); the speculative search performs far fewer and the scene (~20 MB) is L2-resident, so "
                                 "frac can exceed 1 and DRAM traffic is far lower: the HBM roofline is the contractual denominator. The "
                                 "physical bound is instruction issue: issue_frac = warp instructions / (148 SMs x 4 schedulers x clock x "
                                 "time), at threads_per_warp_inst of 32 lanes (ncu, profiles/); l2_frac is against a nominal 20 TB/s"},
        }
        if timeouts:
            line["invalid"] = f"{timeouts} exchange hand-off wait(s) timed out: frames may be incomplete"
        if world == 1 and not args.no_cpu_baseline:
            lib, kind, ob, cflat, clights, b = cpu_scene()
            fixture_ok = bool(np.array_equal(cflat.vertices.view(np.uint32), np.ascontiguousarray(d.vertices, np.float32).reshape(-1, 6).view(np.uint32))
                              and np.array_equal(cflat.triangles, np.ascontiguousarray(d.triangles, np.uint32).reshape(-1, 3)))
            v, cores, rays, secs, n, ref_rgb, ref_cnt = cpu_frames(b, ob, 0, 1, budget_s=CPU_BUDGET_S)
            line["cpu_baseline"] = {"value": v, "unit": "Mrays/s", "cores": cores, "kind": kind, "sample": sample_text(n),
                                    "sample_rays": rays, "sample_seconds": secs}
            line["parity"] = frame_parity(gpu_frame, {"primary": n_primary, "shadow": n_shadow, "bounce": n_bounce}, ref_rgb, ref_cnt)
            line["parity"]["cpu_scene_equals_gpu_scene"] = fixture_ok
        if args.dump_outputs:
            write_outputs(args.dump_outputs, dump)
        print(json.dumps(line))
    if world > 1:
        dist.barrier(device_ids=[local_rank])
        R.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
