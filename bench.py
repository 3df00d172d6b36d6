#!/usr/bin/env python
"""bench.py — headline benchmark of the path-tracing hot path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload C2] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one full render of the workload (default BASELINE.json configs[1]: Cornell box
1024x1024 @ 1024 spp, emissive quad light + mixture-PDF light sampling, adaptive sampling off).
Rank 0 prints ONE JSON line (contract in the task statement):

  value     Mpaths/s, whole job, scene resident in HBM, device-timed (CUDA events, max over ranks)
  e2e       same metric through the public API with HOST buffers: SceneData flatten + BVH build +
            H2D upload + render + framebuffer gather + D2H, wall clock, every step
  roofline  FP32-pipe roofline of the render kernel: algorithmic flops (SURVEY.md §8d model, event
            counts from the CPU oracle on a bounded sample) / CUDA-event time, against the FP32 FMA
            peak measured in this run (MEASURED_PEAKS.json has no FP32 figure); HBM traffic beside it
  cpu_baseline  the C++ restatement of the reference (oracle/, kind "port": the TypeScript reference
            cannot run here) on the box's host cores, parallelised like the reference's worker
            threads (row strips, nproc-1 threads), on a bounded sample

`--impl reference` times that CPU port alone, on the same workload/metric (rank 0 only).
`--dump-outputs DIR` writes the image and statistics of the last timed step as .npy files (dump_outputs): the
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree (it may be read-only)

WORKLOADS = {
    # BASELINE.json configs (SURVEY.md §8d for the concrete inputs)
    "C1": ("spheres-scene 400x225 @16spp depth 10 (BASELINE configs[0])", "spheres", {"count": 100, "seed": 12345},
           {"width": 400, "samples": 16, "depth": 10, "aTolerance": 0}),
    "C2": ("cornell-scene 1024x1024 @1024spp, quad light + PDF light sampling (BASELINE configs[1])", "cornell", {},
           {"width": 1024, "samples": 1024, "aTolerance": 0}),
    "C3": ("weekend-final ~480 spheres 1920x1080 @512spp (BASELINE configs[2])", "weekend", {"seed": 1},
           {"width": 1920, "samples": 512, "aTolerance": 0}),
    "C4": ("rain-scene 100k spheres 3840x2160 @64spp (BASELINE configs[3])", "rain", {"count": 100000, "seed": 1, "sphereRadius": 0.01},
           {"width": 3840, "samples": 64, "aTolerance": 0}),
    "C5": ("layered/mixed-material scene 2048x2048 @256spp (BASELINE configs[4])", "layered", {},
           {"width": 2048, "samples": 256, "aTolerance": 0}),
    # what `benchmark.ts --rain 100000` renders: the generator's default radius 0.05 exceeds the cell spacing, so
    # the spheres overlap massively (SURVEY.md §8d); reported next to C4, not a BASELINE config of its own
    "C4r": ("rain-scene 100k spheres, default radius 0.05, 3840x2160 @64spp", "rain", {"count": 100000, "seed": 1},
            {"width": 3840, "samples": 64, "aTolerance": 0}),
}


def make_scene(kind, options):
    from mcp_raytracer_b200 import scenes

    return {
        "spheres": scenes.generateSpheresSceneData, "cornell": scenes.generateCornellSceneData,
        "weekend": scenes.generateWeekendFinalSceneData, "rain": scenes.generateRainSceneData,
        "layered": scenes.generateLayeredMixedSceneData,
    }[kind](options)


# ------------------------------------------------------------------------------------------
# algorithmic work model — SURVEY.md §8(d): flops the REFERENCE algorithm spends, with event
# counts taken from the oracle walking the reference's own BVH topology.
# ------------------------------------------------------------------------------------------
def shading_flops(cnt, n_lights, aperture):
    """The per-path part of the model: everything except the closest-hit queries."""
    lambert = 110 if n_lights == 0 else 200 + 90 * (n_lights - 1)
    return ((31 + (25 if aperture > 0 else 0)) * cnt["paths"] + 8 * cnt["rr"] + 24 * cnt["background"] + lambert * cnt["lambert"]
            + 62 * cnt["metal"] + 35 * cnt["metal_fuzz0"] + 60 * cnt["dielectric"] + 6 * cnt["hits"])


def algorithmic_flops(cnt, n_lights, aperture):
    ray = (21 * cnt["box_tests"] + 23 * cnt["sphere_miss"] + 52 * cnt["sphere_hit"] + 16 * cnt["planar_treject"]
           + 57 * cnt["quad_outside"] + 72 * cnt["quad_hit"] + 28 * cnt["plane_hit"])
    return ray + shading_flops(cnt, n_lights, aperture)


def executed_events(workload, ropts, spp):
    """Node visits and primitive tests the DEVICE executes on its own tree, counted by the instrumented build of the library
    (csrc/libmcprt_b200_count.so, -DRT_COUNT_EVENTS) in a process of its own: one render at `spp` samples, never timed.
    None when that build is absent."""
    lib = os.path.join(ROOT, "mcp_raytracer_b200", "csrc", "libmcprt_b200_count.so")
    if not os.path.exists(lib):
        return None
    code = (
        "import json, sys, numpy as np\n"
        f"sys.path.insert(0, {ROOT!r})\n"
        "import bench\n"
        "from mcp_raytracer_b200 import createCameraFromSceneData, _native\n"
        f"label, kind, sopts, ro = bench.WORKLOADS[{workload!r}]\n"
        f"ro = dict(ro, **{json.dumps({k: v for k, v in ropts.items()})}, samples={int(spp)}, integrator='megakernel')\n"
        "assert _native.lib().rt_counts_events() == 1\n"
        "sd = bench.make_scene(kind, sopts)\n"
        "with createCameraFromSceneData(sd, ro) as cam:\n"
        "    st = cam.render(np.zeros(cam.imageWidth * cam.imageHeight * 3, np.uint8))\n"
        "print(json.dumps({'paths': st.samples['total'], 'rays': st.rays, 'node_visits': st.nodeVisits, 'prim_tests': st.primTests}))\n"
    )
    try:
        r = subprocess.run([sys.executable, "-B", "-c", code], env=dict(os.environ, RT_B200_LIB=lib), capture_output=True, text=True, timeout=600)
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception:
        return None


ORACLE_BUILD = None
ORACLE_BUILD_DIR = None  # temporary directory of the host-tuned oracle build, removed when the process ends


def cpu_reference_run(sd, opts, target_seconds, threads):
    """Times the oracle on a BOUNDED sample of the workload that lasts about `target_seconds`: the same
    scene and camera, first at a reduced spp (adaptive sampling is off, so cost is linear in spp) and,
    if even 4 spp of the full image would take too long, at a reduced resolution as well (same field of
    view, so the mix of paths is the same).  The size is chosen from a small calibration render, which
    keeps the whole call bounded even where the reference's own BVH is nearly useless (its per-axis box
    test, aabb.ts:30-59, accepts most boxes along a long ray: 100k-sphere rain scene)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_binding
    from oracle_binding import OracleCamera

    global ORACLE_BUILD, ORACLE_BUILD_DIR
    if ORACLE_BUILD is None:  # first use: the host-tuned build (-O3 -march=native, made on this host), else the portable one
        native = None
        if not os.environ.get("RT_ORACLE_LIB"):
            ORACLE_BUILD_DIR = tempfile.TemporaryDirectory(prefix="rt_oracle_")  # never into the tree: it may be read-only
            native = oracle_binding.build_native_oracle(ORACLE_BUILD_DIR.name)
        if native:
            os.environ["RT_ORACLE_LIB"] = native
        ORACLE_BUILD = "-O3 -march=native, built on this host" if (native or os.environ.get("RT_ORACLE_LIB")) else "-O3 (portable build)"
    base = dict(opts)
    full_w, full_spp = int(base["width"]), int(base["samples"])
    # calibration: grow a tiny render until it takes >= 0.2 s (or a hard cap of work is reached)
    cal_w, cal_spp, per_path, ratio = min(full_w, 32), 1, None, 1.0
    for _ in range(8):
        cam = OracleCamera(sd, dict(base, width=cal_w, samples=cal_spp))
        t0 = time.perf_counter()
        r = cam.render(threads=threads)
        dt = max(time.perf_counter() - t0, 1e-5)
        ratio = cam.imageHeight / cam.imageWidth
        per_path = dt / max(1, r["stats"].samples_total)
        if dt >= 0.2 or (cal_w >= full_w and cal_spp >= full_spp):
            break
        if cal_w < min(full_w, 256):
            cal_w = min(full_w, cal_w * 2)
        else:
            cal_spp = min(full_spp, cal_spp * 4)
    budget_paths = target_seconds / per_path
    full_pixels = full_w * max(1, round(full_w * ratio))
    min_spp = min(full_spp, 4)
    if budget_paths >= full_pixels * min_spp:
        width, spp = full_w, int(max(min_spp, min(full_spp, budget_paths / full_pixels)))
    else:
        spp = min_spp
        width = int(max(16, min(full_w, (budget_paths / (spp * ratio)) ** 0.5)))
    cam = OracleCamera(sd, dict(base, width=width, samples=spp))
    t0 = time.perf_counter()
    r = cam.render(threads=threads, want_counters=True)
    dt = time.perf_counter() - t0
    st = r["stats"]
    return {
        "seconds": dt, "spp": spp, "paths": int(st.samples_total), "rays": int(st.rays), "counters": r["counters"],
        "n_lights": cam.n_lights, "width": cam.imageWidth, "height": cam.imageHeight,
        "mpaths_per_s": st.samples_total / dt / 1e6, "grays_per_s": st.rays / dt / 1e9,
        "sample": f"{cam.imageWidth}x{cam.imageHeight} @{spp}spp, same scene and camera (full config: {full_w} wide @{full_spp}spp; adaptive off)",
    }


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(gpu_index)],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def measured_traffic(workload, world, overridden):
    """dram__bytes_read.sum + dram__bytes_write.sum of the render kernel, per launch, from the committed
    `ncu --set full` capture of this command (profiles/r02_bench_traffic.json); None when the run is not that one."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_bench_traffic.json")))
    except Exception:
        return None
    if overridden or t.get("workload") != workload or t.get("n_gpus") != world:
        return None
    return t.get("dram_bytes_total")


DUMP_BYTES = 64_000_000  # what --dump-outputs may write in all, shared by the workloads of the run


def dump_outputs(out_dir, workload, rgb8, stats, budget):
    """Writes DIR/<workload>_<name>.npy: `image`, the RGB8 framebuffer (H, W, 3) as float32, and `stats`, float64
    [pixels, samples_total, samples_min, samples_max, bounces_total, bounces_min, bounces_max, rays] (rt_stats order).
    An image whose float32 copy does not fit `budget` is stored as `image_sample` (n, 3) float32 of the pixels at
    `image_sample_index` (flat y * W + x, ascending, float64), drawn with a fixed seed: the same pixels on every run."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    path = lambda name: os.path.join(out_dir, f"{workload}_{name}.npy")  # noqa: E731
    budget -= 4096  # the stats array and the .npy headers
    pixels = rgb8.reshape(-1, 3)
    if pixels.size * 4 <= budget:
        np.save(path("image"), rgb8.astype(np.float32))
    else:
        idx = np.sort(np.random.default_rng(0).choice(len(pixels), budget // (3 * 4 + 8), replace=False))
        np.save(path("image_sample"), pixels[idx].astype(np.float32))
        np.save(path("image_sample_index"), idx.astype(np.float64))
    np.save(path("stats"), np.asarray(stats, np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C2", help="one of %s, or a comma-separated list (one JSON line each)" % ", ".join(WORKLOADS))
    ap.add_argument("--samples", type=int, default=None, help="override spp (development only; the default is the BASELINE config)")
    ap.add_argument("--width", type=int, default=None, help="override width (development only)")
    ap.add_argument("--bvh", default="auto")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target duration of the CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-threads", type=int, default=None,
                    help="threads of the CPU port (default: host cores - 1 like the reference; 1 = the scalar figure SURVEY 8d asks for)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed to DIR/<workload>_<name>.npy "
                         "(the image as float32, the render statistics as float64), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200: the reference arm sizes its sample from its own timings, so its output varies")
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # `python bench.py --gpus N` without a launcher: become the one-process-per-GPU job the contract describes
        port = 29500 + os.getpid() % 2000
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                                   "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:])
    # stdout carries exactly ONE JSON line: libraries that chat on fd 1 (NCCL prints its version there)
    # are sent to stderr for the duration of the run.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    env = {"group": False}
    rc = 0
    for wl in args.workload.split(","):  # one JSON line per workload (the default, C2, prints exactly one)
        rc |= bench_workload(args, wl, rank, world, local_rank, emit, env)
    if env["group"]:
        import torch.distributed as dist

        dist.destroy_process_group()
    return rc


def bench_workload(args, workload, rank, world, local_rank, emit, env):
    label, kind, scene_opts, ropts = WORKLOADS[workload]
    ropts = dict(ropts)
    overridden = False
    if args.samples:
        ropts["samples"] = args.samples; overridden = True
    if args.width:
        ropts["width"] = args.width; overridden = True
    ropts["bvh"] = args.bvh
    cpu_threads = max(1, (os.cpu_count() or 2) - 1)  # os.cpus().length - 1, src/raytracer.ts:61
    if args.cpu_threads:
        cpu_threads = max(1, args.cpu_threads)

    # ---------------------------------------------------------------- reference arm (CPU port)
    if args.impl == "reference":
        if rank != 0:
            return 0
        sd = make_scene(kind, scene_opts)
        vals, last = [], None
        for i in range(args.warmup + args.steps):
            last = cpu_reference_run(sd, ropts, target_seconds=max(2.0, min(args.cpu_seconds, 60.0 / max(1, args.warmup + args.steps))), threads=cpu_threads)
            if i >= args.warmup:
                vals.append(last)
        v = sum(x["paths"] for x in vals) / sum(x["seconds"] for x in vals) / 1e6
        sample = last["sample"]
        line = {
            "impl": "reference", "metric": "Mpaths/s", "value": v, "unit": "Mpaths/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sum(x["seconds"] for x in vals) / len(vals), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32-store/f64-scalar", "data": "synthetic",
            "config": {"workload": label, "sample": sample},
            "grays_per_s": sum(x["rays"] for x in vals) / sum(x["seconds"] for x in vals) / 1e9,
            "cpu_baseline": {"value": v, "unit": "Mpaths/s", "cores": cpu_threads, "kind": "port", "sample": sample,
                             "note": f"C++ restatement of the TypeScript reference (no node toolchain in the image), {ORACLE_BUILD}; row strips, one per thread, like src/raytracer.ts:60-90"},
            "e2e": {"value": v, "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        emit(line)
        return 0

    # ---------------------------------------------------------------- B200 arm
    import numpy as np
    import torch
    import torch.distributed as dist

    from mcp_raytracer_b200 import _native, createCameraFromSceneData, measureFp32Peak
    from mcp_raytracer_b200.distributed import SharedFramebuffer, gather_owned_blocks, merge_stats
    from mcp_raytracer_b200.scene_data import rt_stats

    if not torch.cuda.is_available() or _native.lib().rt_device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: the render path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1 and not env["group"]:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        env["group"] = True

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sd = make_scene(kind, scene_opts)
    part = {"partIndex": rank, "partCount": world, "device": local_rank}
    cam = createCameraFromSceneData(sd, {**ropts, **part})
    W, H = cam.imageWidth, cam.imageHeight
    stream = torch.cuda.current_stream()
    cam.setStream(stream.cuda_stream)
    # N > 1: ONE framebuffer, in rank 0's memory, that every rank's render kernel writes its own blocks into (CUDA IPC +
    # NVLink peer stores); if the ranks cannot map it, each rank renders into its own buffer and rank 0 gathers the owned
    # pixels (1/N of the image per rank) with one NCCL gather.
    shared = SharedFramebuffer(W, H, local_rank) if world > 1 else None
    peer_writes = bool(shared and shared.ok)
    if peer_writes:
        fb_ptr = shared.ptr
        fb = shared.as_tensor() if rank == 0 else None
    else:
        fb = torch.zeros((H, W, 3), dtype=torch.uint8, device=dev)
        fb_ptr = fb.data_ptr()
    stats_dev = torch.zeros(80, dtype=torch.uint8, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    host_fb = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory()

    def read_stats():
        import ctypes

        raw = bytes(stats_dev.cpu().numpy())
        assert ctypes.sizeof(rt_stats) == 80 == len(raw)
        return rt_stats.from_buffer_copy(raw)

    def step_device():
        cam.renderRegionDevice(None, fb_ptr, 0, 0, stats_dev.data_ptr())

    # warm-up (untimed)
    for _ in range(max(args.warmup, 3) if args.warmup >= 3 else args.warmup):
        step_device()
    barrier()
    fp32_peak, sm_attr_mhz = measureFp32Peak(local_rank) if rank == 0 else (None, None)
    barrier()

    # ---- timed region: EXACTLY K steps, CUDA events per step, L2 flushed between steps ----
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    wall0 = time.perf_counter()
    for k in range(args.steps):
        flush.zero_()
        ev[k][0].record(stream)
        step_device()
        ev[k][1].record(stream)
    barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop() if sampler else None
    step_ms = [a.elapsed_time(b) for a, b in ev]
    local_ms = sum(step_ms)
    st_local = read_stats()
    t = torch.tensor([local_ms], dtype=torch.float64, device=dev)
    sums = torch.tensor([st_local.pixels, st_local.samples_total, st_local.bounces_total, st_local.rays], dtype=torch.int64, device=dev)
    mins = torch.tensor([st_local.samples_min, st_local.bounces_min], dtype=torch.int64, device=dev)
    maxs = torch.tensor([st_local.samples_max, st_local.bounces_max], dtype=torch.int64, device=dev)
    rank_ms = [local_ms / args.steps]
    if world > 1:
        every = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(every, t)
        rank_ms = [float(x.item()) / args.steps for x in every]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    rank_paths = [int(st_local.samples_total)]
    if world > 1:
        mine = torch.tensor([int(st_local.samples_total)], dtype=torch.int64, device=dev)
        every = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        rank_paths = [int(x.item()) for x in every]
    merge_stats(sums, mins, maxs)
    total_ms = float(t.item())
    paths_per_step, rays_per_step = int(sums[1].item()), int(sums[3].item())
    kernel_launches_per_step = int(st_local.kernel_launches)
    if args.dump_outputs:  # the image and statistics of the last timed step, outside every timed region
        if world > 1:
            torch.cuda.synchronize()
            if peer_writes:
                dist.barrier()                                     # every rank's pixels are in rank 0's framebuffer
            else:
                gather_owned_blocks(fb)
        if rank == 0:
            stats = [sums[0], sums[1], mins[0], maxs[0], sums[2], mins[1], maxs[1], sums[3]]
            dump_outputs(args.dump_outputs, workload, fb.cpu().numpy(), [int(x.item()) for x in stats],
                         DUMP_BYTES // len(args.workload.split(",")))

    # ---- end-to-end through the public API, host buffers, every step: flatten + build + H2D +
    #      render + gather + D2H ----
    from mcp_raytracer_b200.scene_data import FlatScene

    phases = {"create": 0.0, "render": 0.0, "exchange": 0.0, "d2h": 0.0, "destroy": 0.0}

    def e2e_step(record):
        t0 = time.perf_counter()
        c = createCameraFromSceneData(sd, {**ropts, **part})       # SceneData flatten + scene compile (BVH build) + H2D upload
        c.setStream(stream.cuda_stream)
        t1 = time.perf_counter()
        if world > 1:
            c.renderRegionDevice(None, fb_ptr, 0, 0, stats_dev.data_ptr())
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            if peer_writes:
                dist.barrier()                                     # every rank's pixels are in rank 0's framebuffer
            else:
                gather_owned_blocks(fb)
                torch.cuda.synchronize()
            t3 = time.perf_counter()
            if rank == 0:
                host_fb.copy_(fb, non_blocking=True)
                stats_dev.cpu()
            torch.cuda.synchronize()
            t4 = time.perf_counter()
        else:
            c.render(host_fb.numpy().reshape(-1))                  # render + D2H of the RGB8 image and the stats, synchronous
            t2 = t3 = t4 = time.perf_counter()
        c.close()
        t5 = time.perf_counter()
        if record:
            for k, v in zip(phases, (t1 - t0, t2 - t1, t3 - t2, t4 - t3, t5 - t4)):
                phases[k] += 1e3 * v / args.steps

    for _ in range(2):
        e2e_step(False)
    barrier()
    e0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step(True)
    barrier()
    e2e_s = time.perf_counter() - e0
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())
    import hashlib
    fb_sha1 = hashlib.sha1(host_fb.numpy().tobytes()).hexdigest() if rank == 0 else None   # identical for every N
    fs = FlatScene(sd)
    h2d = int(sum(a.nbytes for a in (fs.obj_type, fs.obj_pos, fs.obj_u, fs.obj_v, fs.obj_r, fs.obj_material, fs.obj_light,
                                     fs.mat_type_a, fs.mat_color_a, fs.mat_param_a, fs.mat_child_a)))
    d2h = W * H * 3 + 80

    if rank != 0:
        cam.close()
        if shared:
            dist.barrier()
            shared.close()
        return 0

    value = paths_per_step * args.steps / (total_ms * 1e-3) / 1e6
    grays = rays_per_step * args.steps / (total_ms * 1e-3) / 1e9
    e2e_value = paths_per_step * args.steps / e2e_s / 1e6

    # ---- CPU baseline + algorithmic-work model (oracle = checker / baseline only) ----
    cpu, roof = None, None
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    if not args.no_cpu_baseline:
        # the CPU baseline is reported at N=1 only; at N>1 a 1-second run still supplies the event counts of the flop model
        c = cpu_reference_run(sd, ropts, target_seconds=args.cpu_seconds if world == 1 else 1.0, threads=cpu_threads)
        sample = c["sample"]
        if world == 1:
            cpu = {"value": c["mpaths_per_s"], "unit": "Mpaths/s", "cores": cpu_threads, "kind": "port", "sample": sample,
                   "grays_per_s": c["grays_per_s"], "seconds": c["seconds"],
                   "note": f"C++ restatement of the TypeScript reference (cannot run here), {ORACLE_BUILD}; row strips, one per thread, like src/raytracer.ts:60-90"}
        flops_per_path = algorithmic_flops(c["counters"], c["n_lights"], float(sd["camera"].get("aperture", 0))) / max(1, c["counters"]["paths"])
        kernel_s = (total_ms * 1e-3) / args.steps  # one render kernel per step (max over ranks)
        achieved = flops_per_path * paths_per_step / kernel_s / 1e12
        peak = fp32_peak * world
        hbm_bytes = W * H * 3 + h2d  # compulsory traffic: scene once + RGB8 out
        roof = {
            "bound": "fp32", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
            "traffic": measured_traffic(workload, world, overridden),
            "peak_source": f"FP32 FFMA microbenchmark in this run (rt_measure_fp32_peak): {fp32_peak:.1f} TFLOP/s per GPU at <= {sm_attr_mhz:.0f} MHz; "
                           "MEASURED_PEAKS.json holds HBM/bf16 peaks only",
            "flops_per_path": flops_per_path, "flops_model": "SURVEY.md §8d, event counts from the oracle walking the reference BVH",
            "hbm": {"algorithmic_bytes_per_launch": hbm_bytes, "achieved_gbs": hbm_bytes / kernel_s / 1e9,
                    "peak_gbs": peaks.get("hbm_gbs"), "note": "scene is register/L1-resident; HBM is not the bound"},
        }
        roof["algorithmic_frac"] = roof["frac"]
        # What the device EXECUTES on its own structure (instrumented build, separate process, reduced spp): wide-node visits
        # (4 child boxes, 21 flop each) and primitive tests (23 flop, +29 for the one that hits), plus the model's per-path
        # shading part.  On tree scenes the reference's median-split tree and per-axis box rule make the algorithmic figure
        # count boxes no sensible tree visits (rain 100k: ~6000 per ray), so there `frac` is the executed figure and the
        # reference-tree one stays beside it.
        ev = executed_events(workload, {k: v for k, v in ropts.items() if k in ("width", "depth", "bvh")}, max(1, min(int(ropts["samples"]), 8)))
        if ev and ev["paths"]:
            cnt = c["counters"]
            shade = shading_flops(cnt, c["n_lights"], float(sd["camera"].get("aperture", 0))) / max(1, cnt["paths"])
            hit_frac = cnt["hits"] / max(1, cnt["rays"])
            ray_flops = (84.0 * ev["node_visits"] + 23.0 * ev["prim_tests"] + 29.0 * hit_frac * ev["rays"]) / ev["paths"]
            ex = (ray_flops + shade) * paths_per_step / kernel_s / 1e12
            roof["executed"] = {"achieved": ex, "frac": ex / peak, "flops_per_path": ray_flops + shade,
                                "node_visits_per_ray": ev["node_visits"] / max(1, ev["rays"]), "prim_tests_per_ray": ev["prim_tests"] / max(1, ev["rays"]),
                                "counted_at_spp": max(1, min(int(ropts["samples"]), 8)),
                                "source": "libmcprt_b200_count.so (same kernels with counters), one untimed render in its own process"}
            if cam.info.bvh_kind != 3:
                roof["reference_tree"] = {"achieved": roof["achieved"], "frac": roof["frac"], "flops_per_path": flops_per_path}
                roof["achieved"], roof["frac"], roof["flops_per_path"] = ex, ex / peak, ray_flops + shade
                roof["flops_model"] = "SURVEY.md §8d constants on the events the device executes on its own 4-wide SAH tree; reference-tree figure under reference_tree"

    # The same workload with the reference's DEFAULT render options (adaptive sampling on: aTolerance 0.05, aBatch 10 —
    # src/camera.ts:73-83; the headline config turns it off).  One GPU only, outside every timed region, never part of `value`.
    ref_defaults = None
    if world == 1:
        try:
            with createCameraFromSceneData(sd, {**ropts, "aTolerance": 0.05, "aBatch": 10}) as ac:
                abuf = np.zeros(W * H * 3, np.uint8)
                ast = min((ac.render(abuf) for _ in range(2)), key=lambda s_: s_.deviceMs)
            ref_defaults = {"aTolerance": 0.05, "aBatch": 10, "value": ast.samples["total"] / ast.deviceMs / 1e3, "unit": "Mpaths/s",
                            "grays_per_s": ast.rays / ast.deviceMs / 1e6, "ms": ast.deviceMs, "samples_taken": int(ast.samples["total"]),
                            "samples_at_fixed_spp": paths_per_step,
                            "note": "device time of one render (best of 2), scene resident; not the headline configuration"}
        except Exception as e:  # never lets the optional figure break the bench line
            ref_defaults = {"error": str(e)[:200]}

    line = {
        "metric": "Mpaths/s", "value": value, "unit": "Mpaths/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": label + (" [OVERRIDDEN size: development run]" if overridden else ""), "image": f"{W}x{H}", "spp": ropts["samples"],
                   "bvh": {1: "reference", 2: "sah", 3: "list"}.get(cam.info.bvh_kind), "integrator": {1: "megakernel", 2: "wavefront", 3: "sorted"}.get(cam.info.integrator_kind),
                   "partition": f"8x4 pixel blocks, one per rank per run of {world} blocks, order rotated by a hash of the run (rt_block_owner)",
                   "exchange": ("none (1 GPU)" if world == 1 else "render kernels store owned pixels into rank 0's framebuffer over NVLink (CUDA IPC peer mapping); no collective"
                                if peer_writes else "NCCL gather of each rank's owned pixels (1/N of the image)"), "rng": "Philox4x32-7 keyed (pixel,sample), counter (block,bounce)",
                   "l2": "256 MiB memset between steps, outside the per-step CUDA-event pairs"},
        "grays_per_s": grays, "paths_per_step": paths_per_step, "rays_per_step": rays_per_step,
        "wall_s_timed_region": wall, "step_ms": step_ms,
        "rank_ms": {"min": min(rank_ms), "median": statistics.median(rank_ms), "max": max(rank_ms), "per_rank": rank_ms},
        "rank_paths": rank_paths, "fb_sha1": fb_sha1,
        "clocks": {k: clocks[k] for k in ("sm_mhz", "sm_max_mhz", "reasons")} if clocks else None,
        "e2e": {"value": e2e_value, "unit": "Mpaths/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": 1e3 * e2e_s / args.steps, "breakdown_ms": phases,
                "includes": "SceneData flatten + BVH build + H2D + render + gather + D2H of the RGB8 framebuffer and stats"},
        "gpu_launches": kernel_launches_per_step * args.steps * world,
        "roofline": roof, "cpu_baseline": cpu,
        "reference_defaults_adaptive": ref_defaults,
    }
    emit(line)
    cam.close()
    if shared:
        dist.barrier()
        shared.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
