"""The denoiser on every device (MultiCamera.renderDenoised): call times against the plain multi-GPU render and the one-GPU
denoiser, one JSON line per (case, N) (the numbers of profiles/README.md section 9).
usage: gpu_multi_denoise.py <out_dir> [--baseline]   (r04_multi_denoise.jsonl / r04_multi_denoise_baseline.jsonl is written there)

Cases: Cornell 1024x1024 @16 spp, Cornell 3840x2160 @16 spp, rain (100k spheres, radius 0.01) 3840x2160 @64 spp, all
fixed spp (aTolerance 0).  For N in {1, 2, 4, 8} devices (those the box has):
* kind "calls": medians of 5 timed synchronous calls after 2 warm-ups (host clock around the call): MultiCamera.renderDenoised,
  MultiCamera.render with the same options, and the one-GPU Camera.renderDenoised (measured once per case); the SHA-1 of the
  denoised rgb8, which must be the same for every N and equal to the one-GPU image's.
* kind "kernels": a torch.profiler run of its own (3 calls after the warm-ups): device time per call and device of the
  render, features, prepare, a-trous passes and finish kernels.
--baseline: only the one-GPU renderDenoised and MultiCamera.render (for a build without rt_multi_render_denoised).
Every line carries the card name and power limit read in the same process."""
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

from mcp_raytracer_b200 import Camera, MultiCamera, _native, generateCornellSceneData, generateRainSceneData  # noqa: E402

if len(sys.argv) < 2:
    sys.exit(__doc__)
OUT = sys.argv[1]
BASELINE = "--baseline" in sys.argv[2:]
os.makedirs(OUT, exist_ok=True)
card = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"]).decode().strip()
lines = []


def emit(d):
    d["card"] = card
    d["build"] = "baseline" if BASELINE else "this tree"
    print(json.dumps(d), flush=True)
    lines.append(d)


def timed(fn, warmup=2, reps=5):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts), min(ts), max(ts)


CASES = [
    ("cornell-1024", generateCornellSceneData, {"width": 1024, "aspect": 1.0, "samples": 16}),
    ("cornell-3840x2160", generateCornellSceneData, {"width": 3840, "aspect": 16 / 9, "samples": 16}),
    ("rain100k-3840x2160", lambda: generateRainSceneData({"count": 100000, "seed": 1, "sphereRadius": 0.01}),
     {"width": 3840, "aspect": 16 / 9, "samples": 64}),
]
STAGES = (("render", "k_render"), ("features", "k_render_features"), ("prepare", "k_denoise_prepare"), ("passes", "k_denoise_pass"),
          ("finish", "k_denoise_finish"))


def stage_of(name):
    for stage, prefix in reversed(STAGES):  # k_render_features before k_render
        if name.startswith(prefix):
            return stage
    return None


def kernel_split(mc, rgb, n, reps=3):
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            mc.renderDenoised(rgb)
    per = {}
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        name = e.name.split("<")[0].split("(")[0].replace("void ", "").replace("rt::", "")
        stage = stage_of(name)
        if stage:
            key = f"dev{e.device_index}"
            per.setdefault(key, {s: 0.0 for s, _ in STAGES})
            per[key][stage] += e.time_range.elapsed_us() / 1e3 / reps  # ms per call
    return per


ndev = _native.lib().rt_device_count()
for name, scene, o in CASES:
    sd = scene()
    opts = {**o, "aTolerance": 0, "seed": 3}
    with Camera(sd, None, opts) as cam:
        W, H = cam.imageWidth, cam.imageHeight
        rgb1 = np.zeros(W * H * 3, np.uint8)
        one_ms = timed(lambda: cam.renderDenoised(rgb1))
    sha_one = hashlib.sha1(rgb1.tobytes()).hexdigest()
    for n in (1, 2, 4, 8):
        if n > ndev:
            continue
        with MultiCamera(sd, opts, nDevices=n) as mc:
            rgb = np.zeros(W * H * 3, np.uint8)
            plain_ms = timed(lambda: mc.render(rgb))
            d = {"kind": "calls", "case": name, "size": f"{W}x{H}", "spp": opts["samples"], "n_gpus": n, "peer_writes": mc.peerWrites,
                 "one_gpu_render_denoised_ms": one_ms[0], "one_gpu_render_denoised_ms_range": one_ms[1:],
                 "multi_render_ms": plain_ms[0], "multi_render_ms_range": plain_ms[1:]}
            if not BASELINE:
                dn_ms = timed(lambda: mc.renderDenoised(rgb))
                sha = hashlib.sha1(rgb.tobytes()).hexdigest()
                d.update({"multi_render_denoised_ms": dn_ms[0], "multi_render_denoised_ms_range": dn_ms[1:],
                          "denoise_overhead_ms": dn_ms[0] - plain_ms[0], "rgb8_sha1": sha, "one_gpu_rgb8_sha1": sha_one,
                          "equal_to_one_gpu": sha == sha_one})
            emit(d)
            if not BASELINE:
                emit({"kind": "kernels", "case": name, "size": f"{W}x{H}", "n_gpus": n, "ms_per_call": kernel_split(mc, rgb, n)})
with open(os.path.join(OUT, "r04_multi_denoise_baseline.jsonl" if BASELINE else "r04_multi_denoise.jsonl"), "w") as f:
    for d in lines:
        f.write(json.dumps(d) + "\n")
