"""Progressive renders on every device (MultiCamera.renderProgressive / renderProgressiveDenoised): time to the first preview,
the whole call and the device time of each pass, against the same passes through one Camera and the one-shot multi call
(the numbers of profiles/README.md section 9.3).
usage: gpu_multi_progressive.py <out_dir>   -> <out_dir>/r06_multi_progressive.jsonl

Cases (fixed spp, aTolerance 0): Cornell 1024x1024 @64 spp in 8 passes (plain and denoised), Cornell 3840x2160 @16 spp in
4 passes (denoised), rain (100k spheres, radius 0.01) 3840x2160 @64 spp in 4 passes (plain and denoised).
For N in {1, 2, 4, 8} devices (those the box has), and, labelled "overhead only", RT_B200_MULTI_PARTS = 2 and 8 parts on
one GPU (the parts share its SMs: the numbers are the cost of the partitioned passes, not a scaling):
* medians (and ranges) of 5 timed synchronous calls after a warm-up, host clock around the call, the multi call and the
  same passes through one Camera alternating: the whole call, the host clock from the call to the first onPass, and the
  device time of each pass (the difference of the cumulative deviceMs onPass receives);
* the one-shot MultiCamera.render / renderDenoised (median of 5 after a warm-up);
* the SHA-1 of the last pass's rgb8, of one Camera's, and of the one-shot multi call's.
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
os.makedirs(OUT, exist_ok=True)
card = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"]).decode().strip()
lines = []


def emit(d):
    d["card"] = card
    print(json.dumps(d), flush=True)
    lines.append(d)


def rain100k():
    return generateRainSceneData({"count": 100000, "seed": 1, "sphereRadius": 0.01})


CASES = [  # (name, scene, render options, passes, denoised)
    ("cornell-1024-64spp", generateCornellSceneData, {"width": 1024, "aspect": 1.0, "samples": 64}, 8, False),
    ("cornell-1024-64spp", generateCornellSceneData, {"width": 1024, "aspect": 1.0, "samples": 64}, 8, True),
    ("cornell-3840x2160-16spp", generateCornellSceneData, {"width": 3840, "aspect": 16 / 9, "samples": 16}, 4, True),
    ("rain100k-3840x2160-64spp", rain100k, {"width": 3840, "aspect": 16 / 9, "samples": 64}, 4, False),
    ("rain100k-3840x2160-64spp", rain100k, {"width": 3840, "aspect": 16 / 9, "samples": 64}, 4, True),
]


def progressive(cam, rgb, passes, denoised):
    """One synchronous call: (whole call ms, ms to the first onPass, device ms of each pass)."""
    marks, cum = [], []

    def on_pass(k, n, cap, so_far):
        marks.append(time.perf_counter())
        cum.append(so_far.deviceMs)
        return False

    t0 = time.perf_counter()
    if denoised:
        cam.renderProgressiveDenoised(rgb, passes, on_pass)
    else:
        cam.renderProgressive(rgb, passes, on_pass)
    t1 = time.perf_counter()
    return (t1 - t0) * 1e3, (marks[0] - t0) * 1e3, [b - a for a, b in zip([0.0] + cum[:-1], cum)]


def summary(runs):
    call = [r[0] for r in runs]
    first = [r[1] for r in runs]
    per_pass = [statistics.median(p[i] for _, _, p in runs) for i in range(len(runs[0][2]))]
    return {"call_ms": statistics.median(call), "call_ms_range": [min(call), max(call)],
            "first_preview_ms": statistics.median(first), "first_preview_ms_range": [min(first), max(first)],
            "pass_device_ms": per_pass}


def sha(a):
    return hashlib.sha1(a.tobytes()).hexdigest()


ndev = _native.lib().rt_device_count()
configs = [(n, None) for n in (1, 2, 4, 8) if n <= ndev] + [(1, 2), (1, 8)]
scenes = {}
for name, scene, o, passes, denoised in CASES:
    if name not in scenes:
        scenes[name] = scene()
    sd = scenes[name]
    opts = {**o, "aTolerance": 0, "seed": 3}
    with Camera(sd, None, opts) as cam:
        W, H = cam.imageWidth, cam.imageHeight
        rgb1 = np.zeros(W * H * 3, np.uint8)
        progressive(cam, rgb1, passes, denoised)  # warm-up
        for n, parts in configs:
            if parts:
                os.environ["RT_B200_MULTI_PARTS"] = str(parts)
            else:
                os.environ.pop("RT_B200_MULTI_PARTS", None)
            with MultiCamera(sd, opts, nDevices=n) as mc:
                os.environ.pop("RT_B200_MULTI_PARTS", None)
                rgb = np.zeros(W * H * 3, np.uint8)
                progressive(mc, rgb, passes, denoised)  # warm-up
                multi, one = [], []
                for _ in range(5):  # alternating: the spread of both is measured in the same window
                    multi.append(progressive(mc, rgb, passes, denoised))
                    one.append(progressive(cam, rgb1, passes, denoised))
                sha_multi, sha_one = sha(rgb), sha(rgb1)
                shot = np.zeros(W * H * 3, np.uint8)
                call = (lambda: mc.renderDenoised(shot)) if denoised else (lambda: mc.render(shot))
                call()
                ts = []
                for _ in range(5):
                    t0 = time.perf_counter()
                    call()
                    ts.append((time.perf_counter() - t0) * 1e3)
                emit({"case": name, "size": f"{W}x{H}", "spp": opts["samples"], "passes": passes, "denoised": denoised,
                      "n_gpus": n, "parts": mc.nDevices, "overhead_only": bool(parts), "peer_writes": mc.peerWrites,
                      "multi": summary(multi), "one_camera": summary(one),
                      "one_shot_multi_ms": statistics.median(ts), "one_shot_multi_ms_range": [min(ts), max(ts)],
                      "rgb8_sha1": sha_multi, "one_camera_rgb8_sha1": sha_one, "one_shot_multi_rgb8_sha1": sha(shot),
                      "equal": sha_multi == sha_one == sha(shot)})
with open(os.path.join(OUT, "r06_multi_progressive.jsonl"), "w") as f:
    for d in lines:
        f.write(json.dumps(d) + "\n")
