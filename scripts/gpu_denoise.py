"""The denoiser's cost and quality, one JSON line per case (the numbers of profiles/README.md section 9).
usage: gpu_denoise.py <out_dir>   (denoise.jsonl is written there)

* kind "kernels": device time per kernel of one Camera.renderDenoised from a torch.profiler run of its own (warmed up;
  features, prepare, 5 a-trous passes, finish; the render kernel for comparison) at 1024x1024 and 3840x2160, Cornell @16 spp.
* kind "quality": relMSE = mean((x - r)^2 / (r^2 + 0.01)) against an 8192-spp render with another seed, noisy vs denoised,
  Cornell 1024x1024 at 4/16/64 spp and the layered/mixed box (C5) at 384x384.
* kind "equal_time": the spp at which the undenoised render reaches the denoised 16-spp relMSE (log-log interpolation
  between powers of two), with the device time of both renders.
Every line carries the card name and power limit read in the same process."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

from mcp_raytracer_b200 import createCameraFromSceneData, generateCornellSceneData, generateLayeredMixedSceneData  # noqa: E402

if len(sys.argv) != 2:
    sys.exit(__doc__)
OUT = sys.argv[1]
os.makedirs(OUT, exist_ok=True)
card = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"]).decode().strip()
lines = []


def emit(d):
    d["card"] = card
    print(json.dumps(d), flush=True)
    lines.append(d)


def render(sd, opts, denoised=False):
    with createCameraFromSceneData(sd, opts) as cam:
        lin = np.zeros((cam.imageHeight, cam.imageWidth, 3), np.float32)
        st = cam.renderDenoised(None, lin) if denoised else cam.renderRegion(None, None, lin)
    return lin, st.deviceMs


def rel_mse(x, r):
    return float(((x.astype(np.float64) - r) ** 2 / (r.astype(np.float64) ** 2 + 0.01)).mean())


def kernels(width, aspect):
    import torch
    from torch.profiler import ProfilerActivity, profile

    sd = generateCornellSceneData()
    with createCameraFromSceneData(sd, {"width": width, "aspect": aspect, "samples": 16, "aTolerance": 0, "seed": 3}) as cam:
        rgb = np.zeros(cam.imageWidth * cam.imageHeight * 3, np.uint8)
        for _ in range(2):
            cam.renderDenoised(rgb)
        torch.cuda.synchronize()
        reps = 5
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                st = cam.renderDenoised(rgb)
        per = {}
        for e in prof.key_averages():
            if e.device_type.name == "CUDA" and e.count:
                name = e.key.split("<")[0].split("(")[0].replace("void ", "").replace("rt::", "")
                per[name] = per.get(name, 0.0) + e.device_time_total / 1e3 / reps  # ms per call
        emit({"kind": "kernels", "size": f"{cam.imageWidth}x{cam.imageHeight}", "spp": 16, "ms_per_call": per,
              "filter_ms": sum(v for k, v in per.items() if k.startswith("k_denoise") or k.startswith("k_render_features")),
              "call_device_ms": st.deviceMs})


def quality():
    cases = [("C2-cornell", generateCornellSceneData(), 1024, [4, 16, 64]), ("C5-layered", generateLayeredMixedSceneData(), 384, [16])]
    for name, sd, width, spps in cases:
        base = {"width": width, "aspect": 1.0, "aTolerance": 0}
        ref, ref_ms = render(sd, {**base, "samples": 8192, "seed": 1234})
        den16 = None
        for spp in spps:
            noisy, ms_n = render(sd, {**base, "samples": spp, "seed": 7})
            den, ms_d = render(sd, {**base, "samples": spp, "seed": 7}, denoised=True)
            e_n, e_d = rel_mse(noisy, ref), rel_mse(den, ref)
            if spp == 16:
                den16 = (e_d, ms_d)
            emit({"kind": "quality", "scene": name, "size": f"{width}x{width}", "spp": spp, "relmse_noisy": e_n, "relmse_denoised": e_d,
                  "ratio": e_d / e_n, "render_ms": ms_n, "denoised_ms": ms_d, "reference_spp": 8192})
        # equal time: the undenoised spp that reaches the denoised 16-spp error
        prev = None
        spp = 16
        while spp <= 8192:
            noisy, ms_n = render(sd, {**base, "samples": spp, "seed": 7})
            e = rel_mse(noisy, ref)
            if e <= den16[0]:
                s_eq = spp
                if prev:
                    (s0, e0) = prev
                    s_eq = float(np.exp(np.log(s0) + (np.log(den16[0]) - np.log(e0)) / (np.log(e) - np.log(e0)) * (np.log(spp) - np.log(s0))))
                emit({"kind": "equal_time", "scene": name, "size": f"{width}x{width}", "denoised_spp": 16, "relmse_denoised": den16[0],
                      "denoised_ms": den16[1], "equal_error_spp": s_eq, "render_ms_at_bracket": ms_n, "bracket_spp": spp})
                break
            prev = (spp, e)
            spp *= 2
        else:
            emit({"kind": "equal_time", "scene": name, "denoised_spp": 16, "relmse_denoised": den16[0], "equal_error_spp": "> 8192"})


kernels(1024, 1.0)
kernels(3840, 16 / 9)
quality()
with open(os.path.join(OUT, "denoise.jsonl"), "w") as f:
    for d in lines:
        f.write(json.dumps(d) + "\n")
