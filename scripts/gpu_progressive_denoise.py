"""The progressive denoised render (Camera.renderProgressiveDenoised): time to the first preview, per-pass render and filter
device time, the whole call against one-shot renderDenoised and plain renderProgressive, and the relMSE of every preview
(the numbers of profiles/README.md section 9.2).
usage: gpu_progressive_denoise.py <out_dir>               -> <out_dir>/r05_progressive_denoise.jsonl
       gpu_progressive_denoise.py <out_dir> --ab <root>   -> <out_dir>/r05_progressive_denoise_ab.jsonl

Cases: Cornell 1024x1024 @64 spp in 8 passes, rain (100k spheres, radius 0.01) 3840x2160 @64 spp in 4 passes, fixed spp.
* kind "calls": medians of 3 timed synchronous calls after a warm-up (host clock around the call) of renderProgressiveDenoised,
  renderProgressive with the same passes and renderDenoised; the host clock from the call to the first onPass; the device
  time of each pass (the difference of the cumulative deviceMs onPass receives); whether the last preview's rgb8 equals
  renderDenoised's.
* kind "kernels": a torch.profiler run of its own (one call after the warm-ups): per pass, the device time of the render
  kernel, the features (first pass only) and the filter (prepare, a-trous passes, finish).
* kind "quality" (Cornell only): relMSE of every preview against an 8192-spp render with another seed, noisy (the
  preview of renderProgressive) and denoised.
--ab <root>: the non-regression workloads, alternating this tree and the checkout at <root> (built) in child processes, three
rounds: Cornell 1024x1024 with the reference's adaptive defaults through the pixel stream (RT_B200_NO_ADAPTIVE_POOL=1),
rain 100k 3840x2160 with the adaptive defaults (k_render_stream_trav), renderDenoised on Cornell 3840x2160 @16 spp, and
Cornell 1024x1024 @64 spp with shadow rays on the reference tree (k_render_stream<BVH_REFERENCE, true>).  Median
render deviceMs of 5 calls after a warm-up, and the rgb8 SHA-1.
Every line carries the card name and power limit read in the same process."""
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"]).decode().strip()


def rain100k():
    from mcp_raytracer_b200 import generateRainSceneData

    return generateRainSceneData({"count": 100000, "seed": 1, "sphereRadius": 0.01})


AB_WORKLOADS = {  # name: (scene, render options, renderDenoised?, environment)
    "cornell-1024-adaptive-stream": ("cornell", {"width": 1024, "aspect": 1.0, "seed": 3}, False, {"RT_B200_NO_ADAPTIVE_POOL": "1"}),
    "rain100k-3840x2160-adaptive": ("rain100k", {"width": 3840, "aspect": 16 / 9, "seed": 3}, False, {}),
    "cornell-3840x2160-denoised-16": ("cornell", {"width": 3840, "aspect": 16 / 9, "samples": 16, "aTolerance": 0, "seed": 3}, True, {}),
    "cornell-1024-shadow-rays-reference-64": ("cornell", {"width": 1024, "aspect": 1.0, "samples": 64, "aTolerance": 0, "seed": 3,
                                                          "bvh": "reference", "lightSampling": "shadowRays"}, False, {}),
}


def ab_child(name, root):
    """One workload in this process, with the package and library of the tree at `root`: one JSON line."""
    sys.path.insert(0, root)
    import numpy as np

    from mcp_raytracer_b200 import Camera, generateCornellSceneData

    scene, opts, denoised, _env = AB_WORKLOADS[name]
    sd = generateCornellSceneData() if scene == "cornell" else rain100k()
    with Camera(sd, None, opts) as cam:
        rgb = np.zeros(cam.imageWidth * cam.imageHeight * 3, np.uint8)
        call = (lambda: cam.renderDenoised(rgb)) if denoised else (lambda: cam.render(rgb))
        call()
        ms = [call().deviceMs for _ in range(5)]
    print(json.dumps({"ms": statistics.median(ms), "ms_range": [min(ms), max(ms)], "rgb8_sha1": hashlib.sha1(rgb.tobytes()).hexdigest()}))


def ab(out, other):
    lines, c = [], card()
    trees = (("this tree", ROOT), ("other", os.path.abspath(other)))
    for rnd in range(3):
        for name, (_s, _o, _d, env) in AB_WORKLOADS.items():
            for label, root in trees:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", name, root], env={**os.environ, **env},
                                   capture_output=True, text=True, cwd=root)
                if r.returncode != 0:
                    raise SystemExit(f"{label} {name}: {r.stderr.strip()[-2000:]}")
                d = {"kind": "ab", "round": rnd, "workload": name, "build": label, **json.loads(r.stdout.strip().splitlines()[-1]), "card": c}
                print(json.dumps(d), flush=True)
                lines.append(d)
    with open(os.path.join(out, "r05_progressive_denoise_ab.jsonl"), "w") as f:
        f.writelines(json.dumps(d) + "\n" for d in lines)


def rel_mse(x, r):
    import numpy as np

    return float(((x.astype(np.float64) - r) ** 2 / (r.astype(np.float64) ** 2 + 0.01)).mean())


def wall(fn):
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


def progressive_call(cam, rgb, lin, passes, denoised, keep=False):
    """One synchronous call: (wall ms, wall ms to the first onPass, per-pass device ms, [linear copies])."""
    marks, dev, copies = [], [], []

    def on_pass(k, n, cap, so_far):
        marks.append(time.perf_counter())
        dev.append(so_far.deviceMs)
        if keep:
            copies.append((cap, lin.copy()))
        return False

    t0 = time.perf_counter()
    if denoised:
        cam.renderProgressiveDenoised(rgb, passes, on_pass, linear=lin)
    else:
        cam.renderProgressive(rgb, passes, on_pass, linear=lin)
    t1 = time.perf_counter()
    per_pass = [b - a for a, b in zip([0.0] + dev[:-1], dev)]
    return (t1 - t0) * 1e3, (marks[0] - t0) * 1e3, per_pass, copies


def kernel_split(cam, rgb, passes):
    """Device ms per pass of the render kernel, the features and the filter, from torch.profiler (one call)."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        cam.renderProgressiveDenoised(rgb, passes)
        torch.cuda.synchronize()
    evs = sorted((e for e in prof.events() if e.device_type.name == "CUDA"), key=lambda e: e.time_range.start)
    out = []
    for e in evs:
        name = e.name.split("<")[0].split("(")[0].replace("void ", "").replace("rt::", "")
        ms = e.time_range.elapsed_us() / 1e3
        if name.startswith("k_render_features"):
            out[-1]["features_ms"] += ms
        elif name.startswith("k_render"):
            out.append({"render_ms": ms, "features_ms": 0.0, "filter_ms": 0.0, "render_kernel": name})
        elif name.startswith("k_denoise"):
            out[-1]["filter_ms"] += ms
    return out


def main(out):
    import numpy as np

    from mcp_raytracer_b200 import Camera, generateCornellSceneData

    c = card()
    lines = []

    def emit(d):
        d["card"] = c
        print(json.dumps(d), flush=True)
        lines.append(d)

    cases = [("cornell-1024", generateCornellSceneData, {"width": 1024, "aspect": 1.0}, 8),
             ("rain100k-3840x2160", rain100k, {"width": 3840, "aspect": 16 / 9}, 4)]
    for name, scene, o, passes in cases:
        sd = scene()
        opts = {**o, "samples": 64, "aTolerance": 0, "seed": 3}
        with Camera(sd, None, opts) as cam:
            W, H = cam.imageWidth, cam.imageHeight
            rgb = np.zeros((H, W, 3), np.uint8)
            lin = np.zeros((H, W, 3), np.float32)
            one = np.zeros_like(rgb)
            res = {}
            for label, fn in (("progressive_denoised", lambda: progressive_call(cam, rgb, lin, passes, True)),
                              ("progressive", lambda: progressive_call(cam, rgb, lin, passes, False)),
                              ("render_denoised", lambda: (wall(lambda: cam.renderDenoised(one)), None, None, None))):
                fn()
                runs = [fn() for _ in range(3)]
                res[label] = runs
            pd = res["progressive_denoised"]
            cam.renderProgressiveDenoised(rgb, passes)
            cam.renderDenoised(one)
            emit({"kind": "calls", "case": name, "size": f"{W}x{H}", "spp": 64, "passes": passes,
                  "progressive_denoised_ms": statistics.median(r[0] for r in pd),
                  "first_preview_ms": statistics.median(r[1] for r in pd),
                  "pass_device_ms": [statistics.median(r[2][k] for r in pd) for k in range(len(pd[0][2]))],
                  "progressive_ms": statistics.median(r[0] for r in res["progressive"]),
                  "progressive_pass_device_ms": [statistics.median(r[2][k] for r in res["progressive"]) for k in range(len(res["progressive"][0][2]))],
                  "render_denoised_ms": statistics.median(r[0] for r in res["render_denoised"]),
                  "last_preview_equals_render_denoised": bool(np.array_equal(rgb, one))})
            emit({"kind": "kernels", "case": name, "size": f"{W}x{H}", "passes": kernel_split(cam, rgb, passes)})
            if name.startswith("cornell"):
                noisy = progressive_call(cam, rgb, lin, passes, False, keep=True)[3]
                den = progressive_call(cam, rgb, lin, passes, True, keep=True)[3]
                with Camera(sd, None, {**opts, "samples": 8192, "seed": 1234}) as rc:
                    ref = np.zeros((H, W, 3), np.float32)
                    rc.renderRegion(None, None, ref)
                emit({"kind": "quality", "case": name, "size": f"{W}x{H}", "reference_spp": 8192,
                      "passes": [{"cap": cn, "relmse_noisy": rel_mse(ln, ref), "relmse_denoised": rel_mse(ld, ref)}
                                 for (cn, ln), (_cd, ld) in zip(noisy, den)]})
    with open(os.path.join(out, "r05_progressive_denoise.jsonl"), "w") as f:
        f.writelines(json.dumps(d) + "\n" for d in lines)


if __name__ == "__main__":
    if len(sys.argv) >= 4 and sys.argv[1] == "--child":
        ab_child(sys.argv[2], sys.argv[3])
        sys.exit(0)
    if len(sys.argv) < 2:
        sys.exit(__doc__)
    os.makedirs(sys.argv[1], exist_ok=True)
    if "--ab" in sys.argv[2:]:
        ab(sys.argv[1], sys.argv[sys.argv.index("--ab") + 1])
    else:
        sys.path.insert(0, ROOT)
        main(sys.argv[1])
