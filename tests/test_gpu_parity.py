"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle on the
same seeded inputs (north_star bars: primary hits exact on object id and within 1e-4 relative
on t / normal; converged images within 1% RMSE and 3 sigma per pixel).

Run on the B200 box with `-m gpu`.  Nothing here reads /root/reference.
"""
import ctypes as C
import json
import os

import numpy as np
import pytest

import oracle_binding as ob
import parity_stats as pstat
from mcp_raytracer_b200 import (
    Camera, RaytracerError, RenderStats, createCameraFromSceneData, generateCornellSceneData, generateDefaultSceneData,
    generateLayeredMixedSceneData, generateRainSceneData, generateSpheresSceneData, generateWeekendFinalSceneData,
    renderScene,
)
from mcp_raytracer_b200 import _native
from mcp_raytracer_b200.scene_data import FlatScene, merge_render_options, render_opts_struct, rt_render_opts, rt_scene_desc

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")

SCENES = {
    "C1-spheres": lambda: generateSpheresSceneData({"count": 100, "seed": 12345}),
    "C2-cornell": generateCornellSceneData,
    "C3-weekend": generateWeekendFinalSceneData,
    "C4-rain": lambda: generateRainSceneData({"count": 20000, "seed": 1, "sphereRadius": 0.01}),
    "C5-layered": generateLayeredMixedSceneData,
    "default": generateDefaultSceneData,
}


def gpu_render(sd, opts, want_moments=False, region=None):
    with createCameraFromSceneData(sd, opts) as cam:
        W, H = cam.imageWidth, cam.imageHeight
        rgb = np.zeros((H, W, 3), np.uint8)
        lin = np.zeros((H, W, 3), np.float32)
        mom = np.zeros((H, W, 8), np.float32) if want_moments else None
        st = cam.renderRegion(rgb, region, lin, mom)
    return {"rgb8": rgb, "linear": lin, "moments": mom, "stats": st}


# ------------------------------------------------------------------------------------------
# primary visibility: exact object id, 1e-4 relative on t and normal
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(SCENES))
@pytest.mark.parametrize("bvh", ["auto", "reference", "sah"])
def test_primary_hits_match_oracle(gpu, name, bvh):
    sd = SCENES[name]()
    opts = {"width": 384, "samples": 1, "bvh": bvh}
    with createCameraFromSceneData(sd, opts) as cam:
        ids, t, nrm, ff = cam.tracePrimary()
        kind = cam.info.bvh_kind
    oc = ob.OracleCamera(sd, opts)
    oids, ot, onrm, off = oc.trace_primary()
    has_negative = any(o.get("r", 1) < 0 for o in sd["objects"])
    if kind == 2 and has_negative:
        # a SAH tree cannot reproduce the inverted-box quirk of negative-radius spheres
        # (SURVEY.md App. A.4); AUTO never picks SAH for such scenes.
        pytest.skip("forced SAH on a scene with a negative-radius sphere")
    assert np.array_equal(ids, oids), f"{int((ids != oids).sum())} primary-hit ids differ ({name}, bvh kind {kind})"
    hit = oids >= 0
    assert np.all(np.abs(t[hit] - ot[hit]) <= 1e-4 * np.abs(ot[hit]))
    assert np.all(np.abs(nrm[hit] - onrm[hit]) <= 1e-4 * 2)  # unit normals: 1e-4 relative
    assert np.array_equal(ff[hit], off[hit])
    assert np.all(np.isinf(t[~hit]))


def _random_scene(seed, n):
    """Seeded mix of spheres (tiny ... scene-sized), axis-aligned and rotated quads and an occasional infinite
    plane: exercises every AUTO choice (LIST / room rule / SAH), the always-tested prefix and the 4-wide tree."""
    rng = np.random.default_rng(seed)
    objs = []
    mats = [{"type": "lambert", "color": [0.7, 0.6, 0.5]}, {"type": "metal", "color": [0.8, 0.8, 0.8], "fuzz": 0.1},
            {"type": "glass", "ior": 1.5}]
    for k in range(n):
        m = mats[int(rng.integers(0, 3))]
        kind = rng.random()
        c = (rng.random(3) * 8 - 4).tolist()
        if kind < 0.6:
            objs.append({"type": "sphere", "pos": c, "r": float(10 ** rng.uniform(-1.5, 0.2)), "material": m})
        elif kind < 0.8:  # axis-aligned quad
            ax = int(rng.integers(0, 3))
            u, v = [0.0] * 3, [0.0] * 3
            u[(ax + 1) % 3] = float(rng.uniform(0.3, 3))
            v[(ax + 2) % 3] = float(rng.uniform(0.3, 3)) * (1 if rng.random() < 0.5 else -1)
            objs.append({"type": "quad", "pos": c, "u": u, "v": v, "material": m})
        elif kind < 0.97:  # rotated quad
            objs.append({"type": "quad", "pos": c, "u": (rng.random(3) * 2 - 1).tolist(), "v": (rng.random(3) * 2 - 1).tolist(), "material": m})
        else:
            objs.append({"type": "plane", "pos": [0, -4.5, 0], "u": [1, 0, 0.1 * float(rng.random())], "v": [0, 0.05 * float(rng.random()), 1], "material": m})
    if seed % 2 == 0:  # a ground sphere as large as the scene
        objs.append({"type": "sphere", "pos": [0, -1004, 0], "r": 1000, "material": mats[0]})
    return {"type": "custom", "camera": {"vfov": 60, "from": [0.3, 1.1, 9], "at": [0, 0, 0]}, "objects": objs}


@pytest.mark.parametrize("seed,n", [(1, 6), (2, 14), (3, 30), (4, 30), (5, 90), (6, 400), (7, 3000)])
@pytest.mark.parametrize("bvh", ["auto", "sah"])
def test_primary_hits_random_scenes(gpu, seed, n, bvh):
    sd = _random_scene(seed, n)
    opts = {"width": 256, "samples": 1, "bvh": bvh}
    with createCameraFromSceneData(sd, opts) as cam:
        ids, t, nrm, ff = cam.tracePrimary()
    oids, ot, onrm, off = ob.OracleCamera(sd, opts).trace_primary()
    assert np.array_equal(ids, oids), f"{int((ids != oids).sum())} primary-hit ids differ (seed {seed}, {n} objects, bvh {bvh})"
    hit = oids >= 0
    assert np.all(np.abs(t[hit] - ot[hit]) <= 1e-4 * np.abs(ot[hit]))
    assert np.all(np.abs(nrm[hit] - onrm[hit]) <= 2e-4)
    assert np.array_equal(ff[hit], off[hit])


def _degenerate_scenes():
    """Scenes no generator produces (scripts/gpu_degenerate.py has the longer list): (objects, eye)."""
    rng = np.random.default_rng(0)
    m = {"type": "lambert", "color": [0.7, 0.6, 0.5]}
    g = {"type": "glass", "ior": 1.5}
    sph = lambda p, r, mat=m: {"type": "sphere", "pos": [float(x) for x in p], "r": float(r), "material": mat}  # noqa: E731
    return {
        "coincident": ([sph([0, 0, 0], 1.0) for _ in range(200)], [0, 0, 5]),
        "nested": ([sph([0, 0, 0], 1 + i * 1e-2, g if i % 2 else m) for i in range(200)], [0, 0, 9]),
        "zero_radius": ([sph(rng.random(3) * 4 - 2, 0.0) for _ in range(200)] + [sph([0, 0, 0], 0.5)], [0, 0, 5]),
        "fp32_large": ([sph((rng.random(3) - 0.5) * 1e30, 1e29) for _ in range(200)], [0, 0, 2e30]),
        "fp32_tiny": ([sph((rng.random(3) - 0.5) * 1e-15, 1e-16) for _ in range(200)], [0, 0, 2e-15]),
        "zero_area_quads": ([{"type": "quad", "pos": (rng.random(3) * 2 - 1).tolist(), "u": [0, 0, 0], "v": [0, 0, 0], "material": m}
                             for _ in range(100)] + [sph([0, 0, 0], 0.5)], [0, 0, 5]),
        "inverted_boxes": ([sph(rng.random(3) * 4 - 2, -0.3, g) for _ in range(100)] + [sph([0, -101, 0], 100)], [0, 1, 7]),
    }


@pytest.mark.parametrize("name", ["coincident", "nested", "zero_radius", "fp32_large", "fp32_tiny", "zero_area_quads", "inverted_boxes"])
def test_primary_hits_degenerate_scenes(gpu, name):
    """Equal-t ties (which of 200 coincident spheres the reference keeps), FP32 overflow / underflow of the quick
    tests (the guarded FP64 re-test decides), zero-size primitives, the inverted boxes of negative radii."""
    objs, eye = _degenerate_scenes()[name]
    sd = {"type": "custom", "camera": {"vfov": 40, "from": eye, "at": [0, 0, 0], "focus": float(np.linalg.norm(eye))}, "objects": objs}
    # a forced SAH tree cannot reproduce the inverted-box quirk (DESIGN.md section 7): AUTO picks the reference topology there
    for bvh in ("auto", "reference") + (("sah",) if name != "inverted_boxes" else ()):
        opts = {"width": 64, "aspect": 16 / 9, "samples": 8, "depth": 12, "aTolerance": 0, "seed": 3, "bvh": bvh}
        with createCameraFromSceneData(sd, opts) as cam:
            ids, t, _nrm, _ff = cam.tracePrimary()
            rgb = np.zeros(cam.imageWidth * cam.imageHeight * 3, np.uint8)
            st = cam.render(rgb)
        oids, ot, _onrm, _off = ob.OracleCamera(sd, opts).trace_primary()
        assert np.array_equal(ids, oids), (name, bvh, int((ids != oids).sum()))
        hit = oids >= 0
        assert hit.any() and np.all(np.abs(t[hit] - ot[hit]) <= 1e-4 * np.abs(ot[hit])), (name, bvh)
        assert st.samples["total"] == st.pixels * 8  # the integrator terminates on every path


@pytest.mark.parametrize("seed,n", [(2, 14), (3, 30), (6, 400), (7, 3000)])
def test_integrators_agree_on_random_scenes(gpu, seed, n):
    """All integrator layouts and both tree choices walk the same paths: bit-identical images within a build."""
    sd = _random_scene(seed, n)
    opts = {"width": 120, "samples": 12, "aTolerance": 0, "seed": seed}
    ref = gpu_render(sd, {**opts, "integrator": "megakernel"})
    for integ in ("sorted", "wavefront"):
        other = gpu_render(sd, {**opts, "integrator": integ})
        assert np.array_equal(ref["linear"], other["linear"]), integ
        assert ref["stats"].rays == other["stats"].rays
    adaptive = {**opts, "samples": 40, "aTolerance": 0.05}
    a = gpu_render(sd, adaptive, want_moments=True)
    b = gpu_render(sd, {**adaptive, "partIndex": 0, "partCount": 1}, region={"x": 0, "y": 0, "width": 120, "height": 40})
    assert np.array_equal(a["rgb8"][:40], b["rgb8"][:40])


def test_primary_hits_full_size_C1(gpu):
    """BASELINE.json configs[0] at its full size (400x225)."""
    sd = SCENES["C1-spheres"]()
    opts = {"width": 400, "samples": 16, "depth": 10}
    with createCameraFromSceneData(sd, opts) as cam:
        assert (cam.imageWidth, cam.imageHeight) == (400, 225)
        ids, t, nrm, _ = cam.tracePrimary()
    oids, ot, onrm, _ = ob.OracleCamera(sd, opts).trace_primary()
    assert np.array_equal(ids, oids)
    hit = oids >= 0
    assert np.all(np.abs(t[hit] - ot[hit]) <= 1e-4 * np.abs(ot[hit]))


def test_primary_hits_match_committed_golden(gpu):
    """Against the committed fixture (tests/golden/primary_*.npz, made by tests/golden/make_golden.py)."""
    for name in ("C2-cornell", "default"):
        f = np.load(os.path.join(GOLDEN, f"primary_{name}.npz"))
        sd = SCENES[name]()
        with createCameraFromSceneData(sd, {"width": int(f["width"]), "samples": 1}) as cam:
            ids, t, nrm, _ = cam.tracePrimary()
        assert np.array_equal(ids, f["ids"])
        hit = f["ids"] >= 0
        assert np.all(np.abs(t[hit] - f["t"][hit]) <= 1e-4 * np.abs(f["t"][hit]))
        assert np.all(np.abs(nrm[hit] - f["normal"][hit]) <= 2e-4)


def test_camera_block_matches_oracle(gpu):
    for name in ("C2-cornell", "C3-weekend", "default"):
        sd = SCENES[name]()
        opts = {"width": 320, "samples": 4}
        oc = ob.OracleCamera(sd, opts)
        with createCameraFromSceneData(sd, opts) as cam:
            assert (cam.imageWidth, cam.imageHeight) == (oc.imageWidth, oc.imageHeight)
            for a, b in ((cam.center, oc.center), (cam.pixel00Loc, oc.pixel00Loc), (cam.pixelDeltaU, oc.pixelDeltaU),
                         (cam.pixelDeltaV, oc.pixelDeltaV), (cam.u, oc.u), (cam.v, oc.v), (cam.w, oc.w),
                         (cam.defocusDiskU, oc.defocusDiskU), (cam.defocusDiskV, oc.defocusDiskV)):
                assert np.array_equal(a, b)  # bit-exact FP32
            assert cam.focusDistance == oc.focusDistance
            assert cam.nLights == oc.n_lights


# ------------------------------------------------------------------------------------------
# same random streams: GPU paths and oracle paths see the same numbers
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,width,spp", [("C2-cornell", 96, 64), ("C1-spheres", 160, 32), ("C5-layered", 96, 64), ("default", 128, 48), ("C3-weekend", 160, 32)])
def test_same_seed_render_agrees_per_pixel(gpu, name, width, spp):
    sd = SCENES[name]()
    opts = {"width": width, "samples": spp, "aTolerance": 0, "seed": 11}
    g = gpu_render(sd, opts)
    o = ob.OracleCamera(sd, opts).render(seed=11, threads=8)
    gs, os_ = g["stats"], o["stats"]
    assert gs.pixels == os_.pixels and gs.samples["total"] == os_.samples_total
    assert gs.samples["min"] == os_.samples_min and gs.samples["max"] == os_.samples_max
    # FP32 vs FP64-scalar arithmetic flips a branch on a tiny fraction of paths; everything
    # else follows the identical path, so totals agree far inside statistical noise
    assert abs(gs.bounces["total"] - os_.bounces_total) <= 0.005 * os_.bounces_total + 50
    assert abs(gs.rays - os_.rays) <= 0.005 * os_.rays + 50
    d = np.abs(g["linear"].astype(np.float64) - o["linear"].astype(np.float64))
    scale = np.maximum(o["linear"].astype(np.float64), 0.05)
    frac_close = float(np.mean((d / scale) < 0.02))
    assert frac_close > 0.97, f"only {frac_close:.3f} of channels within 2% of the oracle"
    assert abs(float(g["linear"].mean()) - float(o["linear"].mean())) < 0.01 * float(o["linear"].mean()) + 1e-4
    # gamma + quantisation of identical colours is identical (camera.ts:455-472)
    same = d.max(axis=2) == 0
    assert np.array_equal(g["rgb8"][same], o["rgb8"][same])
    assert float(np.mean(np.abs(g["rgb8"].astype(int) - o["rgb8"].astype(int)) <= 2)) > 0.97


# ------------------------------------------------------------------------------------------
# independent random streams: the statistical bar of the north star
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,width,spp", [("C2-cornell", 64, 1024), ("C1-spheres", 96, 1024), ("C5-layered", 48, 1024)])
def test_converged_image_rmse_and_3sigma(gpu, name, width, spp):
    """The quick version of tests/test_gpu_full_parity.py (which runs the same statistics at BASELINE sizes): small images,
    oracle at twice the samples.  Every asserted number is raw — nothing is subtracted (tests/parity_stats.py); with only
    ~10 k channels the tail fractions are themselves noisy, hence the firefly allowance."""
    sd = SCENES[name]()
    opts = {"width": width, "aTolerance": 0}
    g = gpu_render(sd, {**opts, "samples": spp, "seed": 1}, want_moments=True)
    o = ob.OracleCamera(sd, {**opts, "samples": 2 * spp}).render(seed=2, threads=8, want_moments=True)
    g_var = g["moments"][..., 3:6].astype(np.float64) / (spp - 1.0)  # sum of squared deviations from the mean (rt_b200.h)
    o_mean, o_var = pstat.moments_to_mean_var(o["moments"], float(2 * spp))
    r = pstat.compare_converged(g["linear"], g_var, spp, o_mean, o_var, 2 * spp)
    assert r["rel_rmse_raw"] <= 1.10 * r["rel_rmse_noise_floor"] + 1e-6, r
    assert r["frac_within_3sigma"] >= 0.9973 - 0.005 and r["frac_within_4sigma"] >= 0.999, r
    assert 0.85 <= r["z2_mean"] <= 1.2, r
    assert r["rel_rmse_block"]["8"] <= 0.01, r
    for a, b in zip(r["mean_gpu"], r["mean_oracle"]):
        assert abs(a - b) <= 0.01 * abs(b) + 1e-6, r
    assert r["quiet_max_excess"] <= 0.0 and r["gpu_nonfinite_pixels"] == 0, r
    # RGB8 after gamma: the two images differ by Monte-Carlo noise only.  d(255.999*sqrt(c)) = 128*dc/sqrt(c), so compare
    # the mean level difference with what the measured sigma predicts.
    sigma = np.sqrt(g_var / spp + o_var / (2 * spp))
    expected = 128.0 * np.sqrt(2 / np.pi) * sigma / np.sqrt(np.maximum(o_mean, 1e-3))
    got = np.abs(g["rgb8"].astype(int) - o["rgb8"].astype(int))
    assert float(np.mean(got)) <= 1.5 * float(np.mean(expected)) + 0.5


def test_white_furnace_energy(gpu):
    """Analytic check that pins BOTH sides (SURVEY.md §8c): inside a closed emissive-free sphere of
    albedo a lit by a uniform background seen through nothing — here: an open scene with a
    constant background L and one Lambertian sphere of albedo a: every path that escapes carries
    a^k L, so the radiance of a camera ray that hits the sphere lies in (0, L] and a miss is L."""
    sd = {
        "camera": {"vfov": 40, "from": [0, 0, 3], "at": [0, 0, 0], "up": [0, 1, 0], "aperture": 0, "focus": 1,
                   "background": {"type": "gradient", "top": [0.5, 0.5, 0.5], "bottom": [0.5, 0.5, 0.5]}},
        "materials": [{"id": "m", "material": {"type": "lambert", "color": [1.0, 1.0, 1.0]}}],
        "objects": [{"type": "sphere", "pos": [0, 0, 0], "r": 1.0, "material": "m"}],
    }
    opts = {"width": 48, "aspect": 1.0, "samples": 256, "aTolerance": 0, "roulette": False, "depth": 64}
    g = gpu_render(sd, opts)
    # albedo 1, convex object, constant environment: every pixel converges to exactly L
    assert np.allclose(g["linear"], 0.5, atol=2e-3)


# ------------------------------------------------------------------------------------------
# regions, partitions, determinism
# ------------------------------------------------------------------------------------------
def test_render_is_deterministic_and_seeded(gpu):
    sd = SCENES["C2-cornell"]()
    a = gpu_render(sd, {"width": 64, "samples": 8, "aTolerance": 0, "seed": 5})
    b = gpu_render(sd, {"width": 64, "samples": 8, "aTolerance": 0, "seed": 5})
    c = gpu_render(sd, {"width": 64, "samples": 8, "aTolerance": 0, "seed": 6})
    assert np.array_equal(a["linear"], b["linear"]) and np.array_equal(a["rgb8"], b["rgb8"])
    assert not np.array_equal(a["linear"], c["linear"])


def test_bench_dump_outputs_are_what_the_public_api_renders(gpu, tmp_path):
    """bench.py --dump-outputs writes the framebuffer and statistics of its last timed step: the image and the statistics
    Camera.render gives for the same workload and options, after exactly --steps timed steps."""
    import subprocess
    import sys

    bench = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py")
    cmd = [sys.executable, bench, "--steps", "2", "--warmup", "1", "--samples", "16", "--width", "96", "--no-cpu-baseline",
           "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, timeout=600, check=True).stdout.decode()
    line = json.loads(out.strip().splitlines()[-1])
    assert line["steps"] == 2 and len(line["step_ms"]) == 2
    g = gpu_render(SCENES["C2-cornell"](), {"width": 96, "samples": 16, "aTolerance": 0})
    assert np.array_equal(np.load(tmp_path / "C2_image.npy"), g["rgb8"].astype(np.float32))
    s = g["stats"]
    assert np.load(tmp_path / "C2_stats.npy").tolist() == [s.pixels, s.samples["total"], s.samples["min"], s.samples["max"],
                                                          s.bounces["total"], s.bounces["min"], s.bounces["max"], s.rays]


def test_region_writes_only_region_pixels(gpu):  # camera.ts:388-431, camera.test.ts:381-396
    sd = SCENES["C2-cornell"]()
    opts = {"width": 80, "samples": 4, "aTolerance": 0, "seed": 3}
    full = gpu_render(sd, opts)
    with createCameraFromSceneData(sd, opts) as cam:
        buf = np.full((cam.imageHeight, cam.imageWidth, 3), 77, np.uint8)
        st = cam.renderRegion(buf, {"x": 10, "y": 20, "width": 30, "height": 25})
        assert st.pixels == 30 * 25 and st.samples["total"] == 30 * 25 * 4
        inside = np.zeros(buf.shape[:2], bool)
        inside[20:45, 10:40] = True
        assert np.all(buf[~inside] == 77)
        assert np.array_equal(buf[inside], full["rgb8"][inside])  # RNG keyed by global pixel index
        st = cam.renderRegion(buf, {"x": 70, "y": 70, "width": 30, "height": 30})  # clipped (camera.ts:390-391)
        assert st.pixels == 100
        st = cam.renderRegion(buf, {"x": 200, "y": 0, "width": 10, "height": 10})
        assert st.pixels == 0 and st.samples["min"] == float("inf")


@pytest.mark.parametrize("parts", [2, 3, 8])
def test_tile_partition_union_equals_whole_image(gpu, parts):
    """The multi-GPU partition (interleaved 16x16 tiles) rendered part by part on one GPU."""
    sd = SCENES["C2-cornell"]()
    opts = {"width": 100, "samples": 4, "aTolerance": 0, "seed": 9}
    whole = gpu_render(sd, opts)
    H, W = whole["rgb8"].shape[:2]
    buf = np.zeros((H, W, 3), np.uint8)
    stats = []
    for k in range(parts):
        with createCameraFromSceneData(sd, {**opts, "partIndex": k, "partCount": parts}) as cam:
            stats.append(cam.render(buf))
    assert np.array_equal(buf, whole["rgb8"])
    m = RenderStats.merge(stats)
    ws = whole["stats"]
    assert (m.pixels, m.samples["total"], m.bounces["total"], m.rays) == (ws.pixels, ws.samples["total"], ws.bounces["total"], ws.rays)
    assert (m.bounces["min"], m.bounces["max"]) == (ws.bounces["min"], ws.bounces["max"])


def test_row_strip_regions_like_the_reference_workers(gpu):  # raytracer.ts:185-205
    from mcp_raytracer_b200 import divideIntoRegions

    sd = SCENES["C1-spheres"]()
    opts = {"width": 120, "samples": 2, "aTolerance": 0}
    whole = gpu_render(sd, opts)
    with createCameraFromSceneData(sd, opts) as cam:
        buf = np.zeros((cam.imageHeight, cam.imageWidth, 3), np.uint8)
        stats = [cam.renderRegion(buf, r) for r in divideIntoRegions(cam.imageWidth, cam.imageHeight, 7)]
    assert np.array_equal(buf, whole["rgb8"])
    assert RenderStats.merge(stats).pixels == whole["stats"].pixels


# ------------------------------------------------------------------------------------------
# adaptive sampling, render modes, depth / roulette options
# ------------------------------------------------------------------------------------------
def test_adaptive_sampling_matches_oracle(gpu):  # camera.ts:348-368, :406
    sd = SCENES["C1-spheres"]()
    opts = {"width": 160, "samples": 100, "aTolerance": 0.05, "aBatch": 10, "seed": 4}
    g = gpu_render(sd, opts)
    o = ob.OracleCamera(sd, opts).render(seed=4, threads=8)
    gs, os_ = g["stats"], o["stats"]
    assert gs.samples["min"] == os_.samples_min == 10       # flat background pixels stop at aBatch
    assert gs.samples["max"] == os_.samples_max
    assert abs(gs.samples["total"] - os_.samples_total) <= 0.01 * os_.samples_total
    assert gs.samples["total"] < 0.8 * gs.pixels * 100      # adaptive exit really saves samples


@pytest.mark.parametrize("name,bvh", [("C2-cornell", "auto"), ("C3-weekend", "auto"), ("C4-rain", "auto"), ("default", "reference")])
def test_adaptive_pixel_stream_regions_and_partitions(gpu, name, bvh):
    """k_render_stream hands pixels to lanes in scheduling order; a pixel's samples stay in one lane and in order, so
    the image and the per-pixel sample counts cannot depend on regions, partitions or which lane ran what."""
    sd = SCENES[name]()
    opts = {"width": 150, "samples": 48, "aTolerance": 0.05, "aBatch": 10, "seed": 8, "bvh": bvh}
    whole = gpu_render(sd, opts, want_moments=True)
    H, W = whole["rgb8"].shape[:2]
    n = whole["moments"][..., 6]
    assert n.min() >= 10 and n.max() <= 48 and float(n.sum()) == whole["stats"].samples["total"]
    assert np.array_equal(gpu_render(sd, opts)["rgb8"], whole["rgb8"])  # deterministic
    # 3-way tile partition inside a ragged region
    reg = {"x": 7, "y": 9, "width": W - 20, "height": H - 15}
    buf = np.full((H, W, 3), 77, np.uint8)
    px = samples = 0
    for k in range(3):
        with createCameraFromSceneData(sd, {**opts, "partIndex": k, "partCount": 3}) as cam:
            st = cam.renderRegion(buf, reg)
            px += st.pixels
            samples += st.samples["total"]
    inside = np.zeros((H, W), bool)
    inside[reg["y"]:reg["y"] + reg["height"], reg["x"]:reg["x"] + reg["width"]] = True
    assert px == int(inside.sum()) and samples == int(n[inside].sum())
    assert np.all(buf[~inside] == 77) and np.array_equal(buf[inside], whole["rgb8"][inside])


@pytest.mark.parametrize("name,opts", [
    ("C2-cornell", {"width": 160, "samples": 200}),                                   # LIST, groups of 4 blocks
    ("C2-cornell", {"width": 96, "samples": 50, "aBatch": 7}),                        # last batch shorter than aBatch
    ("C1-spheres", {"width": 200, "samples": 100}),                                   # SAH whole-query walk, most pixels stop at 10
    ("C3-weekend", {"width": 160, "samples": 60, "aTolerance": 0.02}),
    ("C5-layered", {"width": 96, "samples": 64, "aBatch": 40}),                       # one block per group (record slice)
    ("default", {"width": 120, "samples": 40, "bvh": "reference"}),
    ("C2-cornell", {"width": 64, "samples": 90, "aBatch": 41}),                       # aBatch too large for a record slice: the stream kernel renders it
])
def test_batch_parallel_adaptive_kernel_equals_the_pixel_stream(gpu, name, opts):
    """k_render_adaptive (plain adaptive renders) deals a pixel's batch out over the lanes of a warp and adds the samples back
    in order: image, sample counts and statistics are those of k_render_stream (which renders when moments are asked for)."""
    sd = SCENES[name]()
    opts = {"aTolerance": 0.05, "aBatch": 10, "seed": 31, **opts}
    a = gpu_render(sd, opts)
    b = gpu_render(sd, opts, want_moments=True)
    assert np.array_equal(a["linear"], b["linear"]) and np.array_equal(a["rgb8"], b["rgb8"])
    sa, sb = a["stats"], b["stats"]
    assert (sa.pixels, sa.samples, sa.bounces, sa.rays) == (sb.pixels, sb.samples, sb.bounces, sb.rays)
    assert sa.samples["min"] < sa.samples["max"] or name == "C5-layered"     # the exit rule is really exercised
    # a ragged region: the same pixels
    H, W = a["rgb8"].shape[:2]
    reg = {"x": 5, "y": 3, "width": W - 11, "height": H - 9}
    c = gpu_render(sd, opts, region=reg)
    ys, xs = slice(reg["y"], reg["y"] + reg["height"]), slice(reg["x"], reg["x"] + reg["width"])
    assert np.array_equal(c["linear"][ys, xs], a["linear"][ys, xs])


def test_zero_samples_gives_black_image(gpu):  # while (pixel.samples < 0) never runs: colour/0 -> NaN -> 0 (camera.ts:406, :455-472)
    g = gpu_render(SCENES["C2-cornell"](), {"width": 40, "samples": 0})
    assert g["stats"].pixels == 1600 and g["stats"].samples["total"] == 0
    assert not g["rgb8"].any()


@pytest.mark.parametrize("integrator", ["auto", "sorted", "megakernel", "wavefront"])
@pytest.mark.parametrize("name", ["C5-layered", "C1-spheres"])
def test_zero_samples_every_integrator(gpu, name, integrator, monkeypatch):
    """AUTO picks the sorted kernel for Mixed/Layered scenes; an image with no samples is black there too, every pixel is
    written and counted (stale device memory of a recycled buffer must not leak out), also with more chunks than samples."""
    sd = SCENES[name]()
    gpu_render(sd, {"width": 64, "samples": 8, "aTolerance": 0, "integrator": integrator})  # leaves a non-black image in the cache
    g = gpu_render(sd, {"width": 64, "samples": 0, "integrator": integrator})
    H, W = g["rgb8"].shape[:2]
    assert g["stats"].pixels == W * H and g["stats"].samples["total"] == 0 and not g["rgb8"].any()
    monkeypatch.setenv("RT_B200_CHUNKS", "16")
    a = gpu_render(sd, {"width": 64, "samples": 3, "aTolerance": 0, "integrator": integrator})
    monkeypatch.delenv("RT_B200_CHUNKS")
    b = gpu_render(sd, {"width": 64, "samples": 3, "aTolerance": 0, "integrator": integrator})
    assert a["stats"].pixels == W * H and np.array_equal(a["rgb8"], b["rgb8"])


def test_render_modes(gpu):  # camera.ts:326-340
    sd = SCENES["C1-spheres"]()
    base = {"width": 96, "samples": 40, "aTolerance": 0.05, "seed": 2}
    for mode in ("bounces", "samples"):
        g = gpu_render(sd, {**base, "mode": mode})
        o = ob.OracleCamera(sd, {**base, "mode": mode}).render(seed=2, threads=8)
        lin, olin = g["linear"], o["linear"]
        if mode == "bounces":
            assert np.all(lin[..., 0] == 0) and np.all(lin[..., 1] == 0)
            assert abs(float(lin[..., 2].mean()) - float(olin[..., 2].mean())) < 0.02 * float(olin[..., 2].mean()) + 1e-4
        else:
            assert np.all(lin[..., 1] == 0) and np.all(lin[..., 2] == 0)
            assert float(np.mean(lin[..., 0] == olin[..., 0])) > 0.97
        assert float(np.mean(np.abs(g["rgb8"].astype(int) - o["rgb8"].astype(int)) <= 1)) > 0.97


def test_depth_limit_and_roulette_options(gpu):  # camera.ts:228-245, camera.test.ts:591-655
    sd = SCENES["C2-cornell"]()
    a = gpu_render(sd, {"width": 48, "samples": 16, "aTolerance": 0, "depth": 3, "roulette": False})["stats"]
    assert a.bounces["max"] <= 3
    b = gpu_render(sd, {"width": 48, "samples": 16, "aTolerance": 0, "depth": 30, "roulette": False})["stats"]
    c = gpu_render(sd, {"width": 48, "samples": 16, "aTolerance": 0, "depth": 30, "roulette": True, "rouletteDepth": 3})["stats"]
    assert c.bounces["total"] < b.bounces["total"] and b.bounces["max"] <= 30
    d = gpu_render(sd, {"width": 48, "samples": 1, "aTolerance": 0})["stats"]  # samples == 1: no jitter (camera.ts:184)
    assert d.samples["total"] == d.pixels


def test_stats_10x10_one_sample(gpu):  # camera.test.ts:332-357
    sd = SCENES["C1-spheres"]()
    st = gpu_render(sd, {"width": 10, "aspect": 1.0, "samples": 1})["stats"]
    assert (st.pixels, st.samples["total"], st.samples["min"], st.samples["max"], st.samples["avg"]) == (100, 100, 1, 1, 1)


def test_output_dimensions_like_raytracer_tests(gpu):  # raytracer.test.ts:38-173
    for width, aspect, (W, H) in ((10, 1.0, (10, 10)), (8, 2.0, (8, 4)), (16, 1.0, (16, 16)), (20, 2.0, (20, 10)), (30, 1.5, (30, 20))):
        rgb, st = renderScene({"type": "default", "render": {"width": width, "aspect": aspect, "samples": 2}})
        assert rgb.shape == (H, W, 3) and st.pixels == W * H
    rgb, st = renderScene({"type": "spheres", "options": {"count": 5, "seed": 3}, "render": {"width": 12, "aspect": 1.0, "samples": 2}},
                          {"parallel": True, "threads": 2})
    assert rgb.shape == (12, 12, 3) and st.pixels == 144


# ------------------------------------------------------------------------------------------
# error behaviour through the C ABI (scenes.ts:137,154,178,191,195; raytracer.ts:97-99)
# ------------------------------------------------------------------------------------------
def test_c_abi_error_codes(gpu):
    L = _native.lib()
    sd = SCENES["C2-cornell"]()
    fs = FlatScene(sd)
    opts = render_opts_struct(merge_render_options(sd.get("render"), {"width": 32, "samples": 1}))
    h = C.c_void_p()
    assert L.rt_camera_create(None, C.byref(opts), C.byref(h)) == 1
    fs.obj_type[0] = 9
    assert L.rt_camera_create(C.byref(fs.desc), C.byref(opts), C.byref(h)) == 2 and b"Unknown object type" in L.rt_last_error()
    fs.obj_type[0] = 2
    fs.mat_type_a[0] = 17
    assert L.rt_camera_create(C.byref(fs.desc), C.byref(opts), C.byref(h)) == 3 and b"Unknown material type" in L.rt_last_error()
    fs.mat_type_a[0] = 0
    fs.obj_material[0] = 99
    assert L.rt_camera_create(C.byref(fs.desc), C.byref(opts), C.byref(h)) == 4 and b"Material not found" in L.rt_last_error()
    fs.obj_material[0] = 0
    assert L.rt_camera_create(C.byref(fs.desc), C.byref(opts), C.byref(h)) == 0
    small = np.zeros(10, np.uint8)
    from mcp_raytracer_b200.scene_data import rt_stats
    st = rt_stats()
    assert L.rt_camera_render(h, small.ctypes.data, small.nbytes, None, C.byref(st)) == 6  # buffer too small
    assert L.rt_camera_destroy(h) == 0
    with pytest.raises(RaytracerError, match="Material is not a dielectric"):
        bad = generateDefaultSceneData()
        bad["materials"][5]["material"]["outer"] = {"type": "lambert", "color": [1, 1, 1]}
        createCameraFromSceneData(bad, {"width": 16})


# ------------------------------------------------------------------------------------------
# the two integrators: same arithmetic, same Philox streams, exact fixed-point sums
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,width,spp", [("C2-cornell", 200, 24), ("C1-spheres", 240, 16), ("C5-layered", 160, 16), ("C4-rain", 320, 8), ("default", 200, 16)])
def test_wavefront_integrator_equals_megakernel(gpu, name, width, spp):
    sd = SCENES[name]()
    opts = {"width": width, "samples": spp, "aTolerance": 0, "seed": 21}
    a = gpu_render(sd, {**opts, "integrator": "megakernel"})
    b = gpu_render(sd, {**opts, "integrator": "wavefront"})
    assert b["stats"].kernelLaunches > 3  # generate / extend / shade per tag / resolve really ran
    assert np.array_equal(a["rgb8"], b["rgb8"]) and np.array_equal(a["linear"], b["linear"])
    sa, sb = a["stats"], b["stats"]
    assert (sa.pixels, sa.samples, sa.bounces, sa.rays) == (sb.pixels, sb.samples, sb.bounces, sb.rays)


@pytest.mark.parametrize("name,width,spp,bvh", [("C2-cornell", 200, 40, "auto"), ("C5-layered", 160, 24, "auto"), ("C1-spheres", 240, 16, "sah"),
                                                ("default", 200, 16, "auto"), ("C4-rain", 160, 4, "auto")])
def test_sorted_integrator_equals_megakernel(gpu, name, width, spp, bvh):
    """CTA-wide sort of the hits by material class (k_render_sorted): other threads run the samples, same image.
    C4 has no sorted kernel (deep tree) and must fall back to the plain megakernel."""
    sd = SCENES[name]()
    opts = {"width": width, "samples": spp, "aTolerance": 0, "seed": 5, "bvh": bvh}
    a = gpu_render(sd, {**opts, "integrator": "megakernel"})
    b = gpu_render(sd, {**opts, "integrator": "sorted"})
    assert np.array_equal(a["rgb8"], b["rgb8"]) and np.array_equal(a["linear"], b["linear"])
    sa, sb = a["stats"], b["stats"]
    assert (sa.pixels, sa.samples, sa.bounces, sa.rays) == (sb.pixels, sb.samples, sb.bounces, sb.rays)
    # region + 3-way partition through the sorted kernel
    H, W = a["rgb8"].shape[:2]
    buf = np.full((H, W, 3), 77, np.uint8)
    reg = {"x": 11, "y": 5, "width": W // 2 + 1, "height": H // 2 + 3}
    for k in range(3):
        with createCameraFromSceneData(sd, {**opts, "integrator": "sorted", "partIndex": k, "partCount": 3}) as cam:
            cam.renderRegion(buf, reg)
    inside = np.zeros((H, W), bool)
    inside[reg["y"]:reg["y"] + reg["height"], reg["x"]:reg["x"] + reg["width"]] = True
    assert np.all(buf[~inside] == 77) and np.array_equal(buf[inside], a["rgb8"][inside])


@pytest.mark.parametrize("name,opts", [
    ("C1-spheres", {"width": 400, "samples": 16, "depth": 10}),          # whole-query walk (k_render_pool<SAH>)
    ("C3-weekend", {"width": 320, "samples": 24}),                        # ... with the ground sphere in the always-tested prefix
    ("C4-rain", {"width": 320, "samples": 6}),                            # 20 k spheres: resumable traversal (k_render_trav)
])
def test_sah_walk_gives_the_image_of_the_reference_topology_walk(gpu, name, opts):
    """The 4-wide SAH nodes hold (centre, half-extent) boxes with the half-extents rounded up and are tested with a slab test of
    their own; the reference-topology tree holds the true min / max boxes.  Both walks decide every hit with the same primitive
    tests, so with the same seed they must give the same image — unless a box test drops a box the ray enters."""
    sd = SCENES[name]()
    opts = {"aTolerance": 0, "seed": 5, **opts}
    a = gpu_render(sd, {**opts, "bvh": "sah"})
    b = gpu_render(sd, {**opts, "bvh": "reference"})
    assert (a["stats"].samples, a["stats"].rays, a["stats"].bounces) == (b["stats"].samples, b["stats"].rays, b["stats"].bounces)
    assert np.array_equal(a["linear"], b["linear"]) and np.array_equal(a["rgb8"], b["rgb8"])


def test_deep_tree_state_machine_kernel(gpu):
    """Big trees run k_render_trav (resumable traversal bursts interleaved with shading): same image as the
    wavefront integrator (its own extend kernel) and as the union of a 3-way partition; primary hits vs the oracle."""
    sd = generateRainSceneData({"count": 60000, "seed": 2, "sphereRadius": 0.012})
    opts = {"width": 160, "samples": 6, "aTolerance": 0, "seed": 13}
    with createCameraFromSceneData(sd, opts) as cam:
        assert cam.info.n_bvh_nodes > 16384 and cam.info.bvh_kind == 2
        ids, t, _, _ = cam.tracePrimary()
    a = gpu_render(sd, {**opts, "integrator": "megakernel"})
    b = gpu_render(sd, {**opts, "integrator": "wavefront"})
    assert np.array_equal(a["rgb8"], b["rgb8"]) and np.array_equal(a["linear"], b["linear"])
    assert (a["stats"].samples, a["stats"].bounces, a["stats"].rays) == (b["stats"].samples, b["stats"].bounces, b["stats"].rays)
    H, W = a["rgb8"].shape[:2]
    buf = np.zeros((H, W, 3), np.uint8)
    for k in range(3):
        with createCameraFromSceneData(sd, {**opts, "partIndex": k, "partCount": 3}) as cam:
            cam.render(buf)
    assert np.array_equal(buf, a["rgb8"])
    # primary visibility against the oracle walking the reference's own tree (≈ 1 s at this size)
    oids, ot, _, _ = ob.OracleCamera(sd, opts).trace_primary()
    assert np.array_equal(ids, oids)
    hit = oids >= 0
    assert np.all(np.abs(t[hit] - ot[hit]) <= 1e-4 * np.abs(ot[hit]))


def test_wavefront_region_and_partition(gpu):
    sd = SCENES["C2-cornell"]()
    opts = {"width": 100, "samples": 8, "aTolerance": 0, "seed": 9}
    whole = gpu_render(sd, {**opts, "integrator": "megakernel"})
    H, W = whole["rgb8"].shape[:2]
    buf = np.zeros((H, W, 3), np.uint8)
    for k in range(3):
        with createCameraFromSceneData(sd, {**opts, "integrator": "wavefront", "partIndex": k, "partCount": 3}) as cam:
            cam.render(buf)
    assert np.array_equal(buf, whole["rgb8"])
    with createCameraFromSceneData(sd, {**opts, "integrator": "wavefront"}) as cam:
        buf = np.full((H, W, 3), 77, np.uint8)
        st = cam.renderRegion(buf, {"x": 10, "y": 20, "width": 30, "height": 25})
        assert st.pixels == 750 and st.samples["total"] == 750 * 8
        inside = np.zeros((H, W), bool)
        inside[20:45, 10:40] = True
        assert np.all(buf[~inside] == 77) and np.array_equal(buf[inside], whole["rgb8"][inside])


def test_image_independent_of_chunking(gpu, monkeypatch):
    """Exact fixed-point radiance sums: the image must not depend on how samples are cut into chunks."""
    sd = SCENES["C2-cornell"]()
    opts = {"width": 96, "samples": 64, "aTolerance": 0, "seed": 4}
    imgs = []
    for k in ("1", "4", "16"):
        monkeypatch.setenv("RT_B200_CHUNKS", k)
        imgs.append(gpu_render(sd, opts))
    monkeypatch.delenv("RT_B200_CHUNKS")
    for im in imgs[1:]:
        assert np.array_equal(im["linear"], imgs[0]["linear"]) and np.array_equal(im["rgb8"], imgs[0]["rgb8"])


# ------------------------------------------------------------------------------------------
# device memory cache: create/destroy per image must not change results, trim gives memory back
# ------------------------------------------------------------------------------------------
def test_device_cache_reuse_and_trim(gpu):
    from mcp_raytracer_b200 import trimDeviceCache
    sd = SCENES["C2-cornell"]()
    opts = {"width": 96, "samples": 40, "aTolerance": 0, "seed": 3}  # 40 spp on a small image: chunked, uses the accumulator
    first = gpu_render(sd, opts)
    trimDeviceCache()
    for _ in range(3):  # buffers of the previous camera are handed out again (stale contents must not leak into the image)
        again = gpu_render(sd, opts)
        assert np.array_equal(first["rgb8"], again["rgb8"])
        other = gpu_render(SCENES["C1-spheres"](), {"width": 120, "samples": 4, "aTolerance": 0})
        assert other["stats"].pixels == other["rgb8"].shape[0] * other["rgb8"].shape[1]
    assert trimDeviceCache() > 0
    assert trimDeviceCache() == 0
    assert np.array_equal(first["rgb8"], gpu_render(sd, opts)["rgb8"])


# ------------------------------------------------------------------------------------------
# one process, N GPUs inside the C ABI (rt_multi_*): the worker pool of src/raytracer.ts:60-90
# ------------------------------------------------------------------------------------------
def _multi_devices():
    n = _native.lib().rt_device_count()
    return [1] + ([n] if n > 1 else [])


@pytest.mark.parametrize("name,opts", [("C2-cornell", {"width": 200, "samples": 24}), ("C5-layered", {"width": 120, "samples": 16}),
                                      ("C3-weekend", {"width": 200, "samples": 8}), ("C1-spheres", {"width": 160, "samples": 40, "aTolerance": 0.05})])
def test_multi_camera_image_equals_single_camera(gpu, name, opts, monkeypatch):
    """Every visible GPU (and the 1-GPU degenerate case): same bytes, same merged RenderStats as one Camera, through the
    peer-write path and through the host-merge fallback, whole image and a ragged region."""
    from mcp_raytracer_b200 import MultiCamera

    sd = SCENES[name]()
    opts = {"aTolerance": 0, "seed": 17, **opts}
    whole = gpu_render(sd, opts)
    H, W = whole["rgb8"].shape[:2]
    ws = whole["stats"]
    for n in _multi_devices():
        for no_p2p in (False, True):
            if no_p2p:
                monkeypatch.setenv("RT_B200_MULTI_NO_P2P", "1")
            else:
                monkeypatch.delenv("RT_B200_MULTI_NO_P2P", raising=False)
            with MultiCamera(sd, opts, nDevices=n) as mc:
                assert mc.nDevices == n and (mc.imageWidth, mc.imageHeight) == (W, H)
                assert mc.peerWrites == (not no_p2p) or n == 1 or not mc.peerWrites  # peer access may be unavailable on a box
                rgb = np.zeros((H, W, 3), np.uint8)
                lin = np.zeros((H, W, 3), np.float32)
                st = mc.render(rgb, lin)
                assert np.array_equal(rgb, whole["rgb8"]) and np.array_equal(lin, whole["linear"]), (n, no_p2p)
                assert (st.pixels, st.samples, st.bounces["total"], st.bounces["min"], st.bounces["max"], st.rays) == \
                       (ws.pixels, ws.samples, ws.bounces["total"], ws.bounces["min"], ws.bounces["max"], ws.rays)
                buf = np.full((H, W, 3), 77, np.uint8)
                reg = {"x": 9, "y": 6, "width": W // 2 + 3, "height": H // 2 + 1}
                st = mc.renderRegion(buf, reg)
                inside = np.zeros((H, W), bool)
                inside[reg["y"]:reg["y"] + reg["height"], reg["x"]:reg["x"] + reg["width"]] = True
                assert st.pixels == int(inside.sum())
                assert np.all(buf[~inside] == 77) and np.array_equal(buf[inside], whole["rgb8"][inside])
    monkeypatch.delenv("RT_B200_MULTI_NO_P2P", raising=False)


def test_multi_camera_errors_and_render_scene_parallel(gpu):
    from mcp_raytracer_b200 import MultiCamera

    sd = SCENES["C2-cornell"]()
    with pytest.raises(RaytracerError, match="device ordinal out of range"):
        MultiCamera(sd, {"width": 32}, devices=[0, 99])
    with pytest.raises(RaytracerError, match="device listed twice"):
        MultiCamera(sd, {"width": 32}, devices=[0, 0])
    bad = generateDefaultSceneData()
    bad["materials"][5]["material"]["outer"] = {"type": "lambert", "color": [1, 1, 1]}
    with pytest.raises(RaytracerError, match="Material is not a dielectric"):
        MultiCamera(bad, {"width": 16})
    # generateImageBuffer(parallel: true) -> all GPUs (raytracer.test.ts:150-173)
    cfg = {"type": "cornell", "render": {"width": 96, "samples": 8, "aTolerance": 0, "seed": 3}}
    a, sa = renderScene(cfg)
    b, sb = renderScene(cfg, {"parallel": True})
    assert np.array_equal(a, b) and sa.samples == sb.samples and sa.rays == sb.rays


def test_partition_blocks_follow_rt_block_owner(gpu):
    """A part renders exactly the pixels rt_block_owner gives it (the host-side mirror used to assemble images)."""
    from mcp_raytracer_b200.distributed import tile_owner_mask

    sd = SCENES["C2-cornell"]()
    opts = {"width": 100, "samples": 2, "aTolerance": 0, "seed": 2}
    for n, k in ((2, 1), (5, 3), (8, 0)):
        with createCameraFromSceneData(sd, {**opts, "partIndex": k, "partCount": n}) as cam:
            buf = np.full((cam.imageHeight, cam.imageWidth, 3), 77, np.uint8)
            lin = np.full((cam.imageHeight, cam.imageWidth, 3), -1.0, np.float32)
            st = cam.render(buf, lin)
            mask = tile_owner_mask(cam.imageWidth, cam.imageHeight, k, n)
            assert st.pixels == int(mask.sum())
            assert np.all(lin[~mask] == -1.0) and np.all(lin[mask] >= 0.0)


# ------------------------------------------------------------------------------------------
# progressive output (rt_camera_render_progressive): same image, delivered in growing prefixes of the samples
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,opts", [
    ("C2-cornell", {"width": 96, "samples": 50}),                                         # k_render_pool<LIST>
    ("C5-layered", {"width": 80, "samples": 24}),                                         # k_render_sorted
    ("C4-rain", {"width": 96, "samples": 9}),                                             # k_render_trav
    ("C1-spheres", {"width": 120, "samples": 100, "aTolerance": 0.05, "aBatch": 10}),     # adaptive: k_render_stream<SAH>
    ("C2-cornell", {"width": 96, "samples": 64, "aTolerance": 0.05, "aBatch": 8}),        # adaptive: k_render_stream<LIST>
    ("C4-rain", {"width": 96, "samples": 30, "aTolerance": 0.1, "aBatch": 10}),           # adaptive: k_render_stream_trav
    ("C1-spheres", {"width": 96, "samples": 12, "mode": "bounces"}),                      # render mode through the pixel stream
])
def test_progressive_render_ends_in_the_one_shot_image(gpu, name, opts):
    sd = SCENES[name]()
    opts = {"aTolerance": 0, "seed": 23, **opts}
    whole = gpu_render(sd, opts)
    H, W = whole["rgb8"].shape[:2]
    ws = whole["stats"]
    for passes in (1, 4, 7):
        seen = []
        with createCameraFromSceneData(sd, opts) as cam:
            rgb = np.zeros((H, W, 3), np.uint8)
            lin = np.zeros((H, W, 3), np.float32)
            first = {}

            def on_pass(k, n, cap, st, rgb=rgb, first=first):
                seen.append((k, n, cap, st.samples["total"]))
                if not first:
                    first["rgb"] = rgb.copy()
                    first["cap"] = cap
                return False

            st = cam.renderProgressive(rgb, passes, on_pass, linear=lin)
        assert np.array_equal(rgb, whole["rgb8"]) and np.array_equal(lin, whole["linear"]), (name, passes)
        assert (st.pixels, st.samples["total"], st.samples["min"], st.samples["max"]) == (ws.pixels, ws.samples["total"], ws.samples["min"], ws.samples["max"])
        assert (st.bounces["total"], st.bounces["min"], st.bounces["max"], st.rays) == (ws.bounces["total"], ws.bounces["min"], ws.bounces["max"], ws.rays)
        caps = [c for _, _, c, _ in seen]
        assert caps == sorted(set(caps)) and caps[-1] == opts["samples"] and len(seen) <= passes
        assert [t for *_, t in seen] == sorted(t for *_, t in seen)           # work only ever adds up
        if passes > 1 and not opts["aTolerance"] and opts.get("mode", "default") == "default" and first["cap"] > 1:
            # fixed spp: the preview after the first pass IS the render with that many samples (streams keyed by (pixel, sample))
            assert np.array_equal(first["rgb"], gpu_render(sd, {**opts, "samples": first["cap"]})["rgb8"])


def test_progressive_render_can_stop_early_and_refuses_partitions(gpu):
    sd = SCENES["C2-cornell"]()
    opts = {"width": 64, "samples": 40, "aTolerance": 0, "seed": 2}
    with createCameraFromSceneData(sd, opts) as cam:
        rgb = np.zeros((cam.imageHeight, cam.imageWidth, 3), np.uint8)
        calls = []
        st = cam.renderProgressive(rgb, 8, lambda k, n, cap, s: calls.append(cap) or len(calls) == 3)
        assert len(calls) == 3 and st.samples["max"] == calls[-1] == 15 and st.samples["total"] == st.pixels * 15
        assert np.array_equal(rgb, gpu_render(sd, {**opts, "samples": 15})["rgb8"])
        with pytest.raises(RuntimeError, match="boom"):
            cam.renderProgressive(rgb, 4, lambda *a: (_ for _ in ()).throw(RuntimeError("boom")))
        assert np.array_equal(gpu_render(sd, opts)["rgb8"], (cam.render(rgb), rgb)[1])   # the camera is still usable
    with createCameraFromSceneData(sd, {**opts, "partIndex": 0, "partCount": 2}) as cam:
        with pytest.raises(RaytracerError, match="not partitioned"):
            cam.renderProgressive(np.zeros((cam.imageHeight, cam.imageWidth, 3), np.uint8), 2)
