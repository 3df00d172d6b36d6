"""CPU-side checks of the boundary: the C-ABI library loads and exports every symbol
include/rt_b200.h declares (no compute without a GPU), fails loudly without a device, and the
multi-rank plumbing works over gloo with world_size 2."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from mcp_raytracer_b200 import _native

    hdr = open(os.path.join(ROOT, "include", "rt_b200.h")).read()
    declared = set(re.findall(r"\b(rt_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_native.EXPORTS), declared ^ set(_native.EXPORTS)
    lib = _native.lib()
    for s in declared:
        assert hasattr(lib, s), f"{s} not exported by {_native.LIB_PATH}"
    assert lib.rt_abi_version() == 2  # RT_B200_ABI_VERSION (round 2: rt_multi_*, rt_shared_buffer_*, rt_debug_*, rt_block_owner)
    out = subprocess.check_output(["nm", "-D", "--defined-only", _native.LIB_PATH]).decode()
    exported_rt = {l.split()[-1] for l in out.splitlines() if " T rt_" in l}
    assert declared <= exported_rt


def test_library_is_built_for_sm_100a():
    from mcp_raytracer_b200 import _native

    out = subprocess.check_output(["cuobjdump", "--list-elf", _native.LIB_PATH]).decode()
    assert "sm_100a" in out


def test_struct_layouts_match_the_header():
    """sizeof of every ctypes mirror equals the C compiler's (guards the ABI)."""
    from mcp_raytracer_b200 import scene_data as sd

    src = r'''
    #include <stdio.h>
    #include "rt_b200.h"
    int main(void){ printf("%zu %zu %zu %zu %zu %zu\n", sizeof(rt_camera_desc), sizeof(rt_scene_desc), sizeof(rt_render_opts),
                           sizeof(rt_region), sizeof(rt_stats), sizeof(rt_camera_info)); return 0; }'''
    exe = os.path.join("/tmp", f"rt_sizes_{os.getpid()}")
    subprocess.run(["gcc", "-x", "c", "-", "-I", os.path.join(ROOT, "include"), "-o", exe], input=src.encode(), check=True)
    sizes = [int(x) for x in subprocess.check_output([exe]).split()]
    os.remove(exe)
    mine = [C.sizeof(t) for t in (sd.rt_camera_desc, sd.rt_scene_desc, sd.rt_render_opts, sd.rt_region, sd.rt_stats, sd.rt_camera_info)]
    assert sizes == mine


def test_no_cpu_fallback_without_device():
    """On a box without a GPU the product path must fail loudly, never fall back."""
    from mcp_raytracer_b200 import RaytracerError, createCameraFromSceneData, generateCornellSceneData, _native

    if _native.lib().rt_device_count() > 0:
        pytest.skip("a CUDA device is visible")
    with pytest.raises(RaytracerError, match="no CPU fallback"):
        createCameraFromSceneData(generateCornellSceneData(), {"width": 16})


def test_render_output_arrays_are_checked_before_the_library_writes_them():
    """The library writes RGB8 and linear through their base pointers as C-contiguous [H][W][3]: every render method
    (Camera.renderRegion / renderProgressive / renderDenoised, MultiCamera.renderRegion / renderDenoised) refuses an
    array it would write past or around."""
    from mcp_raytracer_b200 import RaytracerError
    from mcp_raytracer_b200.camera import _image_outputs

    W, H = 5, 4
    rgb8, linear = np.zeros((H, W, 3), np.uint8), np.zeros((H, W, 3), np.float32)
    assert _image_outputs(rgb8, linear, W, H) == (rgb8.ctypes.data, rgb8.nbytes, linear.ctypes.data)
    assert _image_outputs(None, None, W, H) == (None, 0, None)
    with pytest.raises(RaytracerError, match="linear buffer"):  # a view with strides: writing it as contiguous corrupts it
        _image_outputs(None, np.zeros((H, 2 * W, 3), np.float32)[:, ::2], W, H)
    with pytest.raises(RaytracerError, match="linear buffer"):
        _image_outputs(None, np.zeros((H, W, 3), np.float32).transpose(1, 0, 2).copy(order="F"), W, H)
    with pytest.raises(RaytracerError, match="linear buffer"):
        _image_outputs(None, linear.astype(np.float64), W, H)
    with pytest.raises(RaytracerError, match="linear buffer"):
        _image_outputs(None, linear[:-1], W, H)
    with pytest.raises(RaytracerError, match="pixel buffer"):
        _image_outputs(rgb8[:, ::-1], None, W, H)
    with pytest.raises(RaytracerError, match="pixel buffer"):
        _image_outputs(rgb8.astype(np.int8), None, W, H)


def test_scene_errors_are_reported_before_device_checks():
    from mcp_raytracer_b200 import _native
    from mcp_raytracer_b200.scene_data import FlatScene, merge_render_options, render_opts_struct
    from mcp_raytracer_b200.scenes import generateCornellSceneData

    L = _native.lib()
    sd = generateCornellSceneData()
    fs = FlatScene(sd)
    opts = render_opts_struct(merge_render_options(sd.get("render"), {"width": 32}))
    h = C.c_void_p()
    fs.mat_child_a  # noqa: B018
    fs.obj_type[3] = 7
    assert L.rt_camera_create(C.byref(fs.desc), C.byref(opts), C.byref(h)) == 2
    assert b"Unknown object type" in L.rt_last_error()


def _mixed_scene(seed, n):
    """Seeded mix of spheres (tiny ... scene-sized), axis-aligned / rotated quads and an occasional infinite plane."""
    rng = np.random.default_rng(seed)
    m = {"type": "lambert", "color": [0.7, 0.6, 0.5]}
    objs = []
    for _ in range(n):
        kind = rng.random()
        c = (rng.random(3) * 8 - 4).tolist()
        if kind < 0.6:
            objs.append({"type": "sphere", "pos": c, "r": float(10 ** rng.uniform(-1.5, 0.2)), "material": m})
        elif kind < 0.8:
            ax = int(rng.integers(0, 3))
            u, v = [0.0] * 3, [0.0] * 3
            u[(ax + 1) % 3] = float(rng.uniform(0.3, 3))
            v[(ax + 2) % 3] = -float(rng.uniform(0.3, 3))
            objs.append({"type": "quad", "pos": c, "u": u, "v": v, "material": m})
        elif kind < 0.97:
            objs.append({"type": "quad", "pos": c, "u": (rng.random(3) * 2 - 1).tolist(), "v": (rng.random(3) * 2 - 1).tolist(), "material": m})
        else:
            objs.append({"type": "plane", "pos": [0, -4.5, 0], "u": [1, 0, 0.05], "v": [0, 0.02, 1], "material": m})
    if seed % 2 == 0:
        objs.append({"type": "sphere", "pos": [0, -1004, 0], "r": 1000, "material": m})
    return {"type": "custom", "camera": {"vfov": 60, "from": [0.3, 1.1, 9], "at": [0, 0, 0]}, "objects": objs}


def test_scene_compiler_structures_are_sound():
    """rt_scene_validate (host only): every object in exactly one slot, every leaf primitive inside its child box,
    every child box inside its parent's, for every acceleration structure the kernels walk — the 4-wide SAH tree
    with its always-tested prefix, the reference's own topology, the LIST."""
    from mcp_raytracer_b200 import (generateCornellSceneData, generateDefaultSceneData, generateLayeredMixedSceneData,
                                    generateRainSceneData, generateSpheresSceneData, generateWeekendFinalSceneData, validateScene)

    scenes = {
        "cornell": generateCornellSceneData(), "layered": generateLayeredMixedSceneData(), "default": generateDefaultSceneData(),
        "spheres": generateSpheresSceneData({"count": 100, "seed": 12345}), "weekend": generateWeekendFinalSceneData(),
        "rain": generateRainSceneData({"count": 50000, "seed": 1, "sphereRadius": 0.01}),
    }
    for seed, n in ((1, 5), (2, 14), (3, 40), (4, 300), (6, 5000)):
        scenes[f"mixed{seed}"] = _mixed_scene(seed, n)
    for name, sd in scenes.items():
        n_obj = len(sd["objects"])
        for bvh in ("auto", "sah", "reference") + (("list",) if n_obj <= 128 else ()):
            rep = validateScene(sd, {"bvh": bvh})
            assert rep["errors"] == 0, (name, bvh, rep)
            assert rep["n_slots"] == n_obj
            if rep["bvh_kind"] == 2:
                assert rep["max_depth"] <= 42 and rep["max_leaf_size"] <= 4
                assert rep["n_leaves"] + rep["n_prefix"] <= n_obj
            if rep["bvh_kind"] == 3:
                assert rep["n_prefix"] == n_obj and rep["n_node_slots"] == 0
    # the AUTO rules (include/rt_b200.h): room -> LIST, open scene beyond 16 objects -> SAH, negative radius -> REFERENCE
    assert validateScene(scenes["cornell"])["bvh_kind"] == 3
    assert validateScene(scenes["layered"])["bvh_kind"] == 3
    assert validateScene(scenes["spheres"])["bvh_kind"] == 2
    assert validateScene(scenes["default"])["bvh_kind"] == 1
    weekend = validateScene(scenes["weekend"])
    assert weekend["bvh_kind"] == 2 and weekend["n_prefix"] == 1  # the r = 1000 ground sphere is tested outside the tree
    assert validateScene(scenes["rain"])["n_prefix"] == 0        # big scenes keep everything in the tree


def test_reference_topology_matches_the_oracles_tree():
    """RT_BVH_REFERENCE flattens the reference's own median-split tree (bvh.ts:34-102): same depth as the tree the
    oracle builds from the reference's rules, and as many leaves as that (full binary) tree has leaf-holding nodes."""
    import oracle_binding as ob
    from mcp_raytracer_b200 import (generateCornellSceneData, generateDefaultSceneData, generateRainSceneData,
                                    generateSpheresSceneData, generateWeekendFinalSceneData, validateScene)

    scenes = [generateCornellSceneData(), generateDefaultSceneData(), generateSpheresSceneData({"count": 100, "seed": 12345}),
              generateWeekendFinalSceneData(), generateRainSceneData({"count": 5000, "seed": 1, "sphereRadius": 0.01})]
    scenes += [_mixed_scene(seed, n) for seed, n in ((1, 5), (2, 14), (3, 40), (4, 300), (6, 5000))]
    for sd in scenes:
        o = ob.OracleCamera(sd, {"width": 16, "samples": 1})
        rep = validateScene(sd, {"bvh": "reference"})
        assert rep["errors"] == 0 and rep["bvh_kind"] == 1
        assert rep["max_depth"] == o.bvh_depth, (len(sd["objects"]), rep, o.bvh_depth)
        assert rep["n_leaves"] == (o.bvh_nodes + 1) // 2, (len(sd["objects"]), rep, o.bvh_nodes)


def test_scene_compiler_survives_degenerate_scenes():
    """Inputs a JSON client can send and no generator produces: coincident / collinear / nested primitives (no
    centroid spread for the SAH bins), zero radii, zero-area quads, coordinates near the ends of the FP32 range
    (box areas overflow to inf), twenty decades of scale in one scene.  Every tree must still be sound."""
    from mcp_raytracer_b200 import validateScene

    rng = np.random.default_rng(0)
    m = {"type": "lambert", "color": [0.7, 0.6, 0.5]}
    sph = lambda p, r: {"type": "sphere", "pos": [float(x) for x in p], "r": float(r), "material": m}  # noqa: E731
    cases = {
        "coincident": [sph([1, 2, 3], 0.5) for _ in range(3000)],
        "collinear": [sph([i, 0, 0], 0.1) for i in range(3000)],
        "nested": [sph([0, 0, 0], 1 + i * 1e-3) for i in range(2000)],
        "zero_radius": [sph(rng.random(3), 0.0) for _ in range(500)],
        "fp32_max": [sph(rng.random(3) * 3e38, 1e37) for _ in range(500)],
        "fp32_tiny": [sph(rng.random(3) * 1e-30, 1e-35) for _ in range(500)],
        "scales": [sph(rng.random(3) * 10 ** rng.uniform(-20, 20), 10 ** rng.uniform(-20, 20)) for _ in range(2000)],
        "zero_area_quads": [{"type": "quad", "pos": rng.random(3).tolist(), "u": [0, 0, 0], "v": [0, 0, 0], "material": m}
                            for _ in range(200)],
        "inverted_boxes": [sph(rng.random(3) * 5, -0.1) for _ in range(300)],
    }
    for name, objs in cases.items():
        sd = {"type": "custom", "camera": {"vfov": 60, "from": [0.3, 1.1, 9], "at": [0, 0, 0]}, "objects": objs}
        for bvh in ("auto", "sah", "reference"):
            rep = validateScene(sd, {"bvh": bvh})
            assert rep["errors"] == 0 and rep["n_slots"] == len(objs), (name, bvh, rep)
            assert rep["max_depth"] <= (42 if rep["bvh_kind"] == 2 else 60), (name, bvh, rep)


def test_scene_validate_raises_the_reference_errors():
    from mcp_raytracer_b200 import RaytracerError, generateCornellSceneData, validateScene

    bad = generateCornellSceneData()
    bad["objects"][2]["material"] = "no-such-material"
    with pytest.raises(RaytracerError, match="Material not found"):
        validateScene(bad)
    bad = generateCornellSceneData()
    bad["objects"][0]["type"] = "torus"
    with pytest.raises(RaytracerError, match="Unknown object type"):
        validateScene(bad)
    # not in the reference (it would render NaN): geometry that is not finite in FP32 is refused, for every tree kind
    for field, value in (("pos", [0.0, 1e300, 0.0]), ("r", float("nan")), ("pos", [float("inf"), 0.0, 0.0])):
        for bvh in ("list", "sah", "reference"):
            bad = generateCornellSceneData()
            bad["objects"][6][field] = value
            with pytest.raises(RaytracerError, match="non-finite geometry"):
                validateScene(bad, {"bvh": bvh})
    bad = generateCornellSceneData()
    bad["objects"][0]["u"] = [0.0, float("inf"), 0.0]
    with pytest.raises(RaytracerError, match="non-finite geometry"):
        validateScene(bad)


def test_product_package_never_touches_the_oracle():
    """The oracle is the checker: nothing under the product package may import, link or open it."""
    pkg = os.path.join(ROOT, "mcp_raytracer_b200")
    for dp, _dn, fns in os.walk(pkg):
        for fn in fns:
            if fn.endswith((".py", ".cu", ".cuh", ".cpp", ".h", "Makefile")):
                txt = open(os.path.join(dp, fn), errors="replace").read()
                assert "oracle_binding" not in txt and "liboracle" not in txt and "oracle/" not in txt, os.path.join(dp, fn)


def test_tile_owner_mask_partitions_the_image():
    from mcp_raytracer_b200 import _native
    from mcp_raytracer_b200.distributed import tile_owner_mask

    for W, H, n in ((100, 70, 2), (1024, 1024, 8), (33, 17, 3)):
        total = np.zeros((H, W), int)
        for k in range(n):
            total += tile_owner_mask(W, H, k, n)
        assert np.all(total == 1)
    counts = [tile_owner_mask(1024, 1024, k, 8).sum() for k in range(8)]
    assert max(counts) - min(counts) <= 32  # every run of 8 blocks gives each part one: balanced to ONE 8x4 block
    # each part holds one block of every run of 8: any 64x4 strip aligned to a run is shared by all 8 parts
    m = np.stack([tile_owner_mask(1024, 1024, k, 8) for k in range(8)])
    assert np.all(m[:, 0:4, 0:64].reshape(8, -1).sum(axis=1) == 32)
    # no column or diagonal structure: the owner of block column 0 changes from block row to block row
    col0 = [int(np.argmax(m[:, y, 0])) for y in range(0, 1024, 4)]
    assert len(set(col0)) == 8 and max(np.bincount(col0)) < 60
    # the Python mirror is the C ABI's rule (rt_block_owner = rt::block_owner of the kernels), bit for bit
    L = _native.lib()
    rng = np.random.default_rng(0)
    for W, H, n in ((100, 70, 2), (1000, 700, 8), (33, 17, 3), (3840, 2160, 5)):
        owner = np.argmax(np.stack([tile_owner_mask(W, H, k, n) for k in range(n)]), axis=0)
        for _ in range(300):
            x, y = int(rng.integers(0, W)), int(rng.integers(0, H))
            assert L.rt_block_owner(x, y, W, n) == owner[y, x]


_WORKER = r'''
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from mcp_raytracer_b200.distributed import tile_owner_mask, gather_framebuffer, merge_stats
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
W, H = 100, 52
rng = np.random.default_rng(0)
whole = rng.integers(1, 255, (H, W, 3), dtype=np.uint8)          # what a 1-rank render would produce
mine = np.where(tile_owner_mask(W, H, rank, world)[..., None], whole, 0).astype(np.uint8)
t = gather_framebuffer(torch.from_numpy(mine.copy()))
sums = torch.tensor([int(tile_owner_mask(W, H, rank, world).sum()), 10 * (rank + 1)], dtype=torch.int64)
mins = torch.tensor([rank + 3], dtype=torch.int64); maxs = torch.tensor([rank + 7], dtype=torch.int64)
merge_stats(sums, mins, maxs)
from mcp_raytracer_b200.distributed import SharedFramebuffer
shared = SharedFramebuffer(W, H, device=0)     # no visible GPU: creation fails on rank 0 and EVERY rank learns to fall back
assert shared.ok is False and shared.ptr == 0
shared.close()
if rank == 0:
    assert np.array_equal(t.numpy(), whole), "gathered framebuffer differs"
    assert sums.tolist() == [W * H, 10 * sum(range(1, world + 1))] and mins.item() == 3 and maxs.item() == world + 6
    print("GATHER_OK")
dist.destroy_process_group()
'''


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU port of the reference, no GPU involved): exactly one JSON line on stdout
    with the keys the driver reads; under a 2-process launch only rank 0 prints."""
    import json

    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-seconds", "1"]
    for extra in ([], ["--gpus", "2"]):
        out = subprocess.run(cmd + extra, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, timeout=300, check=True).stdout.decode()
        lines = [l for l in out.splitlines() if l.strip()]
        assert len(lines) == 1, out
        d = json.loads(lines[0])
        assert d["impl"] == "reference" and d["metric"] == "Mpaths/s" and d["unit"] == "Mpaths/s" and d["higher_is_better"] is True
        assert d["value"] > 0 and d["steps"] == 1 and d["n_gpus"] == (2 if extra else 1)
        assert "cornell" in d["config"]["workload"] and "model" not in d["config"]
        assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
        assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]


def test_bench_dump_outputs_fit_the_budget_and_are_deterministic(tmp_path):
    """bench.dump_outputs: the whole image when its float32 copy fits, else the same seeded sample of pixels on every run."""
    import bench

    rng = np.random.default_rng(1)
    small = rng.integers(0, 256, (30, 40, 3), dtype=np.uint8)
    bench.dump_outputs(str(tmp_path / "a"), "C2", small, [1200, 4800, 4, 4, 9000, 1, 7, 13800], 64_000_000)
    assert np.array_equal(np.load(tmp_path / "a" / "C2_image.npy"), small.astype(np.float32))
    st = np.load(tmp_path / "a" / "C2_stats.npy")
    assert st.dtype == np.float64 and st.tolist() == [1200, 4800, 4, 4, 9000, 1, 7, 13800]
    big = rng.integers(0, 256, (300, 400, 3), dtype=np.uint8)
    budget = 300 * 400 * 3 * 4 // 2
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), "C4", big, [0] * 8, budget)
        assert sum(f.stat().st_size for f in (tmp_path / d).iterdir()) <= budget
        assert not (tmp_path / d / "C4_image.npy").exists()
    idx = np.load(tmp_path / "b" / "C4_image_sample_index.npy")
    sample = np.load(tmp_path / "b" / "C4_image_sample.npy")
    assert idx.dtype == np.float64 and sample.dtype == np.float32 and len(idx) > 10000 and np.all(np.diff(idx) > 0)
    assert np.array_equal(sample, big.reshape(-1, 3)[idx.astype(np.int64)].astype(np.float32))
    assert np.array_equal(idx, np.load(tmp_path / "c" / "C4_image_sample_index.npy"))


def test_gloo_world_size_2_gather_and_stats(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    # the workers see no CUDA device, also on a GPU machine: the fallback of SharedFramebuffer is what they check
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29613", WORLD_SIZE="2", CUDA_VISIBLE_DEVICES="")
    procs = [subprocess.Popen([sys.executable, str(script), ROOT], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT) for r in range(2)]
    outs = [p.communicate(timeout=180)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert "GATHER_OK" in outs[0]


def test_napi_shim_compiles_against_the_stub_header():
    """ts/addon/rt_napi.c cannot be built here (no node, no node_api.h); it is type-checked against a stub of the Node-API
    prototypes it uses, and against the real include/rt_b200.h: argument counts and types of every rt_* call are verified."""
    cmd = ["gcc", "-fsyntax-only", "-std=c11", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "ts", "addon", "stub"),
           "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "ts", "addon", "rt_napi.c")]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    assert r.returncode == 0, r.stdout.decode()
    src = open(os.path.join(ROOT, "ts", "addon", "rt_napi.c")).read()
    for fn in ("rt_camera_create", "rt_multi_create", "rt_camera_render_region", "rt_multi_render_region", "rt_camera_destroy", "rt_multi_destroy",
               "napi_async_work", "napi_adjust_external_memory"):
        assert fn in src, fn


def test_scene_camera_options_of_the_mcp_tool_take_effect():
    """src/mcp.ts:132-142 accepts scene.camera and the reference drops it; the native dispatch applies it (SURVEY 8f row 4)."""
    from mcp_raytracer_b200 import generateSceneData, validateScene
    from mcp_raytracer_b200.raytracer import applySceneCameraOptions

    sd = generateSceneData({"type": "cornell"})
    out = applySceneCameraOptions(sd, {"imageWidth": 320, "aspectRatio": 2.0, "vfov": 55, "lookFrom": [1, 2, 3], "lookAt": [0, 0, 1], "vUp": [0, 0, 1],
                                       "samples": 7, "adaptiveTolerance": 0.2, "adaptiveBatchSize": 4})
    assert out["camera"]["vfov"] == 55 and out["camera"]["from"] == [1, 2, 3] and out["camera"]["at"] == [0, 0, 1] and out["camera"]["up"] == [0, 0, 1]
    assert out["render"]["width"] == 320 and out["render"]["aspect"] == 2.0 and out["render"]["samples"] == 7
    assert out["render"]["aTolerance"] == 0.2 and out["render"]["aBatch"] == 4
    assert sd["camera"]["vfov"] != 55 and applySceneCameraOptions(sd, None) is sd   # the input is not modified
    rep = validateScene(out, None)
    assert rep["errors"] == 0
