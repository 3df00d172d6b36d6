"""ctypes binding of the CPU oracle (oracle/liboracle.so) — TEST INFRASTRUCTURE.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  The product package never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys
from typing import Any, Dict, Optional

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from mcp_raytracer_b200.scene_data import (  # noqa: E402
    FlatScene, merge_render_options, render_opts_struct, rt_region, rt_render_opts, rt_scene_desc, rt_stats,
)

_LIB: Optional[C.CDLL] = None
COUNTER_NAMES = [
    "rays", "box_tests", "sphere_miss", "sphere_hit", "planar_treject", "quad_outside", "quad_hit", "plane_hit",
    "rr", "background", "hits", "lambert", "metal", "metal_fuzz0", "dielectric", "light_pdf_evals", "paths", "defocus",
]


def build_oracle() -> str:
    d = os.path.join(ROOT, "oracle")
    so = os.path.join(d, "liboracle.so")
    src = os.path.join(d, "oracle.cpp")
    hdr = os.path.join(ROOT, "include", "rt_b200.h")
    if (not os.path.exists(so)) or os.path.getmtime(so) < max(os.path.getmtime(src), os.path.getmtime(hdr)):
        subprocess.check_call(["make", "-C", d, "liboracle.so"], stdout=subprocess.DEVNULL)
    return so


def build_native_oracle(out_dir: str) -> Optional[str]:
    """`make native`: the oracle compiled with -march=native ON THIS HOST (bench.py's CPU baseline, BASELINE.md section 3),
    written to `out_dir` so that the tree itself may be read-only.
    None when there is no compiler here or the build fails; the portable build is used then."""
    d = os.path.join(ROOT, "oracle")
    out_dir = os.path.abspath(out_dir)
    try:
        subprocess.check_call(["make", "-C", d, "native", f"NATIVE_DIR={out_dir}"], stdout=subprocess.DEVNULL,
                              stderr=subprocess.DEVNULL, timeout=300)
    except Exception:
        return None
    so = os.path.join(out_dir, "liboracle.so")
    return so if os.path.exists(so) else None


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        L = C.CDLL(os.environ.get("RT_ORACLE_LIB") or build_oracle())
        dp = C.POINTER(C.c_double)
        fp = C.POINTER(C.c_float)
        L.orc_last_error.restype = C.c_char_p
        L.orc_camera_create.argtypes = [C.POINTER(rt_scene_desc), C.POINTER(rt_render_opts), C.POINTER(C.c_void_p)]
        L.orc_camera_destroy.argtypes = [C.c_void_p]
        L.orc_camera_info.argtypes = [C.c_void_p, C.POINTER(C.c_int), fp, dp]
        L.orc_render_region.argtypes = [C.c_void_p, C.POINTER(rt_region), C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                        C.POINTER(rt_stats), C.c_int, C.c_uint64, C.c_int, C.c_void_p]
        L.orc_trace_primary.argtypes = [C.c_void_p, C.POINTER(rt_region), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_trace_rays.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_int,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_ray_color.argtypes = [C.c_void_p, fp, fp, C.c_uint32, C.c_uint32, C.c_uint64, fp, C.POINTER(C.c_int)]
        L.orc_get_ray.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_uint32, C.c_uint64, fp, fp]
        L.orc_philox4x32.argtypes = [C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.c_int, C.POINTER(C.c_uint32)]
        L.orc_philox_rounds.restype = C.c_int
        L.orc_stream_uniforms.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, C.c_int, dp]
        L.orc_sphere_hit.argtypes = [dp, C.c_double, dp, dp, C.c_double, C.c_double, dp]
        L.orc_sphere_pdf_value.argtypes = [dp, C.c_double, dp, dp]
        L.orc_sphere_pdf_value.restype = C.c_double
        L.orc_sphere_pdf_random.argtypes = [dp, C.c_double, dp, C.c_uint64, C.c_int, fp]
        L.orc_planar_hit.argtypes = [C.c_int, dp, dp, dp, dp, dp, C.c_double, C.c_double, dp]
        L.orc_plane_intersect.argtypes = [dp, dp, dp, dp, dp, C.c_double, C.c_double, dp]
        L.orc_object_bbox.argtypes = [C.c_int, dp, dp, dp, C.c_double, dp]
        L.orc_quad_pdf_value.argtypes = [dp, dp, dp, dp, dp]
        L.orc_quad_pdf_value.restype = C.c_double
        L.orc_quad_pdf_random.argtypes = [dp, dp, dp, dp, C.c_uint64, C.c_int, fp]
        L.orc_aabb_hit.argtypes = [dp, dp, dp, dp, C.c_double, C.c_double]
        L.orc_surrounding_box.argtypes = [dp, dp, dp, dp, dp]
        L.orc_cosine_pdf_value.argtypes = [dp, dp]
        L.orc_cosine_pdf_value.restype = C.c_double
        L.orc_cosine_pdf_generate.argtypes = [dp, C.c_uint64, C.c_int, fp]
        L.orc_random_cosine_direction.argtypes = [C.c_uint64, C.c_int, fp]
        L.orc_onb.argtypes = [dp, fp]
        L.orc_mixture_value.argtypes = [C.c_int, dp, dp]
        L.orc_mixture_value.restype = C.c_double
        L.orc_mixture_select.argtypes = [C.c_int, dp, C.c_double]
        L.orc_reflect.argtypes = [dp, dp, fp]
        L.orc_refract.argtypes = [dp, dp, C.c_double, fp]
        L.orc_unit.argtypes = [dp, fp]
        L.orc_dielectric_reflectance.argtypes = [C.c_double, C.c_double]
        L.orc_dielectric_reflectance.restype = C.c_double
        L.orc_metal_fuzz_clamp.argtypes = [C.c_double]
        L.orc_metal_fuzz_clamp.restype = C.c_double
        L.orc_mixed_weight_clamp.argtypes = [C.c_double]
        L.orc_mixed_weight_clamp.restype = C.c_double
        L.orc_material_scatter.argtypes = [C.POINTER(rt_scene_desc), C.c_int, dp, dp, dp, dp, C.c_int, C.c_uint64, C.c_uint32, dp, fp]
        ip = C.POINTER(C.c_int)
        L.orc_material_scatter_u.argtypes = [C.POINTER(rt_scene_desc), C.c_int, dp, dp, dp, dp, C.c_int, dp, C.c_int, dp, fp, ip]
        L.orc_get_ray_u.argtypes = [C.c_void_p, C.c_int, C.c_int, dp, C.c_int, fp, fp, ip]
        L.orc_light_pdf_value.argtypes = [C.c_void_p, C.c_int, dp, dp]
        L.orc_light_pdf_value.restype = C.c_double
        L.orc_light_random_vec_u.argtypes = [C.c_void_p, C.c_int, dp, dp, C.c_int, fp, ip]
        L.orc_diffuse_bounce_u.argtypes = [C.c_void_p, dp, dp, dp, C.c_int, dp, ip]
        L.orc_write_color.argtypes = [dp, C.POINTER(C.c_uint8)]
        L.orc_pixel_converged.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double]
        L.orc_vec3_op.argtypes = [C.c_int, dp, dp, C.c_double, fp]
        L.orc_vec3_op.restype = C.c_double
        L.orc_ray_at.argtypes = [dp, dp, C.c_double, fp]
        L.orc_interval_op.argtypes = [C.c_int, C.c_double, C.c_double, C.c_double]
        L.orc_interval_op.restype = C.c_double
        L.orc_sample_vec3.argtypes = [C.c_int, C.c_uint64, C.c_double, C.c_double, C.c_int, fp]
        _LIB = L
    return _LIB


def d3(v):
    return (C.c_double * 3)(*[float(x) for x in v])


class OracleError(Exception):
    pass


class OracleCamera:
    """`createCameraFromSceneData(sceneData, renderOptions)` on the oracle."""

    def __init__(self, sceneData: Dict[str, Any], renderOptions: Optional[Dict[str, Any]] = None):
        self.flat = FlatScene(sceneData)
        self.options = merge_render_options(sceneData.get("render"), renderOptions)
        self.opts = render_opts_struct(self.options)
        h = C.c_void_p()
        st = lib().orc_camera_create(C.byref(self.flat.desc), C.byref(self.opts), C.byref(h))
        if st != 0:
            raise OracleError(f"status {st}: {lib().orc_last_error().decode()}")
        self.h = h
        info = (C.c_int * 5)()
        vecs = (C.c_float * 27)()
        focus = C.c_double()
        lib().orc_camera_info(self.h, info, vecs, C.byref(focus))
        self.imageWidth, self.imageHeight, self.n_lights, self.bvh_nodes, self.bvh_depth = list(info)
        v = np.array(vecs, dtype=np.float32).reshape(9, 3)
        (self.center, self.pixel00Loc, self.pixelDeltaU, self.pixelDeltaV, self.u, self.v, self.w,
         self.defocusDiskU, self.defocusDiskV) = v
        self.focusDistance = focus.value

    def __del__(self):
        try:
            if getattr(self, "h", None):
                lib().orc_camera_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def full_region(self):
        return rt_region(0, 0, self.imageWidth, self.imageHeight)

    def render(self, region=None, rng_mode=0, seed=0, threads=1, want_moments=False, want_counters=False):
        W, H = self.imageWidth, self.imageHeight
        reg = region or self.full_region()
        rgb = np.zeros((H, W, 3), np.uint8)
        lin = np.zeros((H, W, 3), np.float32)
        mom = np.zeros((H, W, 8), np.float64) if want_moments else None
        cnt = np.zeros(len(COUNTER_NAMES), np.uint64)  # always on: stats.rays is an event count
        st = rt_stats()
        rc = lib().orc_render_region(self.h, C.byref(reg), rgb.ctypes.data, rgb.nbytes, lin.ctypes.data,
                                     mom.ctypes.data if mom is not None else None, C.byref(st), rng_mode, seed, threads,
                                     cnt.ctypes.data if cnt is not None else None)
        if rc != 0:
            raise OracleError(f"status {rc}: {lib().orc_last_error().decode()}")
        out = {"rgb8": rgb, "linear": lin, "stats": st}
        if mom is not None:
            out["moments"] = mom
        if cnt is not None:
            out["counters"] = dict(zip(COUNTER_NAMES, [int(x) for x in cnt]))
        return out

    def trace_primary(self, region=None):
        W, H = self.imageWidth, self.imageHeight
        reg = region or self.full_region()
        ids = np.full((H, W), -2, np.int32)
        t = np.zeros((H, W), np.float64)
        nrm = np.zeros((H, W, 3), np.float32)
        ff = np.zeros((H, W), np.uint8)
        lib().orc_trace_primary(self.h, C.byref(reg), ids.ctypes.data, t.ctypes.data, nrm.ctypes.data, ff.ctypes.data)
        return ids, t, nrm, ff

    def trace_rays(self, origins, dirs, tmin=0.001, tmax=float("inf"), use_bvh=True):
        o = np.ascontiguousarray(origins, np.float32)
        d = np.ascontiguousarray(dirs, np.float32)
        n = o.shape[0]
        ids = np.zeros(n, np.int32)
        t = np.zeros(n, np.float64)
        nrm = np.zeros((n, 3), np.float32)
        ff = np.zeros(n, np.uint8)
        lib().orc_trace_rays(self.h, n, o.ctypes.data, d.ctypes.data, tmin, tmax, 1 if use_bvh else 0,
                             ids.ctypes.data, t.ctypes.data, nrm.ctypes.data, ff.ctypes.data)
        return ids, t, nrm, ff

    def ray_color(self, origin, direction, pixel=0, sample=0, seed=0):
        o = (C.c_float * 3)(*origin)
        d = (C.c_float * 3)(*direction)
        rgb = (C.c_float * 3)()
        b = C.c_int()
        lib().orc_ray_color(self.h, o, d, pixel, sample, seed, rgb, C.byref(b))
        return np.array(rgb, dtype=np.float32), b.value

    def get_ray(self, i, j, sample=0, seed=0):
        o = (C.c_float * 3)()
        d = (C.c_float * 3)()
        lib().orc_get_ray(self.h, i, j, sample, seed, o, d)
        return np.array(o, dtype=np.float32), np.array(d, dtype=np.float32)


# ---- per-function hooks with explicit uniforms (the CPU side of tests/test_gpu_functions.py) ----
def _dn(v):
    a = [float(x) for x in v]
    return (C.c_double * len(a))(*a)


def material_scatter_u(flat: FlatScene, root: int, ray_origin, ray_dir, p, normal, front_face, uniforms):
    """material.scatter + emitted with the given Math.random() sequence.
    Returns (kind, attenuation, dir, emitted, used, reflected); kind 0 null / 1 scattered ray / 2 pdf."""
    out = (C.c_double * 9)()
    em = (C.c_float * 3)()
    used = C.c_int()
    rc = lib().orc_material_scatter_u(C.byref(flat.desc), int(root), d3(ray_origin), d3(ray_dir), d3(p), d3(normal), int(bool(front_face)),
                                      _dn(uniforms), len(uniforms), out, em, C.byref(used))
    if rc < 0:
        raise OracleError(f"status {-rc}")
    o = list(out)
    kind = 0 if rc == 0 else (1 if o[0] == 1.0 else 2)
    return kind, np.array(o[2:5]), np.array(o[5:8]), np.array(list(em)), used.value, (bool(o[8]) if rc else False)


def get_ray_u(cam: "OracleCamera", i, j, uniforms):
    o, d, used = (C.c_float * 3)(), (C.c_float * 3)(), C.c_int()
    lib().orc_get_ray_u(cam.h, int(i), int(j), _dn(uniforms), len(uniforms), o, d, C.byref(used))
    return np.array(o, np.float32), np.array(d, np.float32), used.value


def light_pdf_value(cam: "OracleCamera", k, origin, direction) -> float:
    return float(lib().orc_light_pdf_value(cam.h, int(k), d3(origin), d3(direction)))


def light_random_vec_u(cam: "OracleCamera", k, origin, uniforms):
    out, used = (C.c_float * 3)(), C.c_int()
    lib().orc_light_random_vec_u(cam.h, int(k), d3(origin), _dn(uniforms), len(uniforms), out, C.byref(used))
    return np.array(out, np.float32), used.value


def diffuse_bounce_u(cam: "OracleCamera", p, normal, uniforms):
    """[dir x,y,z, mixture pdf value, scatter pdf value, continues], uniforms used"""
    out, used = (C.c_double * 6)(), C.c_int()
    lib().orc_diffuse_bounce_u(cam.h, d3(p), d3(normal), _dn(uniforms), len(uniforms), out, C.byref(used))
    return np.array(list(out)), used.value
