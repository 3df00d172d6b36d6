"""SceneData -> SoA flattening for the C ABI (include/rt_b200.h).

Host-side half of the boundary: what the reference does with objects
(`createSceneObject` / `createMaterial` / `createDielectric`, src/scenes/scenes.ts:109-199)
becomes a table of primitives and a table of material nodes.  Error behaviour mirrors the
reference: the same conditions raise, with the same message text.

The ctypes structures here are the single Python definition of `rt_scene_desc`,
`rt_render_opts`, `rt_region`, `rt_stats`, `rt_camera_info`; tests/ re-use them to drive the
CPU oracle with bit-identical inputs.
"""
from __future__ import annotations

import ctypes as C
from typing import Any, Dict, List, Optional, Union

import numpy as np

# ---- enums (include/rt_b200.h) ----
RT_OBJ_SPHERE, RT_OBJ_PLANE, RT_OBJ_QUAD = 0, 1, 2
RT_MAT_LAMBERT, RT_MAT_METAL, RT_MAT_GLASS, RT_MAT_LIGHT, RT_MAT_MIXED, RT_MAT_LAYERED = range(6)
RT_MODE_DEFAULT, RT_MODE_BOUNCES, RT_MODE_SAMPLES = 0, 1, 2
RT_BVH_AUTO, RT_BVH_REFERENCE, RT_BVH_SAH, RT_BVH_LIST = 0, 1, 2, 3
RT_INTEGRATOR_AUTO, RT_INTEGRATOR_MEGAKERNEL, RT_INTEGRATOR_WAVEFRONT, RT_INTEGRATOR_SORTED = 0, 1, 2, 3

_OBJ_TYPES = {"sphere": RT_OBJ_SPHERE, "plane": RT_OBJ_PLANE, "quad": RT_OBJ_QUAD}
_MODES = {"default": RT_MODE_DEFAULT, "bounces": RT_MODE_BOUNCES, "samples": RT_MODE_SAMPLES}
_BVH = {"auto": RT_BVH_AUTO, "reference": RT_BVH_REFERENCE, "sah": RT_BVH_SAH, "list": RT_BVH_LIST}
_INTEGRATORS = {"auto": RT_INTEGRATOR_AUTO, "megakernel": RT_INTEGRATOR_MEGAKERNEL, "wavefront": RT_INTEGRATOR_WAVEFRONT,
                "sorted": RT_INTEGRATOR_SORTED}
RT_LIGHTS_MIXTURE, RT_LIGHTS_SHADOW_RAYS = 0, 1
_LIGHTS = {"mixture": RT_LIGHTS_MIXTURE, "shadowRays": RT_LIGHTS_SHADOW_RAYS}


class RaytracerError(Exception):
    """Stands in for the JS `Error` the reference throws on the scene-build path."""


class rt_camera_desc(C.Structure):
    _fields_ = [
        ("vfov", C.c_double),
        ("from_", C.c_double * 3),
        ("at", C.c_double * 3),
        ("up", C.c_double * 3),
        ("aperture", C.c_double),
        ("focus", C.c_double),
        ("background_top", C.c_double * 3),
        ("background_bottom", C.c_double * 3),
    ]


class rt_scene_desc(C.Structure):
    _fields_ = [
        ("n_objects", C.c_uint32),
        ("obj_type", C.POINTER(C.c_uint8)),
        ("obj_pos", C.POINTER(C.c_double)),
        ("obj_u", C.POINTER(C.c_double)),
        ("obj_v", C.POINTER(C.c_double)),
        ("obj_r", C.POINTER(C.c_double)),
        ("obj_material", C.POINTER(C.c_int32)),
        ("obj_light", C.POINTER(C.c_uint8)),
        ("n_materials", C.c_uint32),
        ("mat_type", C.POINTER(C.c_uint8)),
        ("mat_color", C.POINTER(C.c_double)),
        ("mat_param", C.POINTER(C.c_double)),
        ("mat_child", C.POINTER(C.c_int32)),
        ("camera", rt_camera_desc),
    ]


class rt_render_opts(C.Structure):
    _fields_ = [
        ("width", C.c_int32),
        ("aspect", C.c_double),
        ("samples", C.c_int32),
        ("depth", C.c_int32),
        ("a_tolerance", C.c_double),
        ("a_batch", C.c_int32),
        ("roulette", C.c_int32),
        ("roulette_depth", C.c_int32),
        ("mode", C.c_int32),
        ("seed", C.c_uint64),
        ("bvh", C.c_int32),
        ("integrator", C.c_int32),
        ("device", C.c_int32),
        ("part_index", C.c_int32),
        ("part_count", C.c_int32),
        ("light_sampling", C.c_int32),
    ]


class rt_region(C.Structure):
    _fields_ = [("x", C.c_int32), ("y", C.c_int32), ("width", C.c_int32), ("height", C.c_int32)]


class rt_stats(C.Structure):
    _fields_ = [
        ("pixels", C.c_uint64),
        ("samples_total", C.c_uint64),
        ("samples_min", C.c_int32),
        ("samples_max", C.c_int32),
        ("bounces_total", C.c_uint64),
        ("bounces_min", C.c_int32),
        ("bounces_max", C.c_int32),
        ("rays", C.c_uint64),
        ("device_ms", C.c_double),
        ("kernel_launches", C.c_int32),
        ("reserved", C.c_int32),
        ("node_visits", C.c_uint64),
        ("prim_tests", C.c_uint64),
    ]


class rt_denoise_opts(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("sigma_luminance", C.c_float), ("sigma_normal", C.c_float), ("sigma_depth", C.c_float)]


DENOISE_OPTION_KEYS = ("iterations", "sigmaLuminance", "sigmaNormal", "sigmaDepth")


def denoise_opts_struct(options: Optional[Dict[str, Any]]) -> rt_denoise_opts:
    """Denoiser options {iterations (default 5), sigmaLuminance, sigmaNormal, sigmaDepth (0 or absent = default)} -> struct."""
    o = dict(options or {})
    unknown = set(o) - set(DENOISE_OPTION_KEYS)
    if unknown:
        raise RaytracerError(f"unknown denoise options: {sorted(unknown)}")
    return rt_denoise_opts(iterations=int(o.get("iterations", 5)), sigma_luminance=float(o.get("sigmaLuminance", 0.0)),
                           sigma_normal=float(o.get("sigmaNormal", 0.0)), sigma_depth=float(o.get("sigmaDepth", 0.0)))


class rt_camera_info(C.Structure):
    _fields_ = [
        ("image_width", C.c_int32), ("image_height", C.c_int32), ("channels", C.c_int32),
        ("n_objects", C.c_int32), ("n_lights", C.c_int32), ("n_bvh_nodes", C.c_int32),
        ("bvh_kind", C.c_int32), ("integrator_kind", C.c_int32),
        ("center", C.c_float * 3), ("pixel00_loc", C.c_float * 3),
        ("pixel_delta_u", C.c_float * 3), ("pixel_delta_v", C.c_float * 3),
        ("u", C.c_float * 3), ("v", C.c_float * 3), ("w", C.c_float * 3),
        ("defocus_disk_u", C.c_float * 3), ("defocus_disk_v", C.c_float * 3),
        ("focus_distance", C.c_double),
        ("use_adaptive_sampling", C.c_int32),
        ("device", C.c_int32),
        ("build_ms", C.c_double),
    ]


# Camera.defaultCameraOptions / defaultRenderData — src/camera.ts:62-83
DEFAULT_CAMERA_OPTIONS: Dict[str, Any] = {
    "vfov": 90, "from": [0, 0, 0], "at": [0, 0, -1], "up": [0, 1, 0], "aperture": 0, "focus": 1.0,
    "background": {"type": "gradient", "top": [1, 1, 1], "bottom": [0.5, 0.7, 1.0]},
}
DEFAULT_RENDER_DATA: Dict[str, Any] = {
    "width": 400, "aspect": 16 / 9, "samples": 100, "aTolerance": 0.05, "aBatch": 10,
    "mode": "default", "depth": 100, "roulette": True, "rouletteDepth": 3,
}
# knobs that exist only on this side of the boundary
DEFAULT_NATIVE_OPTIONS: Dict[str, Any] = {
    "seed": 0, "bvh": "auto", "integrator": "auto", "device": -1, "partIndex": 0, "partCount": 1,
    "lightSampling": "mixture",  # "shadowRays": next-event estimation (rt_b200.h RT_LIGHTS_*)
}


def merge_render_options(scene_render: Optional[Dict[str, Any]], render_options: Optional[Dict[str, Any]]) -> Dict[str, Any]:
    """defaults <- sceneData.render <- caller (src/camera.ts:116, src/scenes/scenes.ts:97-100).

    Deliberate divergence: the reference's object spread copies explicit `undefined`
    (SURVEY.md §5 "Config / flags"), which poisons the camera with NaN; `None` values are
    skipped here instead.
    """
    out = dict(DEFAULT_RENDER_DATA)
    out.update(DEFAULT_NATIVE_OPTIONS)
    for layer in (scene_render, render_options):
        if layer:
            out.update({k: v for k, v in layer.items() if v is not None})
    return out


def render_opts_struct(o: Dict[str, Any]) -> rt_render_opts:
    mode = o["mode"]
    mode = getattr(mode, "value", mode)
    if mode not in _MODES:
        raise RaytracerError(f"Invalid render mode: {mode}")
    return rt_render_opts(
        width=int(o["width"]), aspect=float(o["aspect"]), samples=int(o["samples"]), depth=int(o["depth"]),
        a_tolerance=float(o["aTolerance"]), a_batch=int(o["aBatch"]), roulette=1 if o["roulette"] else 0,
        roulette_depth=int(o["rouletteDepth"]), mode=_MODES[mode], seed=int(o["seed"]) & 0xFFFFFFFFFFFFFFFF,
        bvh=_BVH[o["bvh"]] if isinstance(o["bvh"], str) else int(o["bvh"]),
        integrator=_INTEGRATORS[o["integrator"]] if isinstance(o["integrator"], str) else int(o["integrator"]),
        device=int(o["device"]), part_index=int(o["partIndex"]), part_count=int(o["partCount"]),
        light_sampling=_LIGHTS[o["lightSampling"]] if isinstance(o["lightSampling"], str) else int(o["lightSampling"]),
    )

_OBJ_NAMES = {v: k for k, v in _OBJ_TYPES.items()}


class SoAMaterials:
    """`SceneData.materials` held as arrays (the material node table of rt_scene_desc) that still READS like the
    reference's list of `{id, material}` records (src/scenes/sceneData.ts:76-110): len(), iteration and indexing build
    the dicts on demand.  Large procedural scenes (100 000 rain drops = 100 001 materials) are generated straight into
    this form, so handing them to the C ABI costs no per-object Python work; arbitrary SceneData keeps the dict walk.

    type/color/param/child: node table (children precede parents); `roots` = node index of each named material;
    `ids(k)` = its id string."""

    def __init__(self, type_, color, param, child, roots, ids):
        self.type = np.ascontiguousarray(type_, np.uint8)
        self.color = np.ascontiguousarray(color, np.float64).reshape(-1, 3)
        self.param = np.ascontiguousarray(param, np.float64)
        self.child = np.ascontiguousarray(child, np.int32).reshape(-1, 2)
        self.roots = np.ascontiguousarray(roots, np.int32)
        self._ids = ids  # callable k -> str

    def __len__(self) -> int:
        return int(self.roots.shape[0])

    def node_dict(self, i: int) -> Dict[str, Any]:
        t = int(self.type[i])
        c = [float(x) for x in self.color[i]]
        if t == RT_MAT_LAMBERT:
            return {"type": "lambert", "color": c}
        if t == RT_MAT_METAL:
            return {"type": "metal", "color": c, "fuzz": float(self.param[i])}
        if t == RT_MAT_GLASS:
            return {"type": "glass", "ior": float(self.param[i])}
        if t == RT_MAT_LIGHT:
            return {"type": "light", "emit": c}
        if t == RT_MAT_MIXED:
            return {"type": "mixed", "diff": self.node_dict(int(self.child[i, 0])), "spec": self.node_dict(int(self.child[i, 1])), "weight": float(self.param[i])}
        return {"type": "layered", "inner": self.node_dict(int(self.child[i, 0])), "outer": self.node_dict(int(self.child[i, 1]))}

    def id_of(self, k: int) -> str:
        return self._ids(k)

    def __getitem__(self, k):
        if isinstance(k, slice):
            return [self[i] for i in range(*k.indices(len(self)))]
        if k < 0:
            k += len(self)
        if not 0 <= k < len(self):
            raise IndexError(k)
        return {"id": self._ids(k), "material": self.node_dict(int(self.roots[k]))}

    def __iter__(self):
        return (self[k] for k in range(len(self)))

    def tolist(self) -> List[Dict[str, Any]]:
        return list(self)


class SoAObjects:
    """`SceneData.objects` as arrays; reads like the reference's list of SceneObject records
    (src/scenes/sceneData.ts:40-70).  material[k] = index into `materials` (a SoAMaterials)."""

    def __init__(self, type_, pos, u, v, r, material, light, materials: SoAMaterials):
        n = len(type_)
        self.type = np.ascontiguousarray(type_, np.uint8)
        self.pos = np.ascontiguousarray(pos, np.float64).reshape(n, 3)
        self.u = np.ascontiguousarray(u, np.float64).reshape(n, 3)
        self.v = np.ascontiguousarray(v, np.float64).reshape(n, 3)
        self.r = np.ascontiguousarray(r, np.float64).reshape(n)
        self.material = np.ascontiguousarray(material, np.int32).reshape(n)
        self.light = np.ascontiguousarray(light, np.uint8).reshape(n)
        self.materials = materials

    def __len__(self) -> int:
        return int(self.type.shape[0])

    def __getitem__(self, k):
        if isinstance(k, slice):
            return [self[i] for i in range(*k.indices(len(self)))]
        if k < 0:
            k += len(self)
        if not 0 <= k < len(self):
            raise IndexError(k)
        t = int(self.type[k])
        ob: Dict[str, Any] = {"type": _OBJ_NAMES[t], "pos": [float(x) for x in self.pos[k]]}
        if t == RT_OBJ_SPHERE:
            ob["r"] = float(self.r[k])
        else:
            ob["u"] = [float(x) for x in self.u[k]]
            ob["v"] = [float(x) for x in self.v[k]]
        ob["material"] = self.materials.id_of(int(self.material[k]))
        if self.light[k]:
            ob["light"] = True
        return ob

    def __iter__(self):
        return (self[k] for k in range(len(self)))

    def tolist(self) -> List[Dict[str, Any]]:
        return list(self)


class FlatScene:
    """Owns the numpy arrays behind an `rt_scene_desc` (keeps them alive)."""

    def __init__(self, sceneData: Dict[str, Any]):
        objs0 = sceneData["objects"]
        if isinstance(objs0, SoAObjects) and sceneData.get("materials") is objs0.materials:
            self._from_arrays(objs0, sceneData)  # array-backed scene from a generator: nothing to walk
            return
        materials: Dict[str, Any] = {}
        for m in sceneData.get("materials") or []:  # scenes.ts:62-65
            materials[m["id"]] = m["material"]

        self.mat_type: List[int] = []
        self.mat_color: List[List[float]] = []
        self.mat_param: List[float] = []
        self.mat_child: List[List[int]] = []
        self._by_id: Dict[str, int] = {}

        objs = sceneData["objects"]
        n = len(objs)
        # plain lists, converted once: a 100k-object scene spends its time here otherwise
        types: List[int] = []
        mats: List[int] = []
        pos: List[Any] = []
        us: List[Any] = []
        vs: List[Any] = []
        rs: List[float] = []
        lights: List[int] = []
        zero3 = (0.0, 0.0, 0.0)
        # (the per-object part of this loop is ~60 ms per 100 k objects; the rest of the ~0.2 s is the material
        #  table, one `_material` call per distinct material — comprehensions instead of this loop gained nothing)
        for ob in objs:
            # scenes.ts:113 creates the material first, then switches on the object type
            mats.append(self._material(ob.get("material"), materials))
            t = ob.get("type")
            code = _OBJ_TYPES.get(t) if isinstance(t, str) else None
            if code is None:
                raise RaytracerError(f"Unknown object type: {t}")  # scenes.ts:137
            types.append(code)
            pos.append(ob["pos"])
            if code == RT_OBJ_SPHERE:
                rs.append(ob["r"])
                us.append(zero3)
                vs.append(zero3)
            else:
                rs.append(0.0)
                us.append(ob["u"])
                vs.append(ob["v"])
            lights.append(1 if ob.get("light") else 0)
        self.obj_type = np.array(types, np.uint8).reshape(n)
        self.obj_pos = np.ascontiguousarray(np.array(pos, np.float64).reshape(n, 3))
        self.obj_u = np.ascontiguousarray(np.array(us, np.float64).reshape(n, 3))
        self.obj_v = np.ascontiguousarray(np.array(vs, np.float64).reshape(n, 3))
        self.obj_r = np.array(rs, np.float64).reshape(n)
        self.obj_material = np.array(mats, np.int32).reshape(n)
        self.obj_light = np.array(lights, np.uint8).reshape(n)

        self.mat_type_a = np.asarray(self.mat_type, np.uint8)
        self.mat_color_a = np.asarray(self.mat_color, np.float64).reshape(-1, 3)
        self.mat_param_a = np.asarray(self.mat_param, np.float64)
        self.mat_child_a = np.asarray(self.mat_child, np.int32).reshape(-1, 2)

        self._finish(sceneData, n)

    def _from_arrays(self, objs: "SoAObjects", sceneData: Dict[str, Any]) -> None:
        """Array-backed SceneData: no per-object Python work.  The checks the dict walk makes per record
        (scenes.ts:137, :154, :178) run vectorised; the C side validates the node table again."""
        m = objs.materials
        n = len(objs)
        if n and int(objs.type.max()) > RT_OBJ_QUAD:
            raise RaytracerError(f"Unknown object type: {int(objs.type.max())}")
        if len(m.type) and int(m.type.max()) > RT_MAT_LAYERED:
            raise RaytracerError(f"Unknown material type: {int(m.type.max())}")
        if n and (int(objs.material.min()) < 0 or int(objs.material.max()) >= len(m)):
            raise RaytracerError(f"Material not found: {int(objs.material.max())}")
        self.obj_type, self.obj_pos, self.obj_u, self.obj_v, self.obj_r, self.obj_light = objs.type, objs.pos, objs.u, objs.v, objs.r, objs.light
        self.obj_material = np.ascontiguousarray(m.roots[objs.material], np.int32)  # object -> root node of its material
        self.mat_type_a, self.mat_color_a, self.mat_param_a, self.mat_child_a = m.type, m.color, m.param, m.child
        self._finish(sceneData, n)

    def _finish(self, sceneData: Dict[str, Any], n: int) -> None:
        cam = dict(DEFAULT_CAMERA_OPTIONS)
        cam.update({k: v for k, v in (sceneData.get("camera") or {}).items() if v is not None})
        bg = cam["background"]
        self.camera = rt_camera_desc(
            vfov=float(cam["vfov"]), from_=(C.c_double * 3)(*cam["from"]), at=(C.c_double * 3)(*cam["at"]),
            up=(C.c_double * 3)(*cam["up"]), aperture=float(cam["aperture"]), focus=float(cam["focus"] or 0.0),
            background_top=(C.c_double * 3)(*bg["top"]), background_bottom=(C.c_double * 3)(*bg["bottom"]),
        )
        self.render = sceneData.get("render")

        def p(a, ty):
            return a.ctypes.data_as(C.POINTER(ty))

        self.desc = rt_scene_desc(
            n_objects=n, obj_type=p(self.obj_type, C.c_uint8), obj_pos=p(self.obj_pos, C.c_double),
            obj_u=p(self.obj_u, C.c_double), obj_v=p(self.obj_v, C.c_double), obj_r=p(self.obj_r, C.c_double),
            obj_material=p(self.obj_material, C.c_int32), obj_light=p(self.obj_light, C.c_uint8),
            n_materials=len(self.mat_type_a), mat_type=p(self.mat_type_a, C.c_uint8),
            mat_color=p(self.mat_color_a, C.c_double), mat_param=p(self.mat_param_a, C.c_double),
            mat_child=p(self.mat_child_a, C.c_int32), camera=self.camera,
        )

    # -- createMaterial / createDielectric, src/scenes/scenes.ts:144-199 --
    def _node(self, ty: int, color=(0.0, 0.0, 0.0), param: float = 0.0, child=(-1, -1)) -> int:
        # values are converted (and type-checked) once by numpy at the end of __init__
        self.mat_type.append(ty)
        self.mat_color.append(color if len(color) == 3 else (color[0], color[1], color[2]))
        self.mat_param.append(param)
        self.mat_child.append(child)
        return len(self.mat_type) - 1

    def _material(self, ref: Union[str, Dict[str, Any], None], materials: Dict[str, Any], depth: int = 0) -> int:
        if isinstance(ref, str) and ref in self._by_id:
            return self._by_id[ref]
        data = materials.get(ref) if isinstance(ref, str) else ref
        if not data:
            raise RaytracerError(f"Material not found: {ref}")  # scenes.ts:153-155
        if depth > 64:
            raise RaytracerError(f"Material nesting too deep: {ref}")
        t = data.get("type")
        if t == "lambert":
            idx = self._node(RT_MAT_LAMBERT, data["color"])
        elif t == "metal":
            idx = self._node(RT_MAT_METAL, data["color"], data["fuzz"])
        elif t == "glass":
            idx = self._node(RT_MAT_GLASS, param=data["ior"])
        elif t == "light":
            idx = self._node(RT_MAT_LIGHT, data["emit"])
        elif t == "mixed":
            a = self._material(data["diff"], materials, depth + 1)
            b = self._material(data["spec"], materials, depth + 1)
            idx = self._node(RT_MAT_MIXED, param=data["weight"], child=(a, b))
        elif t == "layered":
            outer_ref = data["outer"]
            outer = materials.get(outer_ref) if isinstance(outer_ref, str) else outer_ref
            if not outer:
                raise RaytracerError(f"Material not found: {outer_ref}")  # scenes.ts:190-192
            if outer.get("type") != "glass":
                raise RaytracerError(f"Material is not a dielectric: {outer_ref}")  # scenes.ts:194-196
            o = self._material(outer_ref, materials, depth + 1)
            i = self._material(data["inner"], materials, depth + 1)
            idx = self._node(RT_MAT_LAYERED, child=(i, o))
        else:
            raise RaytracerError(f"Unknown material type: {t}")  # scenes.ts:178
        if isinstance(ref, str):
            self._by_id[ref] = idx
        return idx
