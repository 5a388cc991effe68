"""ctypes binding of include/yuki_gpu.h (libyuki_gpu.so, built in-tree by build.sh / __graft_entry__.build()).

This is the reference-side binding a host would write (INTEGRATION.md shows the Rust `extern "C"`
equivalent). The library is required: there is no CPU fallback, and importing this module fails loudly
when the shared object is missing.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import desc as D

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("YUKI_GPU_LIB") or os.path.join(_HERE, "libyuki_gpu.so")  # override: A/B builds during development


ERR_CANCELLED = -5  # YK_ERR_CANCELLED


class YukiGpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"yuki_gpu error {code}: {msg}")
        self.code = code


# ---- structs (field order/layout == include/yuki_gpu.h) ---------------------------------------------
class Transform(C.Structure):
    _fields_ = [("m", C.c_float * 16), ("m_inv", C.c_float * 16)]


class CameraParams(C.Structure):
    _fields_ = [("position", C.c_float * 3), ("target", C.c_float * 3), ("up", C.c_float * 3),
                ("fov_axis", C.c_uint32), ("fov_deg", C.c_float)]


class Camera(C.Structure):
    _fields_ = [("camera_to_world", C.c_float * 16), ("raster_to_camera", C.c_float * 16)]


class FilmSettings(C.Structure):
    _fields_ = [("res_x", C.c_uint32), ("res_y", C.c_uint32), ("tile_dim", C.c_uint32), ("accumulate", C.c_uint32)]


class Sampler(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("nx", C.c_uint32), ("ny", C.c_uint32), ("jitter", C.c_uint32), ("seed", C.c_uint64)]


class Integrator(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("max_depth", C.c_uint32), ("has_clamp", C.c_uint32), ("indirect_clamp", C.c_float)]


class Tile(C.Structure):
    _fields_ = [("x0", C.c_uint16), ("y0", C.c_uint16), ("x1", C.c_uint16), ("y1", C.c_uint16),
                ("sample", C.c_uint16), ("_pad", C.c_uint16), ("index", C.c_uint32)]


# yk_integrator_ray (integrators/mod.rs:76-89): ray_type 0 direct, 1 reflection, 2 refraction, 3 normal, 4 shadow
DEBUG_RAY_DTYPE = np.dtype([("o", "<f4", (3,)), ("d", "<f4", (3,)), ("t_max", "<f4"), ("ray_type", "<u4")])
TILE_DTYPE = np.dtype([("x0", "<u2"), ("y0", "<u2"), ("x1", "<u2"), ("y1", "<u2"), ("sample", "<u2"), ("_pad", "<u2"),
                       ("index", "<u4")])


class BvhNode(C.Structure):
    _fields_ = [("p_min", C.c_float * 3), ("p_max", C.c_float * 3), ("offset", C.c_uint32), ("shape_count", C.c_uint16),
                ("split_axis", C.c_uint8), ("is_leaf", C.c_uint8)]


NODE_DTYPE = np.dtype([("p_min", "<f4", 3), ("p_max", "<f4", 3), ("offset", "<u4"), ("shape_count", "<u2"),
                       ("split_axis", "u1"), ("is_leaf", "u1")])


class TextureDesc(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("value", C.c_float * 3), ("width", C.c_uint32), ("height", C.c_uint32),
                ("texels", C.POINTER(C.c_float))]


class MaterialDesc(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("tex", C.c_int32 * 3), ("eta", C.c_float), ("remap_roughness", C.c_uint32)]


class LightDesc(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("light_to_world", Transform), ("intensity", C.c_float * 3),
                ("total_width_deg", C.c_float), ("falloff_start_deg", C.c_float), ("size", C.c_float * 2),
                ("direction", C.c_float * 3)]


class MeshDesc(C.Structure):
    _fields_ = [("object_to_world", Transform), ("n_points", C.c_uint32), ("n_indices", C.c_uint32),
                ("points", C.POINTER(C.c_float)), ("normals", C.POINTER(C.c_float)), ("uvs", C.POINTER(C.c_float)),
                ("indices", C.POINTER(C.c_uint32)), ("material", C.c_int32), ("area_light", C.c_int32)]


class SphereDesc(C.Structure):
    _fields_ = [("object_to_world", Transform), ("radius", C.c_float), ("material", C.c_int32)]


class HostSceneDesc(C.Structure):
    _fields_ = [("n_meshes", C.c_uint32), ("n_textures", C.c_uint32), ("n_materials", C.c_uint32), ("n_lights", C.c_uint32),
                ("meshes", C.POINTER(MeshDesc)), ("textures", C.POINTER(TextureDesc)), ("materials", C.POINTER(MaterialDesc)),
                ("lights", C.POINTER(LightDesc)), ("background", C.c_float * 3), ("max_shapes_in_node", C.c_uint32),
                ("split_method", C.c_uint32), ("n_spheres", C.c_uint32), ("spheres", C.POINTER(SphereDesc)),
                ("n_objects", C.c_uint32), ("objects", C.POINTER(C.c_int32))]


class PbrtResult(C.Structure):
    _fields_ = [("scene", HostSceneDesc), ("camera", CameraParams), ("res_x", C.c_uint32), ("res_y", C.c_uint32)]


class SphereDev(C.Structure):
    _fields_ = [("object_to_world", C.c_float * 16), ("world_to_object", C.c_float * 16), ("radius", C.c_float),
                ("swaps_handedness", C.c_uint32)]


class LightDev(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("p", C.c_float * 3), ("i", C.c_float * 3), ("cos_total_width", C.c_float),
                ("cos_falloff_start", C.c_float), ("world_to_light", C.c_float * 16), ("sample_to_world", C.c_float * 16),
                ("sample_to_world_inv", C.c_float * 16), ("area", C.c_float)]


class SceneDescFlat(C.Structure):
    _fields_ = [("n_nodes", C.c_uint32), ("nodes", C.POINTER(BvhNode)), ("n_tris", C.c_uint32),
                ("tri_vertices", C.POINTER(C.c_float)), ("tri_normals", C.POINTER(C.c_float)), ("tri_uvs", C.POINTER(C.c_float)),
                ("tri_orig_id", C.POINTER(C.c_uint32)), ("tri_material", C.POINTER(C.c_uint32)),
                ("tri_area_light", C.POINTER(C.c_int32)), ("tri_flags", C.POINTER(C.c_uint8)),
                ("n_textures", C.c_uint32), ("n_materials", C.c_uint32), ("n_lights", C.c_uint32),
                ("textures", C.POINTER(TextureDesc)), ("materials", C.POINTER(MaterialDesc)), ("lights", C.POINTER(LightDev)),
                ("background", C.c_float * 3), ("n_spheres", C.c_uint32), ("spheres", C.POINTER(SphereDev)),
                ("tri_sphere", C.POINTER(C.c_int32))]


PROGRESS_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_uint64, C.c_uint64)


class PlyData(C.Structure):
    _fields_ = [("n_points", C.c_uint32), ("n_indices", C.c_uint32), ("points", C.POINTER(C.c_float)),
                ("normals", C.POINTER(C.c_float)), ("uvs", C.POINTER(C.c_float)), ("indices", C.POINTER(C.c_uint32))]


class RenderOpts(C.Structure):
    _fields_ = [("flags", C.c_uint32), ("wavefront_paths", C.c_uint32), ("hit_ids", C.c_void_p), ("aux_sample", C.c_uint32),
                ("pipes", C.c_uint32), ("progress", PROGRESS_FN), ("progress_user", C.c_void_p), ("ray_sort", C.c_uint32),
                ("_reserved", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [("ray_count", C.c_uint64), ("shadow_rays", C.c_uint64), ("samples", C.c_uint64),
                ("closest_nodes", C.c_uint64), ("closest_tris", C.c_uint64), ("any_nodes", C.c_uint64), ("any_tris", C.c_uint64),
                ("primary_hit_hash", C.c_uint64), ("seconds", C.c_double), ("device_ms", C.c_double),
                ("trace_closest_ms", C.c_double), ("trace_any_ms", C.c_double), ("shade_ms", C.c_double),
                ("kernel_launches", C.c_uint64), ("trace_closest_launches", C.c_uint64)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


RENDER_FILM_ON_DEVICE = 1
QUERY_ON_DEVICE = 1


class QueryOpts(C.Structure):
    _fields_ = [("flags", C.c_uint32), ("_reserved", C.c_uint32), ("stream", C.c_void_p)]


class Hits(C.Structure):
    """yk_hits: output pointers of yk_query_intersect (NULL = not produced)."""
    _fields_ = [("t", C.c_void_p), ("orig_id", C.c_void_p), ("counts", C.c_void_p), ("material", C.c_void_p),
                ("area_light", C.c_void_p), ("p", C.c_void_p), ("n", C.c_void_p), ("uv", C.c_void_p), ("shading_n", C.c_void_p),
                ("shading_dpdu", C.c_void_p)]

# Every symbol include/yuki_gpu.h declares (checked by tests/test_abi.py).
EXPORTS = [
    "yk_last_error", "yk_context_create", "yk_context_destroy", "yk_scene_create", "yk_scene_destroy", "yk_render",
    "yk_context_stream", "yk_bvh_build", "yk_host_scene_build", "yk_host_scene_destroy", "yk_host_scene_flat", "yk_camera_make",
    "yk_film_tiles", "yk_xf_identity", "yk_xf_translation", "yk_xf_scale", "yk_xf_rotation", "yk_xf_new", "yk_xf_look_at",
    "yk_xf_mul", "yk_xf_inverted", "yk_xf_point", "yk_xf_vec", "yk_xf_normal", "yk_light_make", "yk_selftest_fastdiv", "yk_ply_load", "yk_ply_view", "yk_ply_destroy", "yk_write_exr", "yk_tonemap_filmic", "yk_heatmap", "yk_pbrt_load", "yk_pbrt_view", "yk_pbrt_destroy", "yk_mitsuba_load",
    "yk_debug_ray", "yk_trace", "yk_occluded", "yk_query_intersect", "yk_query_occluded", "yk_sampler_draws",
    "yk_multi_create", "yk_multi_destroy", "yk_multi_device_count", "yk_multi_context", "yk_multi_peer_stores",
    "yk_multi_scene_create", "yk_multi_scene_destroy", "yk_multi_render",
]

_lib = None


def lib():
    """Loads libyuki_gpu.so. Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: run ./build.sh (or __graft_entry__.build()); there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    fp, vp, u32 = C.POINTER(C.c_float), C.c_void_p, C.c_uint32
    L.yk_last_error.restype = C.c_char_p
    L.yk_context_create.argtypes = [C.c_int, C.POINTER(vp)]
    L.yk_context_destroy.argtypes = [vp]
    L.yk_context_destroy.restype = None
    L.yk_context_stream.argtypes = [vp]
    L.yk_context_stream.restype = vp
    L.yk_scene_create.argtypes = [vp, C.POINTER(SceneDescFlat), C.POINTER(vp)]
    L.yk_scene_destroy.argtypes = [vp]
    L.yk_scene_destroy.restype = None
    L.yk_render.argtypes = [vp, vp, C.POINTER(Camera), C.POINTER(FilmSettings), C.POINTER(Sampler), C.POINTER(Integrator),
                            vp, u32, C.POINTER(RenderOpts), vp, C.POINTER(Stats)]
    L.yk_debug_ray.argtypes = [vp, vp, C.POINTER(Camera), C.POINTER(Sampler), C.POINTER(Integrator), u32, u32, vp, u32,
                               C.POINTER(u32), fp, C.POINTER(C.c_uint64)]
    L.yk_trace.argtypes = [vp, vp, fp, fp, fp, u32, fp, vp, vp]
    L.yk_occluded.argtypes = [vp, vp, fp, fp, u32, vp]
    L.yk_query_intersect.argtypes = [vp, vp, vp, vp, vp, u32, C.POINTER(QueryOpts), C.POINTER(Hits)]
    L.yk_query_occluded.argtypes = [vp, vp, vp, vp, u32, C.POINTER(QueryOpts), vp]
    L.yk_sampler_draws.argtypes = [vp, C.POINTER(Sampler), vp, u32, C.c_char_p, u32, fp]
    L.yk_bvh_build.argtypes = [fp, u32, u32, u32, vp, C.POINTER(u32), C.POINTER(u32)]
    L.yk_host_scene_build.argtypes = [C.POINTER(HostSceneDesc), C.POINTER(vp)]
    L.yk_host_scene_destroy.argtypes = [vp]
    L.yk_host_scene_destroy.restype = None
    L.yk_host_scene_flat.argtypes = [vp, C.POINTER(SceneDescFlat)]
    L.yk_host_scene_flat.restype = None
    L.yk_camera_make.argtypes = [C.POINTER(CameraParams), u32, u32, C.POINTER(Camera)]
    L.yk_film_tiles.argtypes = [u32, u32, u32, vp, u32]
    L.yk_film_tiles.restype = u32
    L.yk_write_exr.argtypes = [C.c_char_p, u32, u32, fp]
    L.yk_tonemap_filmic.argtypes = [vp, fp, u32, u32, fp, u32, u32, C.c_float, fp]
    L.yk_heatmap.argtypes = [vp, fp, u32, u32, u32, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float), fp]
    L.yk_pbrt_load.argtypes = [C.c_char_p, u32, u32, C.POINTER(vp)]
    L.yk_mitsuba_load.argtypes = [C.c_char_p, u32, u32, C.POINTER(vp)]
    L.yk_pbrt_view.argtypes = [vp]
    L.yk_pbrt_view.restype = C.POINTER(PbrtResult)
    L.yk_pbrt_destroy.argtypes = [vp]
    L.yk_pbrt_destroy.restype = None
    L.yk_ply_load.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.yk_ply_view.argtypes = [vp, C.POINTER(PlyData)]
    L.yk_ply_view.restype = None
    L.yk_ply_destroy.argtypes = [vp]
    L.yk_ply_destroy.restype = None
    L.yk_selftest_fastdiv.argtypes = [u32, vp, C.c_uint64]
    L.yk_selftest_fastdiv.restype = C.c_uint64
    T = C.POINTER(Transform)
    L.yk_xf_identity.argtypes = [T]
    L.yk_xf_translation.argtypes = [fp, T]
    L.yk_xf_scale.argtypes = [C.c_float, C.c_float, C.c_float, T]
    L.yk_xf_rotation.argtypes = [C.c_float, fp, T]
    L.yk_xf_new.argtypes = [fp, T]
    L.yk_xf_look_at.argtypes = [fp, fp, fp, T]
    L.yk_xf_mul.argtypes = [T, T, T]
    L.yk_xf_inverted.argtypes = [T, T]
    for n in ("yk_xf_point", "yk_xf_vec", "yk_xf_normal"):
        getattr(L, n).argtypes = [T, fp, fp]
        getattr(L, n).restype = None
    for n in ("yk_xf_identity", "yk_xf_translation", "yk_xf_scale", "yk_xf_rotation", "yk_xf_mul", "yk_xf_inverted"):
        getattr(L, n).restype = None
    L.yk_light_make.argtypes = [C.POINTER(LightDesc), C.POINTER(LightDev)]
    if not hasattr(L, "yk_multi_create"):   # an older development build selected with YUKI_GPU_LIB (A/B runs): no device groups
        _lib = L
        return L
    L.yk_multi_create.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]
    L.yk_multi_destroy.argtypes = [vp]
    L.yk_multi_destroy.restype = None
    L.yk_multi_device_count.argtypes = [vp]
    L.yk_multi_context.argtypes = [vp, C.c_int]
    L.yk_multi_context.restype = vp
    L.yk_multi_peer_stores.argtypes = [vp, C.c_int]
    L.yk_multi_scene_create.argtypes = [vp, C.POINTER(SceneDescFlat), C.POINTER(vp)]
    L.yk_multi_scene_destroy.argtypes = [vp]
    L.yk_multi_scene_destroy.restype = None
    L.yk_multi_render.argtypes = [vp, vp, C.POINTER(Camera), C.POINTER(FilmSettings), C.POINTER(Sampler), C.POINTER(Integrator),
                                  vp, u32, C.POINTER(RenderOpts), vp, C.POINTER(Stats), C.POINTER(Stats)]
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise YukiGpuError(rc, lib().yk_last_error().decode("utf-8", "replace"))


# ---- conversions from the plain-Python description ---------------------------------------------------
def f3(v):
    return (C.c_float * 3)(*[float(x) for x in v])


def fptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def to_c_transform(t: D.Transform, cls=Transform):
    out = cls()
    C.memmove(out.m, np.ascontiguousarray(t.m, np.float32).ctypes.data, 64)
    C.memmove(out.m_inv, np.ascontiguousarray(t.m_inv, np.float32).ctypes.data, 64)
    return out


def from_c_transform(t) -> D.Transform:
    return D.Transform(np.array(t.m, dtype=np.float32), np.array(t.m_inv, dtype=np.float32))


def build_host_scene_desc(scene: D.SceneDesc, S=None):
    """SceneDesc -> (HostSceneDesc, keepalive). `S` lets the oracle binding reuse this with its own
    (layout-identical) struct classes."""
    S = S or {"host": HostSceneDesc, "mesh": MeshDesc, "tex": TextureDesc, "mat": MaterialDesc, "light": LightDesc,
              "xf": Transform, "sphere": SphereDesc}
    keep = []
    meshes = (S["mesh"] * max(len(scene.meshes), 1))()
    for i, m in enumerate(scene.meshes):
        pts = np.ascontiguousarray(m.points, np.float32).reshape(-1, 3)
        idx = np.ascontiguousarray(m.indices, np.uint32).reshape(-1)
        keep += [pts, idx]
        md = meshes[i]
        md.object_to_world = to_c_transform(m.object_to_world, S["xf"])
        md.n_points = pts.shape[0]
        md.n_indices = idx.shape[0]
        md.points = fptr(pts)
        md.indices = idx.ctypes.data_as(C.POINTER(C.c_uint32))
        if m.normals is not None:
            nrm = np.ascontiguousarray(m.normals, np.float32).reshape(-1, 3)
            assert nrm.shape[0] == pts.shape[0]
            keep.append(nrm)
            md.normals = fptr(nrm)
        if m.uvs is not None:
            uv = np.ascontiguousarray(m.uvs, np.float32).reshape(-1, 2)
            assert uv.shape[0] == pts.shape[0]
            keep.append(uv)
            md.uvs = fptr(uv)
        md.material = m.material
        md.area_light = m.area_light
    texs = (S["tex"] * max(len(scene.textures), 1))()
    for i, t in enumerate(scene.textures):
        td = texs[i]
        td.kind = t.kind
        td.value = f3(t.value)
        if t.kind == D.TEX_IMAGE:
            img = np.ascontiguousarray(t.image, np.float32)
            assert img.ndim == 3 and img.shape[2] == 3
            keep.append(img)
            td.height, td.width = img.shape[0], img.shape[1]
            td.texels = fptr(img)
    mats = (S["mat"] * max(len(scene.materials), 1))()
    for i, m in enumerate(scene.materials):
        md = mats[i]
        md.kind = m.kind
        tex = list(m.tex) + [0] * (3 - len(m.tex))
        md.tex = (C.c_int32 * 3)(*tex)
        md.eta = m.eta
        md.remap_roughness = 1 if m.remap_roughness else 0
    lights = (S["light"] * max(len(scene.lights), 1))()
    for i, l in enumerate(scene.lights):
        ld = lights[i]
        ld.kind = l.kind
        ld.light_to_world = to_c_transform(l.light_to_world, S["xf"])
        ld.intensity = f3(l.intensity)
        ld.total_width_deg = l.total_width_deg
        ld.falloff_start_deg = l.falloff_start_deg
        ld.size = (C.c_float * 2)(*[float(x) for x in l.size])
        ld.direction = f3(l.direction)
    hd = S["host"]()
    hd.n_meshes, hd.n_textures, hd.n_materials, hd.n_lights = len(scene.meshes), len(scene.textures), len(scene.materials), len(scene.lights)
    hd.meshes, hd.textures, hd.materials, hd.lights = meshes, texs, mats, lights
    spheres = (S["sphere"] * max(len(scene.spheres), 1))()
    for i, sp in enumerate(scene.spheres):
        spheres[i].object_to_world = to_c_transform(sp.object_to_world, S["xf"])
        spheres[i].radius = float(sp.radius)
        spheres[i].material = int(sp.material)
    hd.n_spheres = len(scene.spheres)
    hd.spheres = spheres
    keep.append(spheres)
    if scene.objects is not None:
        objs = np.ascontiguousarray(scene.objects, np.int32)
        keep.append(objs)
        hd.n_objects = len(objs)
        hd.objects = objs.ctypes.data_as(C.POINTER(C.c_int32))
    hd.background = f3(scene.background)
    hd.max_shapes_in_node = scene.max_shapes_in_node
    hd.split_method = scene.split_method
    keep += [meshes, texs, mats, lights]
    return hd, keep


def camera_params(p: D.CameraParameters, cls=CameraParams):
    cp = cls()
    cp.position, cp.target, cp.up = f3(p.position), f3(p.target), f3(p.up)
    cp.fov_axis, cp.fov_deg = p.fov_axis, p.fov_deg
    return cp


def film_settings(f: D.FilmSettings, cls=FilmSettings):
    return cls(int(f.res[0]), int(f.res[1]), int(f.tile_dim), 1 if f.accumulate else 0)


def sampler(s: D.SamplerType, cls=Sampler):
    return cls(s.kind, s.nx, s.ny, 1 if s.jitter else 0, s.seed)


def integrator(i: D.IntegratorType, cls=Integrator):
    return cls(i.kind, i.max_depth, 0 if i.indirect_clamp is None else 1, 0.0 if i.indirect_clamp is None else i.indirect_clamp)
