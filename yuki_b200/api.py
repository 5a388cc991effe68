"""Host-side mirror of the reference interface for the hot path, over the C ABI.

Names follow yuki: `Scene` (scene/mod.rs:41-49), `Camera` (camera.rs:52), `film_tiles` (film.rs:409),
`Renderer` (renderer/mod.rs:131-177, here blocking: the call returns when the film is complete),
`IntegratorType` / `SamplerType` / `FilmSettings` (desc.py). The GPU does the per-pixel work; this module
only marshals descriptors. It fails loudly when the CUDA library or a GPU is missing.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
import time
from dataclasses import dataclass
from typing import Optional

import numpy as np

from . import capi
from . import desc as D


class Context:
    """One CUDA device + stream (`yk_context`)."""

    def __init__(self, device_id: int = 0):
        self._h = C.c_void_p()
        capi.check(capi.lib().yk_context_create(device_id, C.byref(self._h)))
        self.device_id = device_id

    def close(self):
        if self._h:
            capi.lib().yk_context_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class HostScene:
    """Mesh::new + Triangle::new + BoundingVolumeHierarchy::new + flattening, on the host (no GPU)."""

    def __init__(self, scene: D.SceneDesc):
        hd, keep = capi.build_host_scene_desc(scene)
        self._h = C.c_void_p()
        capi.check(capi.lib().yk_host_scene_build(C.byref(hd), C.byref(self._h)))
        del keep
        self.flat = capi.SceneDescFlat()
        capi.lib().yk_host_scene_flat(self._h, C.byref(self.flat))

    @property
    def n_nodes(self):
        return self.flat.n_nodes

    @property
    def n_tris(self):
        return self.flat.n_tris

    def nodes(self) -> np.ndarray:
        buf = C.string_at(self.flat.nodes, self.flat.n_nodes * 32)
        return np.frombuffer(buf, dtype=capi.NODE_DTYPE).copy()

    def order(self) -> np.ndarray:
        return np.ctypeslib.as_array(self.flat.tri_orig_id, shape=(self.flat.n_tris,)).copy()

    def tri_vertices(self) -> np.ndarray:
        return np.ctypeslib.as_array(self.flat.tri_vertices, shape=(self.flat.n_tris, 3, 3)).copy()

    # ---- one host build shared by the ranks of a node ---------------------------------------------------------------
    # The BVH build is the slow host step (6 s for 10 M triangles); with one process per GPU every rank would repeat it.
    # `save` writes the flattened arrays (the exact bytes yk_scene_create takes) as .npy files, e.g. under /dev/shm;
    # `load` maps them back without copying, so N ranks share one build and one page-cache copy.
    _ARRAYS = (("nodes", "n_nodes", 32, np.uint8), ("tri_vertices", "n_tris", 9, np.float32), ("tri_normals", "n_tris", 9, np.float32),
               ("tri_uvs", "n_tris", 6, np.float32), ("tri_orig_id", "n_tris", 1, np.uint32), ("tri_material", "n_tris", 1, np.uint32),
               ("tri_area_light", "n_tris", 1, np.int32), ("tri_flags", "n_tris", 1, np.uint8), ("tri_sphere", "n_tris", 1, np.int32))

    def save(self, directory: str):
        import json
        os.makedirs(directory, exist_ok=True)
        for stale in os.listdir(directory):   # a directory holds one scene
            if stale.endswith(".npy") or stale.startswith("tables.json"):
                os.remove(os.path.join(directory, stale))
        f = self.flat
        for name, count, per, dtype in self._ARRAYS:
            ptr = getattr(f, name)
            if not ptr:
                continue
            n = getattr(f, count) * per
            arr = np.frombuffer(C.string_at(C.cast(ptr, C.c_void_p), n * np.dtype(dtype).itemsize), dtype=dtype)
            np.save(os.path.join(directory, name + ".npy"), arr)
        tables = {"n_nodes": f.n_nodes, "n_tris": f.n_tris, "background": [float(v) for v in f.background],
                  "materials": C.string_at(C.cast(f.materials, C.c_void_p), f.n_materials * C.sizeof(capi.MaterialDesc)).hex() if f.n_materials else "",
                  "lights": C.string_at(C.cast(f.lights, C.c_void_p), f.n_lights * C.sizeof(capi.LightDev)).hex() if f.n_lights else "",
                  "spheres": C.string_at(C.cast(f.spheres, C.c_void_p), f.n_spheres * C.sizeof(capi.SphereDev)).hex() if f.n_spheres else "",
                  "n_materials": f.n_materials, "n_lights": f.n_lights, "n_spheres": f.n_spheres, "textures": []}
        for i in range(f.n_textures):
            t = f.textures[i]
            tables["textures"].append({"kind": t.kind, "value": [float(v) for v in t.value], "width": t.width, "height": t.height})
            if t.kind == D.TEX_IMAGE:
                np.save(os.path.join(directory, f"texture{i}.npy"), np.ctypeslib.as_array(t.texels, shape=(t.height * t.width * 3,)).copy())
        tmp = os.path.join(directory, "tables.json.tmp")
        with open(tmp, "w") as fh:
            json.dump(tables, fh)
        os.replace(tmp, os.path.join(directory, "tables.json"))   # written last: its presence marks a complete directory

    @classmethod
    def load(cls, directory: str) -> "HostScene":
        import json
        with open(os.path.join(directory, "tables.json")) as fh:
            tables = json.load(fh)
        self = cls.__new__(cls)
        self._h = C.c_void_p()
        keep = []
        f = capi.SceneDescFlat()
        f.n_nodes, f.n_tris = tables["n_nodes"], tables["n_tris"]
        for name, _count, _per, _dtype in cls._ARRAYS:
            path = os.path.join(directory, name + ".npy")
            if os.path.exists(path):
                arr = np.load(path, mmap_mode="r")
                keep.append(arr)
                field_type = dict(capi.SceneDescFlat._fields_)[name]
                setattr(f, name, C.cast(C.c_void_p(arr.ctypes.data), field_type))
        def table(key, struct, n):
            if not n:
                return None
            buf = (struct * n).from_buffer_copy(bytes.fromhex(tables[key]))
            keep.append(buf)
            return buf
        f.n_materials, f.n_lights, f.n_spheres = tables["n_materials"], tables["n_lights"], tables["n_spheres"]
        mats, lights, spheres = table("materials", capi.MaterialDesc, f.n_materials), table("lights", capi.LightDev, f.n_lights), table("spheres", capi.SphereDev, f.n_spheres)
        if mats is not None:
            f.materials = C.cast(mats, C.POINTER(capi.MaterialDesc))
        if lights is not None:
            f.lights = C.cast(lights, C.POINTER(capi.LightDev))
        if spheres is not None:
            f.spheres = C.cast(spheres, C.POINTER(capi.SphereDev))
        f.n_textures = len(tables["textures"])
        if f.n_textures:
            tex = (capi.TextureDesc * f.n_textures)()
            for i, t in enumerate(tables["textures"]):
                tex[i].kind, tex[i].width, tex[i].height = t["kind"], t["width"], t["height"]
                tex[i].value[:] = t["value"]
                if t["kind"] == D.TEX_IMAGE:
                    texels = np.load(os.path.join(directory, f"texture{i}.npy"), mmap_mode="r")
                    keep.append(texels)
                    tex[i].texels = C.cast(C.c_void_p(texels.ctypes.data), C.POINTER(C.c_float))
            keep.append(tex)
            f.textures = C.cast(tex, C.POINTER(capi.TextureDesc))
        f.background[:] = tables["background"]
        self.flat = f
        self._keep = keep
        return self

    def close(self):
        if self._h:
            capi.lib().yk_host_scene_destroy(self._h)
            self._h = C.c_void_p()
        self._keep = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


HIT_FIELDS = ("t", "orig_id", "material", "area_light", "p", "n", "uv", "shading_n", "shading_dpdu")
_HIT_SHAPES = {"t": ((), np.float32), "orig_id": ((), np.int32), "material": ((), np.int32), "area_light": ((), np.int32),
               "p": ((3,), np.float32), "n": ((3,), np.float32), "uv": ((2,), np.float32), "shading_n": ((3,), np.float32),
               "shading_dpdu": ((3,), np.float32)}


@dataclass
class Hits:
    """`Scene::intersect`'s Hit for a batch of rays (numpy arrays, or torch tensors on the GPU when the rays were): hit distance
    (inf on a miss), original shape id and material index (-1 on a miss), and the SurfaceInteraction's area light (-1 for
    none), p, geometric normal n, uv, shading normal and shading dpdu (0 on a miss)."""
    t: object
    orig_id: object
    material: object
    area_light: object
    p: object
    n: object
    uv: object
    shading_n: object
    shading_dpdu: object


def _cuda_rays(ctx, arrays):
    """The torch module when any of `arrays` is a CUDA tensor (then all must be float32 CUDA tensors on the context's device),
    else None: host input keeps the numpy path. torch is only imported by callers that already hold tensors."""
    import sys
    torch = sys.modules.get("torch")
    if torch is None:
        return None
    given = [a for a in arrays if a is not None]
    if not any(isinstance(a, torch.Tensor) and a.is_cuda for a in given):
        return None
    for a in given:
        if not (isinstance(a, torch.Tensor) and a.is_cuda):
            raise TypeError(f"rays mix CUDA tensors with {type(a).__name__} ({getattr(a, 'device', 'host')}): pass o, d and t_max "
                            "all as CUDA tensors or all as host arrays")
        if a.dtype != torch.float32:
            raise TypeError(f"ray tensors must be float32, got {a.dtype}")
        if a.device.index != ctx.device_id:
            raise ValueError(f"ray tensor on {a.device}, but the scene's context is on cuda:{ctx.device_id}")
    return torch


def _device_rays(torch, o, d, t_max):
    if o.dim() != 2 or o.shape[1] != 3 or d.shape != o.shape:
        raise ValueError(f"o and d must have shape (n, 3), got {tuple(o.shape)} and {tuple(d.shape)}")
    n = o.shape[0]
    if t_max is not None and tuple(t_max.shape) != (n,):
        raise ValueError(f"t_max must have shape ({n},), got {tuple(t_max.shape)}")
    return o.contiguous(), d.contiguous(), None if t_max is None else t_max.contiguous(), n


def _device_opts(torch, ctx):
    return capi.QueryOpts(capi.QUERY_ON_DEVICE, 0, torch.cuda.current_stream(ctx.device_id).cuda_stream)


def _ptr(a):
    if a is None:
        return None
    return a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data


class Scene:
    """Device-resident scene (`yk_scene`): SoA node / triangle / material / light / texture buffers in HBM."""

    def __init__(self, ctx: Context, scene: D.SceneDesc, host: Optional[HostScene] = None):
        self.ctx = ctx
        self.host = host or HostScene(scene)
        self._h = C.c_void_p()
        capi.check(capi.lib().yk_scene_create(ctx._h, C.byref(self.host.flat), C.byref(self._h)))

    def intersect(self, o, d, t_max=None, counts: bool = True):
        """`BoundingVolumeHierarchy::intersect` (bvh.rs:160-232) for a batch of rays: (t, original shape id, (tests, hits)
        node counters); t = inf and id = -1 on a miss. Rays held as float32 CUDA tensors on the context's device are traced
        in place, ordered after the current torch stream's work, and the results are tensors on that device."""
        torch = _cuda_rays(self.ctx, (o, d, t_max))
        if torch is not None:
            o, d, t_max, n = _device_rays(torch, o, d, t_max)
            dev = o.device
            t = torch.empty(n, dtype=torch.float32, device=dev)
            ids = torch.empty(n, dtype=torch.int32, device=dev)
            cnt = (torch.empty if counts else torch.zeros)((n, 2), dtype=torch.int32, device=dev).view(torch.uint32)
            hits = capi.Hits(t=_ptr(t), orig_id=_ptr(ids), counts=_ptr(cnt) if counts else None)
            capi.check(capi.lib().yk_query_intersect(self.ctx._h, self._h, _ptr(o), _ptr(d), _ptr(t_max), n,
                                                     C.byref(_device_opts(torch, self.ctx)), C.byref(hits)))
            return t, ids, cnt
        o = np.ascontiguousarray(o, np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(d, np.float32).reshape(-1, 3)
        n = o.shape[0]
        assert d.shape[0] == n
        t = np.zeros(n, np.float32)
        ids = np.zeros(n, np.int32)
        cnt = np.zeros((n, 2), np.uint32)
        tm = None
        if t_max is not None:
            tm_arr = np.ascontiguousarray(t_max, np.float32).reshape(-1)
            assert tm_arr.shape[0] == n
            tm = capi.fptr(tm_arr)
        capi.check(capi.lib().yk_trace(self.ctx._h, self._h, capi.fptr(o), capi.fptr(d), tm, n, capi.fptr(t), ids.ctypes.data,
                                       cnt.ctypes.data if counts else None))
        return t, ids, cnt

    def occluded(self, o, d):
        """`VisibilityTester::unoccluded` negated (visibility.rs:6-23) for a batch of segments o -> o + d (numpy, or CUDA
        tensors as in `intersect`)."""
        torch = _cuda_rays(self.ctx, (o, d))
        if torch is not None:
            o, d, _, n = _device_rays(torch, o, d, None)
            out = torch.empty(n, dtype=torch.uint8, device=o.device)
            capi.check(capi.lib().yk_query_occluded(self.ctx._h, self._h, _ptr(o), _ptr(d), n, C.byref(_device_opts(torch, self.ctx)),
                                                    _ptr(out)))
            return out
        o = np.ascontiguousarray(o, np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(d, np.float32).reshape(-1, 3)
        n = o.shape[0]
        assert d.shape[0] == n
        out = np.zeros(n, np.uint8)
        capi.check(capi.lib().yk_occluded(self.ctx._h, self._h, capi.fptr(o), capi.fptr(d), n, out.ctypes.data))
        return out

    def surface(self, o, d, t_max=None) -> Hits:
        """`Scene::intersect` (scene/mod.rs) for a batch of rays: the hit with its SurfaceInteraction, as a `Hits` record of
        numpy arrays, or of tensors on the GPU when the rays are CUDA tensors (see `intersect`)."""
        torch = _cuda_rays(self.ctx, (o, d, t_max))
        if torch is not None:
            o, d, t_max, n = _device_rays(torch, o, d, t_max)
            out = {k: torch.empty((n,) + shape, dtype=getattr(torch, np.dtype(dt).name), device=o.device) for k, (shape, dt) in _HIT_SHAPES.items()}
            opts = C.byref(_device_opts(torch, self.ctx))
        else:
            o = np.ascontiguousarray(o, np.float32).reshape(-1, 3)
            d = np.ascontiguousarray(d, np.float32).reshape(-1, 3)
            n = o.shape[0]
            if d.shape[0] != n:
                raise ValueError(f"o and d must have the same number of rays, got {n} and {d.shape[0]}")
            if t_max is not None:
                t_max = np.ascontiguousarray(t_max, np.float32).reshape(-1)
                if t_max.shape[0] != n:
                    raise ValueError(f"t_max must have {n} entries, got {t_max.shape[0]}")
            out = {k: np.zeros((n,) + shape, dt) for k, (shape, dt) in _HIT_SHAPES.items()}
            opts = None
        hits = capi.Hits(**{k: _ptr(v) for k, v in out.items()})
        capi.check(capi.lib().yk_query_intersect(self.ctx._h, self._h, _ptr(o), _ptr(d), _ptr(t_max), n, opts, C.byref(hits)))
        return Hits(**out)

    def close(self):
        if self._h:
            capi.lib().yk_scene_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiContext:
    """G devices of this process behind one handle (`yk_multi`): the counterpart of the reference's RenderManager with its
    workers and one shared tile queue (renderer/render_manager.rs:78-97, 197-236)."""

    def __init__(self, device_ids):
        ids = [int(d) for d in device_ids]
        arr = (C.c_int * len(ids))(*ids)
        self._h = C.c_void_p()
        capi.check(capi.lib().yk_multi_create(arr, len(ids), C.byref(self._h)))
        self.device_ids = ids

    @property
    def n_devices(self):
        return len(self.device_ids)

    def peer_stores(self):
        """Per device: does it store finished pixels straight into the first device's film (NVLink peer mapping)?"""
        return [bool(capi.lib().yk_multi_peer_stores(self._h, i)) for i in range(self.n_devices)]

    def close(self):
        if self._h:
            capi.lib().yk_multi_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiScene:
    """The scene replicated on every device of a MultiContext (validated once, uploaded in parallel)."""

    def __init__(self, mctx: MultiContext, scene: D.SceneDesc, host: Optional[HostScene] = None):
        self.mctx = mctx
        self.host = host or HostScene(scene)
        self._h = C.c_void_p()
        capi.check(capi.lib().yk_multi_scene_create(mctx._h, C.byref(self.host.flat), C.byref(self._h)))

    def close(self):
        if self._h:
            capi.lib().yk_multi_scene_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def multi_render(mctx: MultiContext, scene: MultiScene, camera_params: D.CameraParameters, film: D.FilmSettings, sampler: D.SamplerType,
                 integrator: D.IntegratorType, tiles: Optional[np.ndarray] = None, want_hit_ids: bool = False, aux_sample: int = 0,
                 film_out: Optional[np.ndarray] = None, device_film_ptr: Optional[int] = None, pipes: int = 0, ray_sort: int = 0,
                 wavefront_paths: int = 0):
    """`yk_multi_render`: the tile list rendered by all devices of the group, popped from one shared cursor; the film is
    assembled on the first device by peer stores. Returns (RenderResult with the summed stats, per-device stats list)."""
    cam = make_camera(camera_params, film)
    if tiles is None:
        tiles = film_tiles(film)
    tiles = np.ascontiguousarray(tiles, dtype=capi.TILE_DTYPE)
    res_x, res_y = int(film.res[0]), int(film.res[1])
    opts = capi.RenderOpts()
    opts.aux_sample = aux_sample
    opts.pipes = pipes
    opts.ray_sort = ray_sort
    opts.wavefront_paths = wavefront_paths
    hit_ids = None
    if device_film_ptr is not None:
        opts.flags |= capi.RENDER_FILM_ON_DEVICE
        film_arr, film_ptr = None, C.c_void_p(device_film_ptr)
    else:
        film_arr = film_out if film_out is not None else np.zeros((res_y, res_x, 3), dtype=np.float32)
        assert film_arr.dtype == np.float32 and film_arr.flags["C_CONTIGUOUS"] and film_arr.size == res_x * res_y * 3
        film_ptr = C.c_void_p(film_arr.ctypes.data)
        if want_hit_ids:
            hit_ids = np.full((res_y, res_x), -1, dtype=np.int32)
            opts.hit_ids = hit_ids.ctypes.data
    fs, sm, ig = capi.film_settings(film), capi.sampler(sampler), capi.integrator(integrator)
    stats = capi.Stats()
    per = (capi.Stats * mctx.n_devices)()
    capi.check(capi.lib().yk_multi_render(mctx._h, scene._h, C.byref(cam), C.byref(fs), C.byref(sm), C.byref(ig),
                                          C.c_void_p(tiles.ctypes.data), len(tiles), C.byref(opts), film_ptr, C.byref(stats), per))
    return RenderResult(film_arr, hit_ids, stats), list(per)


def sampler_draws(ctx: Context, sampler: D.SamplerType, pixel_index, pattern) -> np.ndarray:
    """`Sampler::{start_pixel_sample, get_1d, get_2d}` on the device: for every (x, y, sample index) row of `pixel_index`
    the draws of `pattern` (1 = get_1d, 2 = get_2d) after `start_pixel_sample(p, index, 0)`; returns (n, sum(pattern))."""
    pi = np.ascontiguousarray(pixel_index, np.uint32).reshape(-1, 3)
    pat = bytes(pattern)
    out = np.zeros((pi.shape[0], sum(pattern)), np.float32)
    sm = capi.sampler(sampler)
    capi.check(capi.lib().yk_sampler_draws(ctx._h, C.byref(sm), pi.ctypes.data, pi.shape[0], pat, len(pat), capi.fptr(out)))
    return out


def make_camera(params: D.CameraParameters, film: D.FilmSettings) -> capi.Camera:
    """Camera::new (camera.rs:52-102)."""
    cam = capi.Camera()
    cp = capi.camera_params(params)
    capi.check(capi.lib().yk_camera_make(C.byref(cp), int(film.res[0]), int(film.res[1]), C.byref(cam)))
    return cam


def film_tiles(film: D.FilmSettings) -> np.ndarray:
    """film_tiles (film.rs:409-475): all tiles of the film in outward-spiral order, as a TILE_DTYPE array."""
    L = capi.lib()
    n = L.yk_film_tiles(int(film.res[0]), int(film.res[1]), int(film.tile_dim), None, 0)
    out = np.zeros(n, dtype=capi.TILE_DTYPE)
    L.yk_film_tiles(int(film.res[0]), int(film.res[1]), int(film.tile_dim), out.ctypes.data, n)
    return out


def write_exr(path: str, film: np.ndarray):
    """app/util.rs `write_exr`: film (H, W, 3) f32 -> OpenEXR with float R, G, B channels."""
    film = np.ascontiguousarray(film, np.float32)
    assert film.ndim == 3 and film.shape[2] == 3
    capi.check(capi.lib().yk_write_exr(str(path).encode(), film.shape[1], film.shape[0], capi.fptr(film)))


def tonemap_filmic(ctx: Context, film: np.ndarray, exposure: float = 1.0, tile_samples: Optional[np.ndarray] = None,
                   tile_dim: int = 16) -> np.ndarray:
    """ToneMapType::Filmic (app/renderpasses/tonemap.rs:318-399). `tile_samples[flat_tile]` = Film::samples (film.rs:74)."""
    film = np.ascontiguousarray(film, np.float32)
    out = np.empty_like(film)
    ts, n_tiles = None, 0
    if tile_samples is not None:
        ts = np.ascontiguousarray(tile_samples, np.float32).reshape(-1)
        n_tiles = len(ts)
    capi.check(capi.lib().yk_tonemap_filmic(ctx._h, capi.fptr(film), film.shape[1], film.shape[0], capi.fptr(ts) if ts is not None else None,
                                             n_tiles, tile_dim, float(exposure), capi.fptr(out)))
    return out


def heatmap(ctx: Context, film: np.ndarray, channel: int = 0, value_range=None):
    """ToneMapType::Heatmap (app/renderpasses/tonemap.rs:401-432); value_range None = `find_min_max` (:447-472).
    Returns (image, (min, max))."""
    film = np.ascontiguousarray(film, np.float32)
    out = np.empty_like(film)
    lo = C.c_float(0.0 if value_range is None else value_range[0])
    hi = C.c_float(0.0 if value_range is None else value_range[1])
    capi.check(capi.lib().yk_heatmap(ctx._h, capi.fptr(film), film.shape[1], film.shape[0], int(channel), 1 if value_range is None else 0,
                                     C.byref(lo), C.byref(hi), capi.fptr(out)))
    return out, (lo.value, hi.value)


def load_pbrt(path: str, max_shapes_in_node: int = 1, split_method: int = D.SPLIT_SAH):
    """scene/pbrt/mod.rs `load`: pbrt-v3 file -> (SceneDesc, CameraParameters, FilmSettings), parsed by the C++ loader
    (csrc/host_pbrt.cpp). The description is copied out of the loader's storage, so it feeds the CUDA backend and the
    test oracle exactly like the programmatic scenes."""
    return _load_scene_file(capi.lib().yk_pbrt_load, path, max_shapes_in_node, split_method)


def load_mitsuba(path: str, max_shapes_in_node: int = 1, split_method: int = D.SPLIT_SAH):
    """scene/mitsuba/mod.rs `load`: Mitsuba 2.1.0 XML file -> (SceneDesc, CameraParameters, FilmSettings), parsed by the
    C++ loader (csrc/host_mitsuba.cpp)."""
    return _load_scene_file(capi.lib().yk_mitsuba_load, path, max_shapes_in_node, split_method)


def _load_scene_file(loader, path, max_shapes_in_node, split_method):
    h = C.c_void_p()
    capi.check(loader(str(path).encode(), int(max_shapes_in_node), int(split_method), C.byref(h)))
    try:
        r = capi.lib().yk_pbrt_view(h).contents
        hd = r.scene

        def xf(t):
            return D.Transform(np.array(t.m[:], np.float32), np.array(t.m_inv[:], np.float32))

        def arr(ptr, n, cols, dtype=np.float32):
            if not ptr or n == 0:
                return None
            return np.ctypeslib.as_array(ptr, shape=(n * cols,)).astype(dtype).reshape((n, cols) if cols > 1 else (n,)).copy()

        sc = D.SceneDesc(split_method=int(hd.split_method), max_shapes_in_node=int(hd.max_shapes_in_node),
                         background=tuple(float(v) for v in hd.background))
        for i in range(hd.n_textures):
            t = hd.textures[i]
            if t.kind == D.TEX_IMAGE:
                img = np.ctypeslib.as_array(t.texels, shape=(t.height, t.width, 3)).copy()
                sc.textures.append(D.Texture(D.TEX_IMAGE, (0.0, 0.0, 0.0), img))
            else:
                sc.textures.append(D.Texture(D.TEX_CONSTANT, tuple(float(v) for v in t.value)))
        for i in range(hd.n_materials):
            m = hd.materials[i]
            sc.materials.append(D.Material(int(m.kind), tuple(int(v) for v in m.tex), eta=float(m.eta), remap_roughness=bool(m.remap_roughness)))
        for i in range(hd.n_lights):
            l = hd.lights[i]
            sc.lights.append(D.Light(int(l.kind), xf(l.light_to_world), tuple(float(v) for v in l.intensity), float(l.total_width_deg),
                                     float(l.falloff_start_deg), tuple(float(v) for v in l.size), tuple(float(v) for v in l.direction)))
        for i in range(hd.n_meshes):
            m = hd.meshes[i]
            pts = arr(m.points, m.n_points, 3)
            sc.meshes.append(D.Mesh(xf(m.object_to_world), pts if pts is not None else np.zeros((0, 3), np.float32),
                                    arr(m.indices, m.n_indices, 1, np.uint32), int(m.material), normals=arr(m.normals, m.n_points, 3),
                                    uvs=arr(m.uvs, m.n_points, 2), area_light=int(m.area_light)))
        for i in range(hd.n_spheres):
            sp = hd.spheres[i]
            sc.spheres.append(D.Sphere(xf(sp.object_to_world), float(sp.radius), int(sp.material)))
        sc.objects = [int(hd.objects[i]) for i in range(hd.n_objects)]
        cam = D.CameraParameters(tuple(float(v) for v in r.camera.position), tuple(float(v) for v in r.camera.target),
                                 tuple(float(v) for v in r.camera.up), int(r.camera.fov_axis), float(r.camera.fov_deg))
        film = D.FilmSettings((int(r.res_x), int(r.res_y)), 16)
    finally:
        capi.lib().yk_pbrt_destroy(h)
    return sc, cam, film


def load_ply(path: str):
    """scene/ply.rs `load` up to the index buffer: returns (points (N,3), indices (T*3,), normals (N,3)|None, uvs (N,2)|None)."""
    h = C.c_void_p()
    capi.check(capi.lib().yk_ply_load(str(path).encode(), C.byref(h)))
    try:
        v = capi.PlyData()
        capi.lib().yk_ply_view(h, C.byref(v))
        pts = np.ctypeslib.as_array(v.points, shape=(v.n_points, 3)).copy() if v.n_points else np.zeros((0, 3), np.float32)
        idx = np.ctypeslib.as_array(v.indices, shape=(v.n_indices,)).copy() if v.n_indices else np.zeros((0,), np.uint32)
        nrm = np.ctypeslib.as_array(v.normals, shape=(v.n_points, 3)).copy() if v.normals and v.n_points else None
        uvs = np.ctypeslib.as_array(v.uvs, shape=(v.n_points, 2)).copy() if v.uvs and v.n_points else None
    finally:
        capi.lib().yk_ply_destroy(h)
    return pts, idx, nrm, uvs


def bvh_build(tri_vertices: np.ndarray, max_shapes_in_node=1, split_method=D.SPLIT_SAH):
    """BoundingVolumeHierarchy::new over world-space triangles (T,3,3) -> (nodes, order)."""
    v = np.ascontiguousarray(tri_vertices, np.float32).reshape(-1, 9)
    n = v.shape[0]
    nodes = np.zeros(max(2 * n - 1, 1), dtype=capi.NODE_DTYPE)
    order = np.zeros(n, dtype=np.uint32)
    n_nodes = C.c_uint32()
    capi.check(capi.lib().yk_bvh_build(capi.fptr(v), n, max_shapes_in_node, split_method, nodes.ctypes.data, C.byref(n_nodes),
                                        order.ctypes.data_as(C.POINTER(C.c_uint32))))
    return nodes[: n_nodes.value].copy(), order


class Film:
    """`Film` (film.rs:60-101): RGB f32 pixels, row-major, plus — for accumulating renders — the per-tile sample counts
    the tone-map pass divides by (`samples[tile.index]`, film.rs:74, 270)."""

    def __init__(self, settings: D.FilmSettings):
        self.settings = settings
        w, h = int(settings.res[0]), int(settings.res[1])
        self.pixels = np.zeros((h, w, 3), np.float32)
        n_tiles = ((w + settings.tile_dim - 1) // settings.tile_dim) * ((h + settings.tile_dim - 1) // settings.tile_dim)
        self.samples = np.zeros(n_tiles, np.uint32) if settings.accumulate else None   # Vec<u32>, film.rs:74
        self.dirty = False
        self.meta = None   # what was rendered into it (set by render_progressive / Film.load)

    def clear(self):
        self.pixels[...] = 0.0
        if self.samples is not None:
            self.samples[...] = 0
        self.dirty = True

    # ---- checkpoint / resume of an accumulating film (SURVEY.md §8f-4) -------------------------------------------
    # The reference keeps the film's running sum and `samples[tile.index]` (film.rs:74, 260-272) but never writes them
    # out. With seekable samplers a (pixel, sample index) evaluation does not depend on what was rendered before, so
    # the pair (sum, counts) is a complete checkpoint: rendering the missing sample indices into a restored film gives
    # the bits of an uninterrupted render (the film adds samples in ascending index order either way).
    def save(self, path: str, meta: Optional[dict] = None):
        """Writes pixels (+ per-tile sample counts and a small `meta` dict naming the render) to `path` (.npz) atomically:
        the file is complete or absent, never torn, so a render killed mid-checkpoint resumes from the previous one."""
        import json
        tmp = f"{path}.tmp.{os.getpid()}"
        arrays = {"pixels": self.pixels, "res": np.array(self.settings.res, np.int64), "tile_dim": np.array(self.settings.tile_dim, np.int64),
                  "accumulate": np.array(1 if self.settings.accumulate else 0, np.int64),
                  "meta": np.frombuffer(json.dumps(meta or {}, sort_keys=True).encode(), dtype=np.uint8)}
        if self.samples is not None:
            arrays["samples"] = self.samples
        with open(tmp, "wb") as f:
            np.savez(f, **arrays)
            f.flush()
            os.fsync(f.fileno())
        os.replace(tmp, path)

    @staticmethod
    def load(path: str, expect_meta: Optional[dict] = None) -> "Film":
        """Restores a film written by `save`. `expect_meta`, when given, must equal the stored dict (a checkpoint of another
        scene / sampler / integrator must not be continued)."""
        import json
        with np.load(path) as z:
            fs = D.FilmSettings((int(z["res"][0]), int(z["res"][1])), int(z["tile_dim"]), accumulate=bool(int(z["accumulate"])))
            film = Film(fs)
            if z["pixels"].shape != film.pixels.shape or z["pixels"].dtype != np.float32:
                raise ValueError(f"{path}: pixel array does not match the stored film settings")
            film.pixels[...] = z["pixels"]
            if film.samples is not None:
                if "samples" not in z or z["samples"].shape != film.samples.shape:
                    raise ValueError(f"{path}: per-tile sample counts missing or of the wrong size")
                if z["samples"].dtype.kind not in "ui":
                    raise ValueError(f"{path}: per-tile sample counts are not integers")
                film.samples[...] = z["samples"]
            meta = json.loads(bytes(z["meta"]).decode() or "{}")
        if expect_meta is not None and json.loads(json.dumps(expect_meta, sort_keys=True)) != meta:
            raise ValueError(f"{path}: checkpoint belongs to another render ({meta} != {expect_meta})")
        film.meta = meta
        film.dirty = True
        return film


def json_roundtrip(obj):
    """`obj` as it comes back from a JSON file (tuples become lists), for comparing in-memory and stored metadata."""
    import json
    return json.loads(json.dumps(obj, sort_keys=True))


@dataclass
class RenderProgress:        # RenderStatus::Progress, renderer/mod.rs:21-28
    active_threads: int
    tiles_done: int
    tiles_total: int
    approx_remaining_s: float
    current_rays_per_s: float


@dataclass
class RenderFinished:        # RenderStatus::Finished, renderer/mod.rs:29-31
    ray_count: int


class RenderResult:
    def __init__(self, film, hit_ids, stats):
        self.film = film
        self.hit_ids = hit_ids
        self.stats = stats


class Renderer:
    """Blocking counterpart of `Renderer::launch` + `check_status` (renderer/mod.rs:61-177): renders the given
    tiles (default: the whole spiral list) with the wavefront CUDA path and returns the film."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        self._thread = None
        self._lock = threading.Lock()
        self._kill = False
        self._render_id = 0
        self._messages = []
        self._in_progress = False
        self.last_result = None
        self.last_error = None

    # ---- the reference's asynchronous surface: launch / check_status / kill (renderer/mod.rs:53-177) ----
    def is_active(self) -> bool:
        return self._in_progress

    def launch(self, scene: Scene, camera_params: D.CameraParameters, film: Film, sampler: D.SamplerType, integrator: D.IntegratorType,
               film_settings: Optional[D.FilmSettings] = None, force_single_sample: bool = False, **render_kw):
        """Starts a render into `film` on a background thread, overriding a running one (renderer/mod.rs:131-177).
        Accumulating film settings render one tile list per sample index, in order (render_manager.rs:135-143) and add
        into the film; otherwise the film's tiles are overwritten with the per-pixel mean."""
        self.kill()
        fs = film_settings or film.settings
        assert tuple(fs.res) == tuple(film.settings.res), "Film does not match settings"   # film.rs:421
        if force_single_sample:   # SamplerType::instantiate(force_single_sample), sampling/mod.rs:21-42
            sampler = D.SamplerType(kind=sampler.kind, nx=1, ny=1, jitter=sampler.jitter, seed=sampler.seed)
        base = film_tiles(fs)
        if fs.accumulate:
            tiles = []
            for smp in range(sampler.samples_per_pixel()):
                t = base.copy()
                t["sample"] = smp
                tiles.append(t)
            tiles = np.concatenate(tiles)
        else:
            tiles = base
        self._render_id += 1
        rid = self._render_id
        self._kill = False
        self._in_progress = True
        self.last_result = None
        self.last_error = None
        t0 = time.perf_counter()

        def progress(done, total):
            now = time.perf_counter() - t0
            frac = done / max(total, 1)
            with self._lock:
                if rid == self._render_id:
                    self._messages.append(RenderProgress(1, int(frac * len(tiles)), len(tiles),
                                                         (now / frac - now) if frac > 0 else float("inf"),
                                                         0.0))
            return self._kill

        def work():
            try:
                res = self.render(scene, camera_params, fs, sampler, integrator, tiles=tiles, film_out=film.pixels, progress=progress,
                                  **render_kw)
                if fs.accumulate and film.samples is not None:
                    np.add.at(film.samples, tiles["index"], 1)   # samples[tile.index] += 1, film.rs:270
                film.dirty = True
                with self._lock:
                    if rid == self._render_id:
                        self.last_result = res
                        self._messages.append(RenderFinished(int(res.stats.ray_count)))
            except Exception as e:  # noqa: BLE001 — whatever went wrong, the task posts its terminal message (the reference always
                # sends Finished, render_manager.rs:170-190); a poller of check_status must not spin forever
                cancelled = isinstance(e, capi.YukiGpuError) and e.code == capi.ERR_CANCELLED
                with self._lock:
                    if rid == self._render_id:
                        if not cancelled:
                            self.last_error = e
                        self._messages.append(RenderFinished(0))

        self._thread = threading.Thread(target=work, daemon=True)
        self._thread.start()

    def render_progressive(self, scene: Scene, camera_params: D.CameraParameters, film: Film, sampler: D.SamplerType,
                           integrator: D.IntegratorType, samples_per_pass: int = 16, checkpoint_path: Optional[str] = None,
                           max_passes: Optional[int] = None, render_fn=None, **render_kw):
        """Accumulating render that can stop and continue (`render_manager.rs:135-143` renders one tile list per sample index
        into a summing film; this drives it in passes of `samples_per_pass` indices). Starts at the film's first missing
        sample index — 0 for a fresh film, k for one restored with `Film.load` — and, after every pass, updates
        `film.samples` and (optionally) rewrites the checkpoint. Returns the number of sample indices the film now holds.
        `render_fn(tiles, film_out)` defaults to this renderer's `render`; tests on CPU pass the oracle's."""
        fs = film.settings
        if not fs.accumulate or film.samples is None:
            raise ValueError("render_progressive needs an accumulating film (FilmSettings.accumulate)")
        spp = sampler.samples_per_pixel()
        done = int(film.samples.min()) if film.samples.size else spp
        if film.samples.size and int(film.samples.max()) != done:
            raise ValueError("film tiles hold different sample counts: not a checkpoint of complete passes")
        if done > spp:
            raise ValueError(f"film already holds {done} samples per pixel, the sampler has {spp}")
        import hashlib
        clamp = getattr(integrator, "indirect_clamp", None)
        cam_bytes = np.asarray(list(camera_params.position) + list(camera_params.target) + list(camera_params.up) +
                               [float(camera_params.fov_axis), float(camera_params.fov_deg)], np.float32).tobytes()
        scene_id = None
        if getattr(scene, "host", None) is not None:
            flat = scene.host.flat
            scene_id = hashlib.sha256(C.string_at(flat.nodes, min(flat.n_nodes, 4096) * 32) + C.string_at(flat.tri_vertices, min(flat.n_tris, 4096) * 36) +
                                      np.asarray([flat.n_nodes, flat.n_tris, flat.n_lights, flat.n_materials], np.int64).tobytes()).hexdigest()[:16]
        meta = {"spp": spp, "sampler": [sampler.kind, sampler.nx, sampler.ny, bool(sampler.jitter), int(sampler.seed)],
                "integrator": [integrator.kind, integrator.max_depth, None if clamp is None else float(clamp)],
                "camera": hashlib.sha256(cam_bytes).hexdigest()[:16], "scene": scene_id}
        if film.meta and film.meta != json_roundtrip(meta):
            raise ValueError(f"film was rendered with other settings: {film.meta}")
        film.meta = json_roundtrip(meta)
        base = film_tiles(fs)
        if render_fn is None:
            def render_fn(tiles, film_out):
                return self.render(scene, camera_params, fs, sampler, integrator, tiles=tiles, film_out=film_out, **render_kw)
        passes = 0
        while done < spp and (max_passes is None or passes < max_passes):
            hi = min(spp, done + max(1, int(samples_per_pass)))
            tiles = np.concatenate([base] * (hi - done))
            tiles["sample"] = np.repeat(np.arange(done, hi, dtype=np.uint16), len(base))
            render_fn(tiles, film.pixels)
            np.add.at(film.samples, tiles["index"], 1)   # samples[tile.index] += 1, film.rs:270
            film.dirty = True
            done = hi
            passes += 1
            if checkpoint_path:
                film.save(checkpoint_path, meta=film.meta)
        return done

    def check_status(self):
        """Latest `RenderProgress`, or `RenderFinished` once the task is done; None when nothing new (renderer/mod.rs:61-120)."""
        ret = None
        if self._in_progress:
            with self._lock:
                msgs, self._messages = self._messages, []
            for m in msgs:
                ret = m
                if isinstance(m, RenderFinished):
                    self._in_progress = False
                    break
        return ret

    def kill(self):
        """Stops the running task (polled between wavefront batches) and joins the worker (renderer/mod.rs:122-128)."""
        if self._thread is not None:
            self._kill = True
            self._thread.join()
            self._thread = None
        with self._lock:
            self._messages = []
        self._in_progress = False

    def debug_ray(self, scene: Scene, camera_params: D.CameraParameters, film: D.FilmSettings, sampler: D.SamplerType,
                  integrator: D.IntegratorType, film_px, max_rays: int = 4096):
        """`launch_debug_ray` (app/window.rs:812-905): the rays `Integrator::li_debug` collects for one path through film pixel
        `film_px`, as a DEBUG_RAY_DTYPE array in the reference's order, plus li_debug's (li, ray_scene_intersections). None
        when the pixel lies outside the film (window.rs:866-869, 898-901)."""
        x, y = int(film_px[0]), int(film_px[1])
        if x < 0 or y < 0 or x >= int(film.res[0]) or y >= int(film.res[1]):
            return None
        cam = make_camera(camera_params, film)
        sm, ig = capi.sampler(sampler), capi.integrator(integrator)
        rays = np.zeros(max_rays, dtype=capi.DEBUG_RAY_DTYPE)
        n = C.c_uint32(0)
        li = np.zeros(3, np.float32)
        count = C.c_uint64(0)
        capi.check(capi.lib().yk_debug_ray(self.ctx._h, scene._h, C.byref(cam), C.byref(sm), C.byref(ig), x, y,
                                           C.c_void_p(rays.ctypes.data), max_rays, C.byref(n), capi.fptr(li), C.byref(count)))
        if n.value > max_rays:
            return self.debug_ray(scene, camera_params, film, sampler, integrator, film_px, max_rays=n.value)
        return rays[:n.value].copy(), li, int(count.value)

    def render(self, scene: Scene, camera_params: D.CameraParameters, film: D.FilmSettings, sampler: D.SamplerType,
               integrator: D.IntegratorType, tiles: Optional[np.ndarray] = None, want_hit_ids: bool = False,
               aux_sample: int = 0, wavefront_paths: int = 0, film_out: Optional[np.ndarray] = None,
               device_film_ptr: Optional[int] = None, progress=None, pipes: int = 0, ray_sort: int = 0) -> RenderResult:
        cam = make_camera(camera_params, film)
        if tiles is None:
            tiles = film_tiles(film)
        tiles = np.ascontiguousarray(tiles, dtype=capi.TILE_DTYPE)
        res_x, res_y = int(film.res[0]), int(film.res[1])
        opts = capi.RenderOpts()
        opts.wavefront_paths = wavefront_paths
        opts.aux_sample = aux_sample
        opts.pipes = pipes
        opts.ray_sort = ray_sort   # 0 default, 1 off, 2 leaf-slot key, 3 Morton key (yk_render_opts.ray_sort)
        hit_ids = None
        if device_film_ptr is not None:
            opts.flags |= capi.RENDER_FILM_ON_DEVICE
            film_arr, film_ptr = None, C.c_void_p(device_film_ptr)
        else:
            film_arr = film_out if film_out is not None else np.zeros((res_y, res_x, 3), dtype=np.float32)
            assert film_arr.dtype == np.float32 and film_arr.flags["C_CONTIGUOUS"] and film_arr.size == res_x * res_y * 3
            film_ptr = C.c_void_p(film_arr.ctypes.data)
            if want_hit_ids:
                hit_ids = np.full((res_y, res_x), -1, dtype=np.int32)
                opts.hit_ids = hit_ids.ctypes.data
        cb = None
        if progress is not None:
            cb = capi.PROGRESS_FN(lambda user, done, total: int(bool(progress(done, total))))
            opts.progress = cb
        fs, sm, ig = capi.film_settings(film), capi.sampler(sampler), capi.integrator(integrator)
        stats = capi.Stats()
        capi.check(capi.lib().yk_render(self.ctx._h, scene._h, C.byref(cam), C.byref(fs), C.byref(sm), C.byref(ig),
                                        C.c_void_p(tiles.ctypes.data), len(tiles), C.byref(opts), film_ptr, C.byref(stats)))
        return RenderResult(film_arr, hit_ids, stats)
