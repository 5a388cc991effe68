"""yk_query_intersect / yk_query_occluded: Scene::intersect's Hit { t, si, shape } (scene/mod.rs, bvh.rs:160-232) for caller
ray batches, on host arrays and on device-resident (torch CUDA) arrays. The oracle's yko_intersect_surface is first pinned
to the oracle's own debug integrators (GeometryNormals / ShadingNormals / UVs films, already pinned to the GPU); the GPU's
surface fields are then compared with it bit for bit, and the device path with the host path."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from yuki_b200 import api, capi, desc as D, scenes
from test_ray_queries import _grid_scene, _random_rays
from test_sphere import sphere_field

FIELDS = api.HIT_FIELDS
SURFACE = ("p", "n", "uv", "shading_n", "shading_dpdu")
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="session")
def osurf(oracle, tmp_path_factory):
    """OracleScene with `surface(o, d, t_max)`: yko_intersect_surface of tests/oracle_surface.cpp, compiled here with
    oracle/Makefile's flags into a library that carries the oracle's own entry points (its scenes are the oracle's)."""
    lib_path = tmp_path_factory.mktemp("oracle_surface") / "liboracle_surface.so"
    subprocess.check_call([os.environ.get("CXX", "g++"), "-O3", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-Wall",
                           "-Wextra", "-pthread", "-shared", "-Wl,-Bsymbolic", "-I", os.path.join(os.path.dirname(HERE), "oracle"),
                           "-o", str(lib_path), os.path.join(HERE, "oracle_surface.cpp")])
    L = C.CDLL(str(lib_path))
    vp, u32, fp = C.c_void_p, C.c_uint32, C.POINTER(C.c_float)
    L.yko_scene_create.argtypes = [C.POINTER(capi.HostSceneDesc)]
    L.yko_scene_create.restype = vp
    L.yko_scene_destroy.argtypes = [vp]
    L.yko_scene_destroy.restype = None
    L.yko_intersect_surface.argtypes = [vp, fp, fp, fp, u32, fp, vp, vp, vp, fp, fp, fp, fp, fp]
    L.yko_intersect_surface.restype = None

    class SurfaceScene(oracle.OracleScene):
        def __init__(self, scene):
            super().__init__(scene)
            hd, keep = capi.build_host_scene_desc(scene)
            self._hs = L.yko_scene_create(C.byref(hd))
            del keep
            if not self._hs:
                raise RuntimeError("oracle: BVH build failed")

        def surface(self, o, d, t_max=None):
            """`Scene::intersect`'s Hit: dict of t, orig_id, material, area_light, p, n, uv, shading_n, shading_dpdu (the
            surface fields 0 and the indices -1 on a miss)."""
            o = np.ascontiguousarray(o, np.float32).reshape(-1, 3)
            d = np.ascontiguousarray(d, np.float32).reshape(-1, 3)
            n = o.shape[0]
            out = {"t": np.zeros(n, np.float32), "orig_id": np.zeros(n, np.int32), "material": np.zeros(n, np.int32),
                   "area_light": np.zeros(n, np.int32), "p": np.zeros((n, 3), np.float32), "n": np.zeros((n, 3), np.float32),
                   "uv": np.zeros((n, 2), np.float32), "shading_n": np.zeros((n, 3), np.float32),
                   "shading_dpdu": np.zeros((n, 3), np.float32)}
            tm = None if t_max is None else capi.fptr(np.ascontiguousarray(t_max, np.float32))
            L.yko_intersect_surface(self._hs, capi.fptr(o), capi.fptr(d), tm, n, capi.fptr(out["t"]), out["orig_id"].ctypes.data,
                                    out["material"].ctypes.data, out["area_light"].ctypes.data, capi.fptr(out["p"]),
                                    capi.fptr(out["n"]), capi.fptr(out["uv"]), capi.fptr(out["shading_n"]),
                                    capi.fptr(out["shading_dpdu"]))
            return out

        def close(self):
            if getattr(self, "_hs", None):
                L.yko_scene_destroy(self._hs)
                self._hs = None
            super().close()

    return SurfaceScene


def _debug_scenes(xf):
    return {"material_room": scenes.material_room(xf),
            "sphere_field": sphere_field(xf, 40),
            "cornell": scenes.cornell(xf, light="rect", tall_box="glass", textured_back_wall=True, sphere=True)}


@pytest.mark.parametrize("name", ["material_room", "sphere_field", "cornell"])
def test_oracle_surface_equals_the_debug_integrator_films(oracle, osurf, xf, name):
    """Every pixel's 1-spp uniform camera ray, rebuilt from the sampler's first get_2d (integrators/mod.rs:163-166):
    n / 2 + 0.5, shading_n / 2 + 0.5 and (u, v, 0) of the oracle's surface are the debug integrators' film values."""
    scene, cam = _debug_scenes(xf)[name]
    film = D.FilmSettings((64, 40), 16)
    smp = D.SamplerType.uniform(1, seed=3)
    osc = osurf(scene)
    w, h = film.res
    pf = np.zeros((h * w, 2), np.float32)
    for y in range(h):
        for x in range(w):
            u = oracle.sampler_draws(smp, x, y, 0, [2])
            pf[y * w + x] = (np.float32(x) + u[0], np.float32(y) + u[1])
    o, d = oracle.camera_rays(cam, film, pf)
    s = osc.surface(o, d)
    t, ids, _ = osc.trace(o, d)
    assert np.array_equal(s["orig_id"], ids) and np.array_equal(s["t"].view(np.uint32), t.view(np.uint32))
    hit = ids >= 0
    assert hit.sum() > 500
    half, two = np.float32(0.5), np.float32(2.0)
    zero = np.zeros((h * w, 1), np.float32)
    want = {D.INTEGRATOR_GEOMETRY_NORMALS: s["n"] / two + half, D.INTEGRATOR_SHADING_NORMALS: s["shading_n"] / two + half,
            D.INTEGRATOR_SHADING_UVS: np.concatenate([s["uv"], zero], axis=1)}
    for kind, rgb in want.items():
        img, _, _ = osc.render(cam, film, smp, D.IntegratorType.debug(kind))
        img = img.reshape(-1, 3)
        assert np.array_equal(img[hit].view(np.uint32), rgb[hit].astype(np.float32).view(np.uint32)), kind
        assert not img[~hit].any()
    # misses carry the documented fill values
    for k in SURFACE:
        assert not s[k][~hit].any()
    assert (s["material"][~hit] == -1).all() and (s["area_light"][~hit] == -1).all()
    assert (s["material"][hit] >= 0).all() and (s["material"] < len(scene.materials)).all()
    assert ((s["area_light"] >= -1) & (s["area_light"] < len(scene.lights))).all()


def test_query_symbols_reject_null_arguments():
    L = capi.lib()
    assert L.yk_query_intersect(None, None, None, None, None, 4, None, None) == -1
    assert b"null argument" in L.yk_last_error()
    assert L.yk_query_occluded(None, None, None, None, 4, None, None) == -1
    assert b"null argument" in L.yk_last_error()


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _host(x):
    """torch tensor or numpy array -> numpy (uint32 tensors through an int32 view)."""
    if isinstance(x, np.ndarray):
        return x
    import torch
    if x.dtype == torch.uint32:
        return x.view(torch.int32).cpu().numpy().view(np.uint32)
    return x.cpu().numpy()


def _bits_equal(a, b):
    """Bit equality; NaNs by NaN-ness only (their payloads differ between x86 and the GPU, see test_ray_queries._same)."""
    a, b = _host(a), _host(b)
    assert a.shape == b.shape and a.dtype == b.dtype
    if a.dtype != np.float32:
        return np.array_equal(a, b)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(np.where(na, 0, a.view(np.uint32)), np.where(nb, 0, b.view(np.uint32)))


def _same_hits(got, want, tag=""):
    for k in FIELDS:
        g = getattr(got, k)
        w = want[k] if isinstance(want, dict) else getattr(want, k)
        assert _bits_equal(g, w), f"{tag} {k}"


def _check(dev, osc, o, d, t_max=None):
    """Host path vs the oracle, device path vs the host path; the old t / id / counts path too."""
    import torch
    got = dev.surface(o, d, t_max)
    want = osc.surface(o, d, t_max)
    _same_hits(got, want, "host")
    cu = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()
    got_dev = dev.surface(cu(o), cu(d), cu(t_max))
    assert got_dev.p.is_cuda and got_dev.p.shape == (len(o), 3)
    _same_hits(got_dev, got, "device")
    t, ids, cnt = dev.intersect(cu(o), cu(d), cu(t_max))
    ht, hids, hcnt = dev.intersect(o, d, t_max)
    assert _bits_equal(t, ht) and _bits_equal(ids, hids) and _bits_equal(cnt, hcnt)
    assert _bits_equal(dev.occluded(cu(o), cu(d)), dev.occluded(o, d))
    return got


def _degenerate_uv_scene(xf):
    """Quads whose uvs give uv_det == 0 (all equal, collinear), one with vertex normals, and a reference quad."""
    s = D.SceneDesc()
    zero = s.add_texture(D.Texture.constant(0.0))
    m = s.add_material(D.Material(D.MAT_MATTE, (s.add_texture(D.Texture.constant(0.5)), zero)))
    m2 = s.add_material(D.Material(D.MAT_METAL, (s.add_texture(D.Texture.constant(0.2)), s.add_texture(D.Texture.constant(3.0)),
                                                 s.add_texture(D.Texture.constant(0.1)))))
    quad = lambda x0: np.array([(x0, 0, 0), (x0 + 1, 0, 0.1), (x0 + 1, 1, 0.2), (x0, 1, 0)], np.float32)
    idx = np.array([0, 1, 2, 0, 2, 3], np.uint32)
    nrm = np.array([(0.1, 0.0, 1.0), (0.0, 0.2, 1.0), (-0.1, 0.1, 1.0), (0.0, -0.1, 1.0)], np.float32)
    s.meshes.append(D.Mesh(xf.identity(), quad(0.0), idx, m, uvs=np.full((4, 2), 0.5, np.float32)))
    s.meshes.append(D.Mesh(xf.identity(), quad(1.5), idx, m2, uvs=np.array([(0, 0), (1, 1), (2, 2), (3, 3)], np.float32), normals=nrm))
    s.meshes.append(D.Mesh(xf.identity(), quad(3.0), idx, m, uvs=np.array([(0, 0), (1, 0), (1, 1), (0, 1)], np.float32), normals=nrm))
    s.lights.append(D.Light(D.LIGHT_POINT, xf.translation((2.0, 0.5, 3.0)), (5.0, 5.0, 5.0)))
    return s, ((-0.5, -0.5, 1.0), (4.5, 1.5, 2.0), (-0.5, -0.5, -1.0), (4.5, 1.5, 0.3))


def _mirrored_scene(xf):
    """A heightfield with normals and uvs under a transform that swaps handedness (YK_TRI_SWAPS_HANDEDNESS)."""
    pts, idx = scenes.grid_mesh(24, 20, seed=6)
    s = D.SceneDesc(max_shapes_in_node=4)
    zero = s.add_texture(D.Texture.constant(0.0))
    m = s.add_material(D.Material(D.MAT_MATTE, (s.add_texture(D.Texture.from_image(scenes.checker_texture(64, 8))), zero)))
    nrm = np.tile(np.array([[0.0, 1.0, 0.0]], np.float32), (len(pts), 1)) + np.float32(0.2) * np.sin(pts).astype(np.float32)
    uvs = (pts[:, [0, 2]] * np.float32(0.5) + np.float32(0.5)).astype(np.float32)
    s.meshes.append(D.Mesh(xf.mul(xf.rotation(0.4, (0.0, 1.0, 0.3)), xf.scale(-1.0, 1.0, 1.0)), pts, idx, m, normals=nrm, uvs=uvs))
    s.lights.append(D.Light(D.LIGHT_POINT, xf.translation((0.0, 3.0, 0.0)), (5.0, 5.0, 5.0)))
    return s


def _rays_between(rng, n, src, dst):
    o = rng.uniform(src[0], src[1], (n, 3)).astype(np.float32)
    tgt = rng.uniform(dst[0], dst[1], (n, 3)).astype(np.float32)
    return o, (tgt - o).astype(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("split,leaf", [(D.SPLIT_SAH, 1), (D.SPLIT_MIDDLE, 4), (D.SPLIT_EQUAL_COUNTS, 7)])
def test_surface_on_a_heightfield(gpu_ctx, osurf, xf, split, leaf):
    scene, _ = scenes.heightfield(xf, 48, 48, seed=9, split_method=split, max_shapes_in_node=leaf)
    dev, osc = api.Scene(gpu_ctx, scene), osurf(scene)
    rng = np.random.default_rng(20 + split)
    o, d = _random_rays(rng, 40000, (-0.7, -0.4, -0.7), (0.7, 0.6, 0.7))
    got = _check(dev, osc, o, d)
    assert (got.orig_id >= 0).sum() > 5000 and (got.orig_id < 0).sum() > 500
    _check(dev, osc, o, d, rng.uniform(0.0, 1.5, len(o)).astype(np.float32))   # bounded: some hits now lie beyond t_max
    dev.close()


@pytest.mark.gpu
def test_surface_in_the_material_room(gpu_ctx, oracle, osurf, xf):
    """Vertex normals, uvs and an image texture; rect / spot / point lights."""
    scene, cam = scenes.material_room(xf)
    dev, osc = api.Scene(gpu_ctx, scene), osurf(scene)
    rng = np.random.default_rng(4)
    o, d = _rays_between(rng, 30000, ((-1.1, 0.05, -1.1), (1.1, 1.2, 1.1)), ((-1.3, -0.1, -1.3), (1.3, 1.3, 1.3)))
    film = D.FilmSettings((160, 100), 16)
    co, cd = oracle.camera_rays(cam, film, rng.uniform((0, 0), film.res, (20000, 2)).astype(np.float32))
    got = _check(dev, osc, np.concatenate([o, co]), np.concatenate([d, cd]))
    assert len(np.unique(got.material)) >= 4 and (got.area_light >= 0).any()
    dev.close()


@pytest.mark.gpu
def test_surface_with_degenerate_uvs_and_a_mirroring_transform(gpu_ctx, osurf, xf):
    scene, (lo, hi, lo2, hi2) = _degenerate_uv_scene(xf)
    dev, osc = api.Scene(gpu_ctx, scene), osurf(scene)
    rng = np.random.default_rng(7)
    o, d = _rays_between(rng, 20000, (lo, hi), (lo2, hi2))
    got = _check(dev, osc, o, d)
    assert (got.orig_id >= 0).sum() > 5000 and len(np.unique(got.material[got.orig_id >= 0])) == 2
    dev.close()
    scene = _mirrored_scene(xf)
    dev, osc = api.Scene(gpu_ctx, scene), osurf(scene)
    o, d = _random_rays(rng, 30000, (-1.2, -0.5, -1.2), (1.2, 0.8, 1.2))
    got = _check(dev, osc, o, d)
    assert (got.orig_id >= 0).sum() > 5000
    dev.close()


@pytest.mark.gpu
def test_surface_on_spheres_and_leaf_tables(gpu_ctx, osurf, xf):
    """Scaled, rotated and mirrored spheres; leaves of more than 16 shapes (the leaf table), with and without spheres."""
    cases = [(sphere_field(xf, 60)[0], (-2.0, 0.0, -2.0), (2.0, 1.5, 2.0)),
             (scenes.cornell(xf, light="rect", tall_box="glass", sphere=True, max_shapes_in_node=40)[0], (0.0, 0.0, -0.56), (0.555, 0.55, 0.0)),
             (scenes.heightfield(xf, 24, 24, seed=4, max_shapes_in_node=40)[0], (-0.6, -0.4, -0.6), (0.6, 0.6, 0.6))]
    for scene, lo, hi in cases:
        dev, osc = api.Scene(gpu_ctx, scene), osurf(scene)
        rng = np.random.default_rng(5)
        o, d = _random_rays(rng, 30000, lo, hi)
        got = _check(dev, osc, o, d)
        assert (got.orig_id >= 0).sum() > 3000
        if scene.spheres and scene.lights[0].kind == D.LIGHT_RECT:   # the Cornell box's light quad
            assert (got.area_light >= 0).any()
        dev.close()


@pytest.mark.gpu
def test_surface_of_corner_case_rays(gpu_ctx, osurf, xf):
    """test_ray_queries' corner cases: vertices, shared edges, negative zeros, t_max at and one ulp short of the hit, rays in
    a triangle's plane, tiny and huge directions, far origins, a zero direction."""
    n = 6
    scene = _grid_scene(xf, n)
    dev, osc = api.Scene(gpu_ctx, scene), osurf(scene)
    o, d, tm = [], [], []
    for i in range(n + 1):
        for j in range(n + 1):
            for oo, dd, t in (((i, 1.0, j), (0.0, -1.0, 0.0), np.inf), ((i, 1.0, j), (-0.0, -1.0, 0.0), np.inf),
                              ((i + 0.5, 2.0, j), (0.0, -1.0, 0.0), np.inf), ((i, 1.0, j), (0.0, -1.0, 0.0), 1.0),
                              ((i, 1.0, j), (0.0, -1.0, 0.0), np.float32(1.0) - np.float32(2.0 ** -24)),
                              ((i, -1.0, j), (0.0, 1.0, 0.0), np.inf), ((i, 0.0, j), (1.0, 0.0, 0.0), np.inf),
                              ((i + 0.25, 0.0, j + 0.25), (0.0, 0.0, 1.0), np.inf), ((i, 0.5, j), (1.0, 0.0, 0.0), np.inf),
                              ((i, 0.5, j), (1.0, 0.0, 0.0), 0.0), ((i, 0.5, j), (1e-30, 0.0, 0.0), np.inf),
                              ((i, 0.5, j), (1e30, 0.0, 0.0), np.inf), ((i, 0.5, j), (-1.0, 0.0, 0.0), np.inf),
                              ((i, 1.0, j), (1.0, -1.0, 1.0), np.inf), ((i, 1.0, j), (1.0, -1.0, 0.0), np.inf),
                              ((i - 1e30, 1.0, j), (1.0, 0.0, 0.0), np.inf)):
                o.append(oo); d.append(dd); tm.append(t)
    for oo, dd in (((3.0, 1.0, 3.0), (0.0, 0.0, 0.0)), ((n, 1.0, 3.0), (0.0, 0.0, 1.0)), ((n, 1.0, 3.0), (1.0, 0.0, 0.0)),
                   ((n, 1.0, 3.0), (-1.0, 0.0, 0.0))):
        o.append(oo); d.append(dd); tm.append(np.inf)
    o, d, tm = np.array(o, np.float32), np.array(d, np.float32), np.array(tm, np.float32)
    got = _check(dev, osc, o, d, tm)
    assert (got.orig_id >= 0).sum() > 100
    _check(dev, osc, o, d)
    dev.close()


@pytest.mark.gpu
def test_device_path_equals_host_path_over_two_chunks(gpu_ctx, xf):
    """4 Mi + 4099 rays: two chunks of the query loop with a ragged tail. Every output of the device path, counters included,
    equals the host path's; yk_query_occluded on the device equals yk_occluded."""
    import torch
    scene, _ = scenes.heightfield(xf, 64, 64, seed=2)
    dev = api.Scene(gpu_ctx, scene)
    rng = np.random.default_rng(12)
    n = (1 << 22) + 4099
    o, d = _random_rays(rng, n, (-0.7, -0.4, -0.7), (0.7, 0.6, 0.7))
    tm = rng.uniform(0.2, 2.0, n).astype(np.float32)
    to, td, ttm = (torch.from_numpy(a).cuda() for a in (o, d, tm))
    for args, targs in (((o, d, tm), (to, td, ttm)), ((o, d), (to, td))):
        t, ids, cnt = dev.intersect(*args)
        gt, gids, gcnt = dev.intersect(*targs)
        assert _bits_equal(gt, t) and _bits_equal(gids, ids) and _bits_equal(gcnt, cnt)
        _same_hits(dev.surface(*targs), dev.surface(*args), "two chunks")
    gt, gids, gcnt = dev.intersect(to, td, counts=False)
    assert _bits_equal(gt, t) and _bits_equal(gids, ids) and not _host(gcnt).any()
    occ = dev.occluded(o, d)
    assert 0 < occ.sum() < n
    assert _bits_equal(dev.occluded(to, td), occ)
    dev.close()


@pytest.mark.gpu
def test_device_query_orders_after_the_callers_stream(gpu_ctx, xf):
    """The rays are written on a side stream behind a long matrix product queued there; the query is given that stream and
    must see the written rays, not the zeros they replace."""
    import torch
    scene, _ = scenes.heightfield(xf, 48, 48, seed=2)
    dev = api.Scene(gpu_ctx, scene)
    rng = np.random.default_rng(13)
    n = 1 << 20
    o, d = _random_rays(rng, n, (-0.7, -0.4, -0.7), (0.7, 0.6, 0.7))
    want = dev.surface(o, d)
    src_o, src_d = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    a = torch.randn(8192, 8192, device="cuda")
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        to = torch.zeros_like(src_o)
        td = torch.zeros_like(src_d)
        for _ in range(4):
            a = a @ a / 8192.0                 # ~4 TFLOP of float32 queued ahead of the copies
        to.copy_(src_o)
        td.copy_(src_d)
        got = dev.surface(to, td)
        t, ids, _ = dev.intersect(to, td)
        occ = dev.occluded(to, td)
    _same_hits(got, want, "stream")
    assert _bits_equal(t, want.t) and _bits_equal(ids, want.orig_id)
    assert _bits_equal(occ, dev.occluded(o, d))
    torch.cuda.synchronize()
    dev.close()


def _raw_intersect(dev, o, d, tm, n, hits, flags=capi.QUERY_ON_DEVICE, reserved=0, stream=None):
    opts = capi.QueryOpts(flags, reserved, stream)
    return capi.lib().yk_query_intersect(dev.ctx._h, dev._h, o, d, tm, n, C.byref(opts), C.byref(hits))


@pytest.mark.gpu
def test_refusals_leave_the_context_usable(gpu_ctx, osurf, xf):
    import torch
    scene, cam = scenes.heightfield(xf, 32, 32, seed=3)
    dev, osc = api.Scene(gpu_ctx, scene), osurf(scene)
    rng = np.random.default_rng(14)
    n = 5000
    o, d = _random_rays(rng, n, (-0.7, -0.4, -0.7), (0.7, 0.6, 0.7))
    tm = np.full(n, 3.0, np.float32)
    to, td, ttm = (torch.from_numpy(a).cuda() for a in (o, d, tm))
    t_out = torch.empty(n, dtype=torch.float32, device="cuda")
    film = D.FilmSettings((48, 32), 16)
    want_img, _, _ = osc.render(cam, film, D.SamplerType.uniform(1), D.IntegratorType.bvh_intersections())
    L = capi.lib()

    def refused(rc, text):
        assert rc == -1, rc
        assert text in L.yk_last_error().decode(), L.yk_last_error()
        # the context still answers queries and renders correctly
        got = dev.surface(to[:2000], td[:2000])
        _same_hits(got, osc.surface(o[:2000], d[:2000]), "after refusal")
        r = api.Renderer(gpu_ctx).render(dev, cam, film, D.SamplerType.uniform(1), D.IntegratorType.bvh_intersections())
        assert np.array_equal(r.film.view(np.uint32), want_img.view(np.uint32))

    dev_hits = capi.Hits(t=t_out.data_ptr())
    # host (numpy) memory under YK_QUERY_ON_DEVICE
    refused(_raw_intersect(dev, o.ctypes.data, d.ctypes.data, None, n, dev_hits), "not device memory")
    refused(_raw_intersect(dev, to.data_ptr(), td.data_ptr(), None, n, capi.Hits(t=np.zeros(n, np.float32).ctypes.data)), "not device memory")
    pinned = to.cpu().pin_memory()
    refused(_raw_intersect(dev, pinned.data_ptr(), td.data_ptr(), None, n, dev_hits), "not device memory")
    occ_np = np.zeros(n, np.uint8)
    refused(L.yk_query_occluded(dev.ctx._h, dev._h, to.data_ptr(), td.data_ptr(), n, C.byref(capi.QueryOpts(capi.QUERY_ON_DEVICE, 0, None)),
                                occ_np.ctypes.data), "not device memory")
    # a pointer one byte off
    refused(_raw_intersect(dev, to.data_ptr() + 1, td.data_ptr(), None, n - 1, dev_hits), "not 4-byte aligned")
    # a NaN t_max in device memory: found by the kernel, reported at the end of the call
    bad = ttm.clone()
    bad[n // 2] = float("nan")
    refused(_raw_intersect(dev, to.data_ptr(), td.data_ptr(), bad.data_ptr(), n, dev_hits), "NaN t_max")
    with pytest.raises(capi.YukiGpuError):
        dev.surface(to, td, bad)
    # unknown flags, non-zero _reserved
    refused(_raw_intersect(dev, to.data_ptr(), td.data_ptr(), None, n, dev_hits, flags=capi.QUERY_ON_DEVICE | 2), "unknown flag")
    refused(_raw_intersect(dev, to.data_ptr(), td.data_ptr(), None, n, dev_hits, reserved=1), "_reserved")
    refused(L.yk_query_occluded(dev.ctx._h, dev._h, to.data_ptr(), td.data_ptr(), n, C.byref(capi.QueryOpts(0, 7, None)),
                                occ_np.ctypes.data), "_reserved")
    # the Python surface refuses mixed, mistyped and misplaced input before the library sees it
    with pytest.raises(TypeError):
        dev.surface(to, d)
    with pytest.raises(TypeError):
        dev.intersect(to.double(), td.double())
    with pytest.raises(TypeError):
        dev.occluded(to, td.cpu())
    # a valid device call after all of that, with a t_max
    _same_hits(dev.surface(to, td, ttm), osc.surface(o, d, tm), "final")
    dev.close()


@pytest.mark.gpu
def test_tensor_on_another_gpu_is_refused(gpu_ctx, osurf, xf):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    scene, _ = scenes.heightfield(xf, 32, 32, seed=3)
    dev, osc = api.Scene(gpu_ctx, scene), osurf(scene)
    rng = np.random.default_rng(15)
    o, d = _random_rays(rng, 3000, (-0.7, -0.4, -0.7), (0.7, 0.6, 0.7))
    o1, d1 = torch.from_numpy(o).to("cuda:1"), torch.from_numpy(d).to("cuda:1")
    with pytest.raises(ValueError):
        dev.surface(o1, d1)
    t0 = torch.empty(len(o), dtype=torch.float32, device="cuda:0")
    assert _raw_intersect(dev, o1.data_ptr(), d1.data_ptr(), None, len(o), capi.Hits(t=t0.data_ptr())) == -1
    assert "not device memory of the context's GPU" in capi.lib().yk_last_error().decode()
    o0, d0 = o1.to("cuda:0"), d1.to("cuda:0")
    _same_hits(dev.surface(o0, d0), osc.surface(o, d), "after refusal")
    dev.close()
