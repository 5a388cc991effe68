"""Companion films of one Path / Whitted render (`yk_render_opts.aovs`, `Renderer.render(aovs=...)`).

The four views are the debug integrators' films (bvh_heatmap.rs, geometry_normals.rs, shading_normals.rs, shading_uvs.rs)
from the camera rays the render traces anyway, and `radiance_sq` is each pixel's float32 sum of li*li over its samples in
the film's order, divided by spp. Every GPU test compares bits: a view must equal the film `yk_render` returns with the
corresponding debug integrator (itself equal to the oracle's), and the main film, hit ids and ray / traversal counters must
equal those of the same render without companion films.
"""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from test_render_limits import COUNTERS
from test_shadow_modes import _plus_point_light
from test_sphere import sphere_field
from yuki_b200 import api, capi, desc as D, headless, scenes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VIEWS = {"bvh_intersections": D.INTEGRATOR_BVH_INTERSECTIONS, "geometry_normals": D.INTEGRATOR_GEOMETRY_NORMALS,
         "shading_normals": D.INTEGRATOR_SHADING_NORMALS, "shading_uvs": D.INTEGRATOR_SHADING_UVS}
ALL = capi.AOV_NAMES
S2, U3 = D.SamplerType.stratified(2, 2), D.SamplerType.uniform(3)
P8, W5 = D.IntegratorType.path(8), D.IntegratorType.whitted(5)


def _debug_integrator(name):
    k = VIEWS[name]
    return D.IntegratorType.bvh_intersections() if k == D.INTEGRATOR_BVH_INTERSECTIONS else D.IntegratorType.debug(k)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _scenes(xf):
    return {
        "glass-cornell-rect": lambda: scenes.cornell(xf, light="rect", tall_box="glass"),
        "material-room": lambda: scenes.material_room(xf),
        "sphere-field": lambda: sphere_field(xf, 24),
        "open-scene": lambda: scenes.open_scene(xf),
        "leaves-40": lambda: _plus_point_light(scenes.heightfield(xf, 40, 40, seed=5, split_method=D.SPLIT_EQUAL_COUNTS, max_shapes_in_node=40),
                                               (-3.0, 4.0, 2.0), (300.0, 250.0, 200.0)),
    }


SCENE_IDS = ("glass-cornell-rect", "material-room", "sphere-field", "open-scene", "leaves-40")
FILM = D.FilmSettings((40, 24), 8)


def _render(ctx, dev, cam, film, smp, integ, **kw):
    return api.Renderer(ctx).render(dev, cam, film, smp, integ, **kw)


def _assert_same_render(r, ref, what=""):
    """Main film, hit ids and every ray / traversal counter of `r` equal those of `ref`."""
    assert np.array_equal(_bits(r.film), _bits(ref.film)), what
    if ref.hit_ids is not None:
        assert np.array_equal(r.hit_ids, ref.hit_ids), what
    for k in COUNTERS + ("samples", "primary_hit_hash"):
        assert getattr(r.stats, k) == getattr(ref.stats, k), (what, k)


# ---- CPU: ABI layout, name validation, --aov parsing --------------------------------------------------------------
LAYOUT_C = r"""
#include <stddef.h>
#include <stdio.h>
#include "yuki_gpu.h"
int main(void) {
    printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(yk_render_opts), offsetof(yk_render_opts, ray_sort),
           offsetof(yk_render_opts, _reserved), offsetof(yk_render_opts, aovs), sizeof(yk_aov_films),
           offsetof(yk_aov_films, bvh_intersections), offsetof(yk_aov_films, geometry_normals),
           offsetof(yk_aov_films, shading_normals), offsetof(yk_aov_films, shading_uvs), offsetof(yk_aov_films, radiance_sq));
    printf("%u\n", (unsigned)YK_RENDER_AOVS);
    return 0;
}
"""


def test_ctypes_layout_matches_the_header(tmp_path):
    if not shutil.which("gcc"):
        pytest.skip("no gcc")
    src = tmp_path / "layout.c"
    src.write_text(LAYOUT_C)
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    lines = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n")
    got = [int(v) for v in lines[0].split()]
    A, R = capi.AovFilms, capi.RenderOpts
    assert got == [C.sizeof(R), R.ray_sort.offset, R._reserved.offset, R.aovs.offset, C.sizeof(A), A.bvh_intersections.offset,
                   A.geometry_normals.offset, A.shading_normals.offset, A.shading_uvs.offset, A.radiance_sq.offset]
    assert int(lines[1]) == capi.RENDER_AOVS
    # appended: every field an old caller sets keeps its offset
    assert R.aovs.offset == R._reserved.offset + 4


def test_aov_names_are_validated_before_the_gpu():
    assert api.aov_names(["radiance_sq", "bvh_intersections", "radiance_sq"]) == ("bvh_intersections", "radiance_sq")
    assert api.aov_names(None, {"shading_uvs": None}) == ("shading_uvs",)
    assert api.aov_names() == ()
    for bad in (["albedo"], ["depth", "shading_uvs"]):
        with pytest.raises(ValueError, match="unknown companion film"):
            api.aov_names(bad)
    rn = api.Renderer(None)   # no context: a bad name must fail before anything touches the library
    with pytest.raises(ValueError):
        rn.render(None, None, FILM, S2, P8, aovs=["normals"])
    with pytest.raises(ValueError):
        rn.render(None, None, FILM, S2, P8, aov_out={"position": np.zeros((24, 40, 3), np.float32)})
    with pytest.raises(ValueError):
        rn.launch(None, None, api.Film(FILM), S2, P8, aovs=["albedo"])
    with pytest.raises(ValueError):
        rn.render_progressive(None, None, api.Film(D.FilmSettings((8, 8), 8, accumulate=True)), S2, P8, aovs=["albedo"])


def test_headless_aov_arguments():
    a = headless.parse_args(["--out", "x.exr", "--aov", "shading_uvs=uv.exr", "--aov", "radiance_sq=/tmp/r sq.exr"])
    assert a.aov == [("shading_uvs", "uv.exr"), ("radiance_sq", "/tmp/r sq.exr")]
    assert headless.parse_args(["--out", "x.exr"]).aov == []
    for bad in ("albedo=a.exr", "shading_uvs", "shading_uvs="):
        with pytest.raises(SystemExit):
            headless.parse_args(["--out", "x.exr", "--aov", bad])


# ---- GPU -------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def scene_cache(gpu_ctx, xf):
    made = {}

    def get(name):
        if name not in made:
            scene, cam = _scenes(xf)[name]()
            made[name] = (scene, cam, api.Scene(gpu_ctx, scene))
        return made[name]
    yield get
    for _, _, dev in made.values():
        dev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("smp", [S2, U3], ids=["stratified-2x2", "uniform-3"])
@pytest.mark.parametrize("integ", [P8, W5], ids=["path-8", "whitted-5"])
@pytest.mark.parametrize("scene_id", SCENE_IDS)
def test_views_equal_the_debug_integrators(gpu_ctx, scene_cache, oracle, scene_id, integ, smp):
    scene, cam, dev = scene_cache(scene_id)
    plain = _render(gpu_ctx, dev, cam, FILM, smp, integ, want_hit_ids=True)
    r = _render(gpu_ctx, dev, cam, FILM, smp, integ, want_hit_ids=True, aovs=ALL)
    _assert_same_render(r, plain, scene_id)
    assert r.stats.trace_closest_launches == plain.stats.trace_closest_launches   # the BVH view swaps bounce 0's kernel, adds none
    assert set(r.aovs) == set(ALL)
    osc = oracle.OracleScene(scene)
    for name in VIEWS:
        dbg = _render(gpu_ctx, dev, cam, FILM, smp, _debug_integrator(name))
        o_img = osc.render(cam, FILM, smp, _debug_integrator(name))[0]
        assert np.array_equal(_bits(dbg.film), _bits(o_img)), (scene_id, name)
        assert r.aovs[name].shape == (24, 40, 3) and r.aovs[name].dtype == np.float32
        assert np.array_equal(_bits(r.aovs[name]), _bits(dbg.film)), (scene_id, name)
    assert float(r.aovs["bvh_intersections"].max()) > 0 and float(r.aovs["radiance_sq"].max()) > 0
    if scene_id == "open-scene":   # misses give 0: pixels whose every camera ray leaves the scene (hit_ids is sample 0's only)
        assert ((r.aovs["geometry_normals"] == 0).all(axis=2) & (plain.hit_ids < 0)).any()


def _per_sample_films(oracle, scene, cam, film, smp, integ):
    """li_k for every sample index k: the oracle's accumulating film over tiles of sample k, onto zeros."""
    acc = D.FilmSettings(tuple(film.res), film.tile_dim, accumulate=True)
    base = api.film_tiles(acc)
    osc = oracle.OracleScene(scene)
    out = []
    for k in range(smp.samples_per_pixel()):
        t = base.copy()
        t["sample"] = k
        out.append(osc.render(cam, acc, smp, integ, tiles=t, film_out=np.zeros((film.res[1], film.res[0], 3), np.float32), threads=1)[0])
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("smp", [S2, U3], ids=["stratified-2x2", "uniform-3"])
@pytest.mark.parametrize("integ", [P8, W5], ids=["path-8", "whitted-5"])
def test_radiance_sq_equals_a_float32_reference_from_the_oracle(gpu_ctx, scene_cache, oracle, integ, smp):
    scene, cam, dev = scene_cache("glass-cornell-rect")
    film = D.FilmSettings((24, 16), 8)
    lis = _per_sample_films(oracle, scene, cam, film, smp, integ)
    spp = np.float32(smp.samples_per_pixel())
    mean, sq = np.zeros_like(lis[0]), np.zeros_like(lis[0])
    for li in lis:   # ascending sample index, float32, as integrators/mod.rs:172 sums the film
        mean = mean + li
        sq = sq + li * li
    mean, sq = mean / spp, sq / spp
    o_img = oracle.OracleScene(scene).render(cam, film, smp, integ)[0]
    assert np.array_equal(_bits(mean), _bits(o_img))   # the method reproduces the mean film: li_k is exact
    r = _render(gpu_ctx, dev, cam, film, smp, integ, aovs=["radiance_sq"])
    assert np.array_equal(_bits(r.film), _bits(o_img))
    assert np.array_equal(_bits(r.aovs["radiance_sq"]), _bits(sq)) and float(sq.max()) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("integ", [P8, W5], ids=["path-8", "whitted-5"])
def test_accumulating_views_add_onto_existing_films(gpu_ctx, scene_cache, oracle, integ):
    """Four sample indices added onto a non-zero film and non-zero views, in tile-list order."""
    scene, cam, dev = scene_cache("material-room")
    film = D.FilmSettings((32, 16), 8)
    acc = D.FilmSettings((32, 16), 8, accumulate=True)
    base = api.film_tiles(acc)
    tiles = np.concatenate([base] * 4)
    tiles["sample"] = np.repeat(np.arange(4, dtype=np.uint16), len(base))
    rng = np.random.default_rng(7)
    start = {n: rng.random((16, 32, 3), dtype=np.float32) for n in ("film",) + ALL}
    out = {n: start[n].copy() for n in ALL}
    r = _render(gpu_ctx, dev, cam, acc, S2, integ, tiles=tiles, film_out=start["film"].copy(), aov_out=out)
    plain = _render(gpu_ctx, dev, cam, acc, S2, integ, tiles=tiles, film_out=start["film"].copy())
    _assert_same_render(r, plain)
    osc = oracle.OracleScene(scene)
    for name in VIEWS:
        dbg = _render(gpu_ctx, dev, cam, acc, S2, _debug_integrator(name), tiles=tiles, film_out=start[name].copy())
        o_img = osc.render(cam, acc, S2, _debug_integrator(name), tiles=tiles, film_out=start[name].copy(), threads=1)[0]
        assert np.array_equal(_bits(dbg.film), _bits(o_img)), name
        assert r.aovs[name] is out[name] and np.array_equal(_bits(out[name]), _bits(dbg.film)), name
    lis = _per_sample_films(oracle, scene, cam, film, S2, integ)
    sq = start["radiance_sq"].copy()
    for li in lis:
        sq = sq + li * li
    assert np.array_equal(_bits(out["radiance_sq"]), _bits(sq))
    # every tile listed twice within its sample index: each pixel is added twice in one batch, as the main film is
    twice = np.concatenate([tiles[tiles["sample"] == k].repeat(2) for k in range(4)])
    out2 = {n: start[n].copy() for n in ALL}
    r2 = _render(gpu_ctx, dev, cam, acc, S2, integ, tiles=twice, film_out=start["film"].copy(), aov_out=out2)
    _assert_same_render(r2, _render(gpu_ctx, dev, cam, acc, S2, integ, tiles=twice, film_out=start["film"].copy()))
    for name in VIEWS:
        dbg = _render(gpu_ctx, dev, cam, acc, S2, _debug_integrator(name), tiles=twice, film_out=start[name].copy())
        assert np.array_equal(_bits(out2[name]), _bits(dbg.film)), name
    sq = start["radiance_sq"].copy()
    for li in lis:
        sq = (sq + li * li) + li * li
    assert np.array_equal(_bits(out2["radiance_sq"]), _bits(sq))


@pytest.mark.gpu
def test_views_do_not_depend_on_the_batch_shape(gpu_ctx, scene_cache, monkeypatch):
    """More than 1024 spp (a pixel's samples over several batches), small batches, two pipes and YK_MAX_BATCH_SAMPLES=7 all
    give the bits of the one-batch render; the views still equal the debug integrators."""
    scene, cam, dev = scene_cache("glass-cornell-rect")
    film = D.FilmSettings((8, 4), 8)
    smp = D.SamplerType.uniform(1100)
    ref = _render(gpu_ctx, dev, cam, film, smp, P8, want_hit_ids=True, aovs=ALL, pipes=1)
    for name in VIEWS:
        dbg = _render(gpu_ctx, dev, cam, film, smp, _debug_integrator(name))
        assert np.array_equal(_bits(ref.aovs[name]), _bits(dbg.film)), name
    # 200 paths per batch: 4 samples of the 32 pixels per batch, 275 batches
    r = _render(gpu_ctx, dev, cam, film, smp, P8, want_hit_ids=True, aovs=ALL, wavefront_paths=200)
    _assert_same_render(r, ref)
    for name in ALL:
        assert np.array_equal(_bits(r.aovs[name]), _bits(ref.aovs[name])), name
    # Two pipes: the 960 pixels of FILM at 4 spp in batches of 200 / 300 paths are 6 / 4 pixel groups of 160 / 240 pixels, one
    # sample each per batch (render.cu keeps both pipes when there are more groups than pipes), alternating between the streams,
    # which share the context's per-pixel view sums
    one = _render(gpu_ctx, dev, cam, FILM, S2, P8, want_hit_ids=True, aovs=ALL, pipes=1)
    for name in VIEWS:
        dbg = _render(gpu_ctx, dev, cam, FILM, S2, _debug_integrator(name))
        assert np.array_equal(_bits(one.aovs[name]), _bits(dbg.film)), name
    for cap in (200, 300):
        r = _render(gpu_ctx, dev, cam, FILM, S2, P8, want_hit_ids=True, aovs=ALL, pipes=2, wavefront_paths=cap)
        _assert_same_render(r, one, cap)
        for name in ALL:
            assert np.array_equal(_bits(r.aovs[name]), _bits(one.aovs[name])), (cap, name)
    monkeypatch.setenv("YK_MAX_BATCH_SAMPLES", "7")
    for smp_, film_ in ((smp, film), (S2, FILM)):
        r = _render(gpu_ctx, dev, cam, film_, smp_, W5, want_hit_ids=True, aovs=ALL)
        monkeypatch.delenv("YK_MAX_BATCH_SAMPLES")
        base = _render(gpu_ctx, dev, cam, film_, smp_, W5, want_hit_ids=True, aovs=ALL)
        monkeypatch.setenv("YK_MAX_BATCH_SAMPLES", "7")
        _assert_same_render(r, base)
        for name in ALL:
            assert np.array_equal(_bits(r.aovs[name]), _bits(base.aovs[name])), name


def _partial_tiles(film):
    t = api.film_tiles(film)
    return t[: len(t) // 2]


@pytest.mark.gpu
def test_partial_tiles_and_device_buffers(gpu_ctx, scene_cache):
    """Pixels outside `tiles` are left untouched in host and device buffers; device views equal the host path."""
    import torch
    scene, cam, dev = scene_cache("sphere-field")
    full = _render(gpu_ctx, dev, cam, FILM, S2, P8, aovs=ALL)
    tiles = _partial_tiles(FILM)
    inside = np.zeros((24, 40), bool)
    for t in tiles:
        inside[t["y0"]:t["y1"], t["x0"]:t["x1"]] = True
    assert inside.any() and not inside.all()
    sentinel = np.float32(-7.25)
    host = {n: np.full((24, 40, 3), sentinel, np.float32) for n in ALL}
    r = _render(gpu_ctx, dev, cam, FILM, S2, P8, tiles=tiles, film_out=np.full((24, 40, 3), sentinel, np.float32), aov_out=host)
    for n in ALL:
        assert (host[n][~inside] == sentinel).all(), n
        assert np.array_equal(_bits(host[n][inside]), _bits(full.aovs[n][inside])), n
    assert np.array_equal(_bits(r.film[inside]), _bits(full.film[inside]))
    # the same render into torch CUDA tensors
    film_t = torch.full((24, 40, 3), float(sentinel), dtype=torch.float32, device="cuda")
    views_t = {n: torch.full((24, 40, 3), float(sentinel), dtype=torch.float32, device="cuda") for n in ALL}
    torch.cuda.synchronize()
    rd = _render(gpu_ctx, dev, cam, FILM, S2, P8, tiles=tiles, device_film_ptr=film_t.data_ptr(),
                 aov_out={n: v.data_ptr() for n, v in views_t.items()})
    assert rd.aovs == {n: v.data_ptr() for n, v in views_t.items()}
    assert np.array_equal(_bits(film_t.cpu().numpy()), _bits(r.film))
    for n in ALL:
        assert np.array_equal(_bits(views_t[n].cpu().numpy()), _bits(host[n])), n
    # full cover on the device
    views_t = {n: torch.zeros((24, 40, 3), dtype=torch.float32, device="cuda") for n in ALL}
    film_t = torch.zeros((24, 40, 3), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    _render(gpu_ctx, dev, cam, FILM, S2, P8, device_film_ptr=film_t.data_ptr(), aov_out={n: v.data_ptr() for n, v in views_t.items()})
    for n in ALL:
        assert np.array_equal(_bits(views_t[n].cpu().numpy()), _bits(full.aovs[n])), n
    with pytest.raises(ValueError):   # device films need a pointer per requested view
        _render(gpu_ctx, dev, cam, FILM, S2, P8, device_film_ptr=film_t.data_ptr(), aovs=["shading_uvs"])


@pytest.mark.gpu
def test_views_under_shadow_modes_and_ray_sorts(gpu_ctx, xf):
    """Both forced YK_SHADOW_MODEs and ray sort 2 and 3 leave the views (and the render) unchanged."""
    scene, cam = _scenes(xf)["leaves-40"]()
    scene.lights.append(D.Light(D.LIGHT_POINT, xf.translation((2.0, 3.0, -1.0)), (100.0, 100.0, 100.0)))
    ctxs = {}
    try:
        with pytest.MonkeyPatch.context() as mp:
            for mode in ("0", "1"):
                mp.setenv("YK_SHADOW_MODE", mode)
                ctxs[mode] = api.Context(0)
        dev = api.Scene(gpu_ctx, scene)
        ref = _render(gpu_ctx, dev, cam, FILM, S2, P8, want_hit_ids=True, aovs=ALL, ray_sort=1)
        dev.close()
        runs = [(gpu_ctx, dict(ray_sort=2)), (gpu_ctx, dict(ray_sort=3)), (ctxs["0"], {}), (ctxs["1"], {}), (ctxs["1"], dict(ray_sort=3))]
        for ctx, kw in runs:
            d = api.Scene(ctx, scene)
            r = _render(ctx, d, cam, FILM, S2, P8, want_hit_ids=True, aovs=ALL, **kw)
            d.close()
            _assert_same_render(r, ref, kw)
            for name in ALL:
                assert np.array_equal(_bits(r.aovs[name]), _bits(ref.aovs[name])), (kw, name)
    finally:
        for c in ctxs.values():
            c.close()


@pytest.mark.gpu
def test_refusals_leave_the_context_usable(gpu_ctx, scene_cache):
    scene, cam, dev = scene_cache("glass-cornell-rect")
    film = D.FilmSettings((16, 8), 8)
    ref = _render(gpu_ctx, dev, cam, film, S2, P8, aovs=ALL)
    L = capi.lib()
    cam_c = api.make_camera(cam, film)
    fs, sm = capi.film_settings(film), capi.sampler(S2)
    tiles = api.film_tiles(film)
    img = np.zeros((8, 16, 3), np.float32)

    def call(integ, opts):
        ig = capi.integrator(integ)
        stats = capi.Stats()
        return L.yk_render(gpu_ctx._h, dev._h, C.byref(cam_c), C.byref(fs), C.byref(sm), C.byref(ig), C.c_void_p(tiles.ctypes.data),
                           len(tiles), C.byref(opts), C.c_void_p(img.ctypes.data), C.byref(stats))

    view = np.full((8, 16, 3), 3.0, np.float32)
    films = capi.AovFilms()
    films.shading_uvs = view.ctypes.data
    opts = capi.RenderOpts()
    opts.flags = capi.RENDER_AOVS   # aovs NULL
    assert call(P8, opts) == -1 and b"aovs" in L.yk_last_error()
    opts.aovs = C.pointer(films)
    for integ in [_debug_integrator(n) for n in VIEWS] + [D.IntegratorType.path(0)]:
        assert call(integ, opts) == -1, integ
        assert (view == 3.0).all() and not img.any()   # nothing launched, nothing written
    with pytest.raises(capi.YukiGpuError):
        _render(gpu_ctx, dev, cam, film, S2, D.IntegratorType.path(0), aovs=["radiance_sq"])
    # every pointer NULL: a plain render
    opts.aovs = C.pointer(capi.AovFilms())
    assert call(P8, opts) == 0 and np.array_equal(_bits(img), _bits(ref.film))
    mctx = api.MultiContext([0])
    try:
        ms = api.MultiScene(mctx, scene)
        opts = capi.RenderOpts()
        opts.flags = capi.RENDER_AOVS
        opts.aovs = C.pointer(films)
        ig = capi.integrator(P8)
        stats, per = capi.Stats(), (capi.Stats * 1)()
        rc = L.yk_multi_render(mctx._h, ms._h, C.byref(cam_c), C.byref(fs), C.byref(sm), C.byref(ig), C.c_void_p(tiles.ctypes.data),
                               len(tiles), C.byref(opts), C.c_void_p(img.ctypes.data), C.byref(stats), per)
        assert rc == -1 and b"yk_multi_render" in L.yk_last_error()
        ms.close()
    finally:
        mctx.close()
    r = _render(gpu_ctx, dev, cam, film, S2, P8, aovs=ALL)
    for name in ALL:
        assert np.array_equal(_bits(r.aovs[name]), _bits(ref.aovs[name])), name


@pytest.mark.gpu
def test_headless_writes_the_views(tmp_path):
    import io
    from oracle import post
    out = tmp_path / "box.exr"
    paths = {n: tmp_path / f"{n}.exr" for n in ALL}
    argv = ["--out", str(out), "--integrator", "path", "--max-depth", "8", "--sampler", "stratified", "2", "2", "--res", "48", "32",
            "--tone-map", "raw"]
    for n, p in paths.items():
        argv += ["--aov", f"{n}={p}"]
    log = io.StringIO()
    headless.render(headless.parse_args(argv), out=log)
    # the same render through the API
    scene, cam, fs = headless.try_load_scene("")
    ctx = api.Context(0)
    dev = api.Scene(ctx, scene)
    try:
        r = _render(ctx, dev, cam, D.FilmSettings((48, 32), 16), D.SamplerType.stratified(2, 2), P8, aovs=ALL)
    finally:
        dev.close()
        ctx.close()
    assert np.array_equal(_bits(post.read_exr_rgb(str(out))), _bits(r.film))
    for n, p in paths.items():
        assert f"wrote {n} to {p}" in log.getvalue()
        assert np.array_equal(_bits(post.read_exr_rgb(str(p))), _bits(r.aovs[n])), n
