"""Depth of field: the thin-lens camera of `yk_render_opts.lens` (YK_RENDER_THIN_LENS), `Renderer.render(lens=...)`.

pbrt-v3's PerspectiveCamera::GenerateRay: after the film jitter (dimensions 0-1) a camera sample draws the lens sample
(dimensions 2-3), maps it to the disk of radius R and aims the ray at the point of the pinhole ray on the plane of focus at
depth F (include/yuki_gpu.h states the float32 ops). The GPU is compared bit for bit with the oracle's render under the same
lens (`yko_render_lens`, tests/oracle_lens.cpp, built here from the oracle's own sources), and its geometry with a float64
restatement that shares nothing with either. Radius 0 is the pinhole, bit for bit.
"""
import ctypes as C
import io
import os
import shutil
import subprocess

import numpy as np
import pytest

from test_adaptive_sampling import adaptive_counts, sums_over_counts
from test_render_aovs import VIEWS, _bits, _debug_integrator, _scenes
from test_render_limits import (COUNTERS, DEEP_FILM, DEEP_PINS, DEEP_SAMPLER, LARGE_TREE_DEPTH, LARGE_TREE_FILM, glass_plates,
                                one_pixel_tiles, white_box)
from yuki_b200 import api, capi, desc as D, headless

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
S44, U16 = D.SamplerType.stratified(4, 4), D.SamplerType.uniform(16)
P8, W5 = D.IntegratorType.path(8), D.IntegratorType.whitted(5)
FILM = D.FilmSettings((40, 24), 8)
# The Cornell box's camera sits at z = 0.8 looking down -z; the tall box's faces lie 1.05 ... 1.26 m in front of it.
LENSES = {"r0.02-f1.1-tall-box": D.ThinLens(0.02, 1.1), "r0.06-f0.6": D.ThinLens(0.06, 0.6)}
LENS_SCENES = ("glass-cornell-rect", "material-room", "sphere-field", "open-scene")
STATS = COUNTERS + ("samples", "primary_hit_hash")


# ---- the oracle with a lens ------------------------------------------------------------------------------------------
@pytest.fixture(scope="session")
def olens(oracle, tmp_path_factory):
    """OracleScene with `render(..., lens=D.ThinLens)`: yko_render_lens of tests/oracle_lens.cpp, compiled here with
    oracle/Makefile's flags into a library that carries the oracle's own entry points (its scenes are the oracle's)."""
    lib_path = tmp_path_factory.mktemp("oracle_lens") / "liboracle_lens.so"
    subprocess.check_call([os.environ.get("CXX", "g++"), "-O3", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-Wall",
                           "-Wextra", "-pthread", "-shared", "-Wl,-Bsymbolic", "-I", os.path.join(ROOT, "oracle"),
                           "-o", str(lib_path), os.path.join(HERE, "oracle_lens.cpp")])
    L = C.CDLL(str(lib_path))
    vp, u32 = C.c_void_p, C.c_uint32
    L.yko_scene_create.argtypes = [C.POINTER(capi.HostSceneDesc)]
    L.yko_scene_create.restype = vp
    L.yko_scene_destroy.argtypes = [vp]
    L.yko_scene_destroy.restype = None
    L.yko_render_lens.argtypes = [vp, C.POINTER(capi.CameraParams), C.POINTER(capi.FilmSettings), C.POINTER(capi.Sampler),
                                  C.POINTER(capi.Integrator), vp, u32, u32, vp, vp, u32, C.POINTER(oracle.OStats), C.c_float, C.c_float]

    class LensScene:
        def __init__(self, scene):
            hd, keep = capi.build_host_scene_desc(scene)
            self._h = L.yko_scene_create(C.byref(hd))
            del keep
            assert self._h

        def render(self, cam, film, smp, integ, lens, tiles=None, want_hit_ids=False, film_out=None, threads=0):
            res_x, res_y = int(film.res[0]), int(film.res[1])
            out = film_out if film_out is not None else np.zeros((res_y, res_x, 3), np.float32)
            ids = np.full((res_y, res_x), -1, np.int32) if want_hit_ids else None
            cp, fs, sm, ig = capi.camera_params(cam), capi.film_settings(film), capi.sampler(smp), capi.integrator(integ)
            st = oracle.OStats()
            tptr, nt = None, 0
            if tiles is not None:
                tiles = np.ascontiguousarray(tiles, dtype=capi.TILE_DTYPE)
                tptr, nt = tiles.ctypes.data, len(tiles)
            assert L.yko_render_lens(self._h, C.byref(cp), C.byref(fs), C.byref(sm), C.byref(ig), tptr, nt, threads, out.ctypes.data,
                                     ids.ctypes.data if ids is not None else None, 0, C.byref(st), float(lens.radius),
                                     float(lens.focal_distance)) == 0
            return out, ids, st

        def __del__(self):
            L.yko_scene_destroy(self._h)

    return LensScene


def _assert_parity(r, o, what=""):
    o_img, o_ids, o_st = o
    assert np.array_equal(_bits(r.film), _bits(o_img)), what
    if o_ids is not None:
        assert np.array_equal(r.hit_ids, o_ids), what
    for k in COUNTERS + ("samples", "primary_hit_hash"):
        assert getattr(r.stats, k) == getattr(o_st, k), (what, k)


def _assert_same(r, ref, what=""):
    assert np.array_equal(_bits(r.film), _bits(ref.film)), what
    if ref.hit_ids is not None:
        assert np.array_equal(r.hit_ids, ref.hit_ids), what
    for k in STATS:
        assert getattr(r.stats, k) == getattr(ref.stats, k), (what, k)


# ---- CPU: ABI layout, loader, validation, CLI, checkpoint meta ------------------------------------------------------
LAYOUT_C = r"""
#include <stddef.h>
#include <stdio.h>
#include "yuki_gpu.h"
int main(void) {
    printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(yk_thin_lens), offsetof(yk_thin_lens, lens_radius),
           offsetof(yk_thin_lens, focal_distance), sizeof(yk_render_opts), offsetof(yk_render_opts, adaptive),
           offsetof(yk_render_opts, lens), sizeof(yk_pbrt_result), offsetof(yk_pbrt_result, res_y),
           offsetof(yk_pbrt_result, lens_radius), offsetof(yk_pbrt_result, focal_distance));
    printf("%u\n", (unsigned)YK_RENDER_THIN_LENS);
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
    T, R, P = capi.ThinLens, capi.RenderOpts, capi.PbrtResult
    assert got == [C.sizeof(T), T.lens_radius.offset, T.focal_distance.offset, C.sizeof(R), R.adaptive.offset, R.lens.offset,
                   C.sizeof(P), P.res_y.offset, P.lens_radius.offset, P.focal_distance.offset]
    assert int(lines[1]) == capi.RENDER_THIN_LENS
    # appended: every field an older caller sets keeps its offset
    assert R.lens.offset == R.adaptive.offset + 8 and P.lens_radius.offset == P.res_y.offset + 4


def _pbrt(tmp_path, camera_params=""):
    f = tmp_path / "lens.pbrt"
    f.write_text(f'LookAt 0 0 5  0 0 0  0 1 0\nCamera "perspective" "float fov" [30]{camera_params}\nWorldBegin\n'
                 'Shape "trianglemesh" "integer indices" [0 1 2] "point P" [0 0 0 1 0 0 0 1 0]\nWorldEnd\n')
    return f


def test_pbrt_loader_reads_lensradius_and_focaldistance(tmp_path):
    _, cam, _, lens = api.load_pbrt(str(_pbrt(tmp_path, ' "float lensradius" [0.125] "float focaldistance" [3.5]')), with_lens=True)
    assert lens == D.ThinLens(0.125, 3.5) and cam.fov_deg == 30.0
    _, _, _, lens = api.load_pbrt(str(_pbrt(tmp_path, ' "float lensradius" 0.25')), with_lens=True)
    assert lens == D.ThinLens(0.25, 1e6)                                  # pbrt-v3's default focal distance
    _, _, _, lens = api.load_pbrt(str(_pbrt(tmp_path)), with_lens=True)
    assert lens == D.ThinLens(0.0, np.float32(1e6))
    # without with_lens the call returns what it always did
    assert len(api.load_pbrt(str(_pbrt(tmp_path)))) == 3


def test_mitsuba_loader_reports_a_pinhole(tmp_path):
    from test_mitsuba import write_scene
    h = C.c_void_p()
    capi.check(capi.lib().yk_mitsuba_load(str(write_scene(tmp_path)).encode(), 1, D.SPLIT_SAH, C.byref(h)))
    try:
        r = capi.lib().yk_pbrt_view(h).contents
        assert (r.lens_radius, r.focal_distance) == (0.0, np.float32(1e6))
    finally:
        capi.lib().yk_pbrt_destroy(h)


@pytest.mark.parametrize("radius,focal", [(-0.1, 1.0), (float("nan"), 1.0), (float("inf"), 1.0), (1e39, 1.0), (0.1, 0.0), (0.1, -1.0),
                                          (0.1, float("nan")), (0.1, float("inf"))])
def test_thin_lens_is_validated_when_constructed(radius, focal):
    with pytest.raises(ValueError):
        D.ThinLens(radius, focal)


def test_thin_lens_accepts_the_pinhole_and_defaults():
    assert D.ThinLens(0.0).focal_distance == 1e6
    assert D.ThinLens(0.5, 2.0).radius == 0.5


@pytest.mark.parametrize("argv", [["--lens-radius", "-1"], ["--lens-radius", "nan"], ["--lens-radius", "0.1", "--focal-distance", "0"],
                                  ["--thin-lens", "--focal-distance", "-2"], ["--focal-distance", "2"], ["--lens-radius", "inf"]])
def test_headless_lens_arguments_are_parser_errors(argv):
    with pytest.raises(SystemExit):
        headless.parse_args(["--out", "x.exr"] + argv)


def test_headless_lens_arguments(tmp_path):
    file_lens = D.ThinLens(0.1, 4.0)
    a = headless.parse_args(["--out", "x.exr"])
    assert headless.lens_from_args(a, file_lens) is None                 # the pinhole, as the reference
    a = headless.parse_args(["--out", "x.exr", "--thin-lens"])
    assert headless.lens_from_args(a, file_lens) == file_lens
    a = headless.parse_args(["--out", "x.exr", "--lens-radius", "0.3"])
    assert headless.lens_from_args(a, file_lens) == D.ThinLens(0.3, 4.0)
    a = headless.parse_args(["--out", "x.exr", "--lens-radius", "0.3", "--focal-distance", "2.5"])
    assert headless.lens_from_args(a, file_lens) == D.ThinLens(0.3, 2.5)
    a = headless.parse_args(["--out", "x.exr", "--thin-lens", "--focal-distance", "2.5"])
    assert headless.lens_from_args(a, file_lens) == D.ThinLens(0.1, 2.5)
    *_, lens = headless.try_load_scene(str(_pbrt(tmp_path, ' "float lensradius" [0.125] "float focaldistance" [3.5]')), with_lens=True)
    assert lens == D.ThinLens(0.125, 3.5)
    *_, lens = headless.try_load_scene("", with_lens=True)
    assert lens.radius == 0.0


def test_checkpoint_meta_names_the_lens(tmp_path, xf):
    from yuki_b200 import scenes
    _, cam = scenes.cornell(xf)
    fs = D.FilmSettings((16, 16), 8, accumulate=True)
    smp, integ = D.SamplerType.stratified(2, 2), D.IntegratorType.path(3)
    rn = api.Renderer.__new__(api.Renderer)

    def run(lens, film=None, path=None):
        film = film or api.Film(fs)
        kw = {} if lens is None else {"lens": lens}
        rn.render_progressive(None, cam, film, smp, integ, samples_per_pass=2, max_passes=1, checkpoint_path=path,
                              render_fn=lambda tiles, out: None, **kw)
        return film
    plain = run(None).meta
    assert "lens" not in plain and run(D.ThinLens(0.0, 2.0)).meta == plain   # radius 0 is the pinhole's render
    path = str(tmp_path / "ck.npz")
    film = run(D.ThinLens(0.05, 1.5), path=path)
    assert film.meta["lens"] == [float(np.float32(0.05)), 1.5] and {k: v for k, v in film.meta.items() if k != "lens"} == plain
    resumed = api.Film.load(path)
    run(D.ThinLens(0.05, 1.5), film=resumed)                                # the same lens continues
    for other in (None, D.ThinLens(0.05, 2.0), D.ThinLens(0.04, 1.5)):
        with pytest.raises(ValueError, match="other settings"):
            run(other, film=api.Film.load(path))


# ---- GPU: bit-exact against the oracle ------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def scene_cache(gpu_ctx, xf):
    cache = {}
    yield lambda sid: cache.setdefault(sid, _load(gpu_ctx, xf, sid))
    for _, _, dev in cache.values():
        dev.close()


def _load(gpu_ctx, xf, sid):
    scene, cam = _scenes(xf)[sid]()
    return scene, cam, api.Scene(gpu_ctx, scene)


def _render(ctx, dev, cam, film, smp, integ, **kw):
    return api.Renderer(ctx).render(dev, cam, film, smp, integ, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("lens_id", sorted(LENSES))
@pytest.mark.parametrize("smp", [S44, U16], ids=["stratified-4x4", "uniform-16"])
@pytest.mark.parametrize("integ", [P8, W5], ids=["path-8", "whitted-5"])
@pytest.mark.parametrize("scene_id", LENS_SCENES)
def test_lens_render_equals_the_oracle(gpu_ctx, scene_cache, olens, scene_id, integ, smp, lens_id):
    scene, cam, dev = scene_cache(scene_id)
    lens = LENSES[lens_id]
    r = _render(gpu_ctx, dev, cam, FILM, smp, integ, want_hit_ids=True, lens=lens)
    o = olens(scene).render(cam, FILM, smp, integ, lens, want_hit_ids=True)
    _assert_parity(r, o, (scene_id, lens_id))
    pin = _render(gpu_ctx, dev, cam, FILM, smp, integ, want_hit_ids=True)
    assert not np.array_equal(_bits(r.film), _bits(pin.film))               # the lens did change the picture


@pytest.mark.gpu
@pytest.mark.parametrize("integ", [P8, W5, D.IntegratorType.bvh_intersections(), D.IntegratorType.debug(D.INTEGRATOR_SHADING_UVS)],
                         ids=["path-8", "whitted-5", "bvh-intersections", "shading-uvs"])
def test_radius_zero_is_the_pinhole_bit_for_bit(gpu_ctx, scene_cache, integ):
    _, cam, dev = scene_cache("glass-cornell-rect")
    ref = _render(gpu_ctx, dev, cam, FILM, S44, integ, want_hit_ids=True)
    for lens in (D.ThinLens(0.0), D.ThinLens(0.0, 0.5)):
        _assert_same(_render(gpu_ctx, dev, cam, FILM, S44, integ, want_hit_ids=True, lens=lens), ref, lens)


@pytest.mark.gpu
@pytest.mark.parametrize("integ", [P8, W5], ids=["path-8", "whitted-5"])
def test_accumulating_film_with_a_lens(gpu_ctx, scene_cache, olens, integ):
    scene, cam, dev = scene_cache("glass-cornell-rect")
    lens = LENSES["r0.02-f1.1-tall-box"]
    acc = D.FilmSettings(FILM.res, FILM.tile_dim, accumulate=True)
    base = api.film_tiles(acc)
    tiles = np.concatenate([base] * 3)
    tiles["sample"] = np.repeat(np.arange(3, dtype=np.uint16), len(base))
    start = np.full((FILM.res[1], FILM.res[0], 3), 0.125, np.float32)
    r = _render(gpu_ctx, dev, cam, acc, S44, integ, tiles=tiles, film_out=start.copy(), lens=lens)
    o = olens(scene).render(cam, acc, S44, integ, lens, tiles=tiles, film_out=start.copy())
    _assert_parity(r, o, "accumulate")


@pytest.mark.gpu
@pytest.mark.parametrize("integ", [P8, W5], ids=["path-8", "whitted-5"])
def test_adaptive_render_with_a_lens(gpu_ctx, scene_cache, olens, integ):
    """The counts are the numpy rule over the oracle's per-sample films under the lens, the film their float32 sums / n."""
    scene, cam, dev = scene_cache("glass-cornell-rect")
    lens = LENSES["r0.06-f0.6"]
    a = D.Adaptive(4, 4, 0.2, 0.0)
    acc = D.FilmSettings(FILM.res, FILM.tile_dim, accumulate=True)
    base = api.film_tiles(acc)
    osc = olens(scene)
    lis = []
    for k in range(S44.samples_per_pixel()):
        t = base.copy()
        t["sample"] = k
        lis.append(osc.render(cam, acc, S44, integ, lens, tiles=t, film_out=np.zeros((FILM.res[1], FILM.res[0], 3), np.float32))[0])
    counts = adaptive_counts(lis, a)
    assert counts.min() < counts.max()
    r = _render(gpu_ctx, dev, cam, FILM, S44, integ, adaptive=a, aovs=["radiance_sq"], lens=lens)
    assert np.array_equal(r.sample_counts, counts)
    assert np.array_equal(_bits(r.film), _bits(sums_over_counts(lis, counts)))
    assert np.array_equal(_bits(r.aovs["radiance_sq"]), _bits(sums_over_counts(lis, counts, square=True)))
    assert r.stats.samples == int(counts.sum())


@pytest.mark.gpu
@pytest.mark.parametrize("integ", [P8, W5], ids=["path-8", "whitted-5"])
def test_companion_views_equal_the_debug_integrators_under_the_lens(gpu_ctx, scene_cache, olens, integ):
    scene, cam, dev = scene_cache("material-room")
    lens = LENSES["r0.02-f1.1-tall-box"]
    r = _render(gpu_ctx, dev, cam, FILM, S44, integ, aovs=list(VIEWS), lens=lens)
    osc = olens(scene)
    for name in VIEWS:
        d = _render(gpu_ctx, dev, cam, FILM, S44, _debug_integrator(name), want_hit_ids=True, lens=lens)
        assert np.array_equal(_bits(r.aovs[name]), _bits(d.film)), name
        _assert_parity(d, osc.render(cam, FILM, S44, _debug_integrator(name), lens, want_hit_ids=True), name)


@pytest.mark.gpu
def test_pipes_ray_sorts_and_batch_shapes_leave_the_lens_film_unchanged(gpu_ctx, scene_cache, olens, monkeypatch):
    scene, cam, dev = scene_cache("glass-cornell-rect")
    lens = LENSES["r0.06-f0.6"]
    film = D.FilmSettings((64, 48), 16)
    o = olens(scene).render(cam, film, S44, P8, lens, want_hit_ids=True)
    for kw in ({"pipes": 1, "ray_sort": 1}, {"pipes": 2, "ray_sort": 2}, {"pipes": 2, "ray_sort": 3},
               {"pipes": 2, "ray_sort": 2 | 16, "wavefront_paths": 4096}):   # 16: YK_RAY_SORT_TRACE_ONLY
        _assert_parity(_render(gpu_ctx, dev, cam, film, S44, P8, want_hit_ids=True, lens=lens, **kw), o, kw)
    monkeypatch.setenv("YK_MAX_BATCH_SAMPLES", "3")
    _assert_parity(_render(gpu_ctx, dev, cam, film, S44, P8, want_hit_ids=True, lens=lens, pipes=2), o, "3 samples per batch")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["0", "1"])
def test_both_shadow_modes_with_a_lens(xf, olens, monkeypatch, mode):
    monkeypatch.setenv("YK_SHADOW_MODE", mode)
    scene, cam = _scenes(xf)["material-room"]()
    lens = LENSES["r0.02-f1.1-tall-box"]
    ctx = api.Context(0)
    try:
        dev = api.Scene(ctx, scene)
        for integ in (P8, W5):
            _assert_parity(_render(ctx, dev, cam, FILM, S44, integ, want_hit_ids=True, lens=lens),
                           olens(scene).render(cam, FILM, S44, integ, lens, want_hit_ids=True), (mode, integ))
        dev.close()
    finally:
        ctx.close()


# ---- GPU: the limits yk_render admits, with the 2 lens dimensions -------------------------------------------------
@pytest.mark.gpu
def test_deep_path_with_a_lens_matches_the_oracle(gpu_ctx, olens, xf):
    """Path keeps its sampler dimension in 21 bits: depth 255 with 32 lights draws at most 4 + 255 * 67 = 17089 dimensions."""
    lens = D.ThinLens(0.05, 1.5)
    scene, cam = white_box(xf)
    dev = api.Scene(gpu_ctx, scene)
    tiles = one_pixel_tiles(DEEP_FILM, DEEP_PINS)
    r = _render(gpu_ctx, dev, cam, DEEP_FILM, DEEP_SAMPLER, D.IntegratorType.path(255), tiles=tiles,
                film_out=np.zeros((DEEP_FILM.res[1], DEEP_FILM.res[0], 3), np.float32), lens=lens)
    _assert_parity(r, olens(scene).render(cam, DEEP_FILM, DEEP_SAMPLER, D.IntegratorType.path(255), lens, tiles=tiles), "pinned deep paths")
    film = D.FilmSettings((64, 48), 16)
    r = _render(gpu_ctx, dev, cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.path(255), want_hit_ids=True, lens=lens)
    o = olens(scene).render(cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.path(255), lens, want_hit_ids=True)
    _assert_parity(r, o, "full film at depth 255")
    dev.close()
    scene, cam = white_box(xf, n_lights=32)
    dev = api.Scene(gpu_ctx, scene)
    film = D.FilmSettings((24, 24), 16)
    r = _render(gpu_ctx, dev, cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.path(80), want_hit_ids=True, lens=lens)
    _assert_parity(r, olens(scene).render(cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.path(80), lens, want_hit_ids=True),
                   "32 lights at depth 80: the 4096-dimension table ends inside the paths")
    dev.close()


@pytest.mark.gpu
@pytest.mark.parametrize("smp", [D.SamplerType.stratified(2, 2), D.SamplerType.uniform(4)], ids=["stratified", "uniform"])
def test_large_whitted_tree_with_a_lens_matches_the_oracle(gpu_ctx, olens, xf, smp):
    """Whitted keeps its dimension in beta.x (32 bits): a ~54 k-node tree with 32 lights passes 2^21 dimensions."""
    lens = D.ThinLens(0.01, 2.0)
    scene, cam = glass_plates(xf)
    dev = api.Scene(gpu_ctx, scene)
    integ = D.IntegratorType.whitted(LARGE_TREE_DEPTH)
    r = _render(gpu_ctx, dev, cam, LARGE_TREE_FILM, smp, integ, want_hit_ids=True, lens=lens)
    o = olens(scene).render(cam, LARGE_TREE_FILM, smp, integ, lens, want_hit_ids=True)
    assert o[2].ray_count > 40000 * smp.samples_per_pixel() // 2
    _assert_parity(r, o, "32 lights")
    dev.close()


# ---- GPU: the geometry against float64 ------------------------------------------------------------------------------
QUAD_HALF = 4.0


def _quad_scene(xf, z):
    """A uv-mapped quad facing the camera (which sits at the origin looking down -z) at depth z: u, v = (x, y) / 8 + 1/2."""
    s = D.SceneDesc()
    white = s.add_material(D.Material(D.MAT_MATTE, (s.add_texture(D.Texture.constant(0.5)), s.add_texture(D.Texture.constant(0.0)))))
    h = QUAD_HALF
    pts = np.array([[-h, -h, -z], [h, -h, -z], [h, h, -z], [-h, h, -z]], np.float32)
    uvs = np.array([[0, 0], [1, 0], [1, 1], [0, 1]], np.float32)
    s.meshes.append(D.Mesh(xf.identity(), pts, np.array([0, 1, 2, 0, 2, 3], np.uint32), white, uvs=uvs))
    return s


def _disk64(u):
    o = u * 2.0 - 1.0
    out = np.zeros_like(o)
    nz = (o[:, 0] != 0) | (o[:, 1] != 0)
    ax = np.abs(o[:, 0]) > np.abs(o[:, 1])
    with np.errstate(divide="ignore", invalid="ignore"):
        theta = np.where(ax, np.pi / 4 * (o[:, 1] / o[:, 0]), np.pi / 2 - np.pi / 4 * (o[:, 0] / o[:, 1]))
    r = np.where(ax, o[:, 0], o[:, 1])
    out[:, 0] = np.where(nz, r * np.cos(theta), 0.0)
    out[:, 1] = np.where(nz, r * np.sin(theta), 0.0)
    return out


def _hits64(c2w, r2c, pf, u, lens, z):
    """float64 thin lens: world hit point on the plane at depth z of each camera sample, and the lens offset (lx, ly)."""
    p = np.concatenate([pf, np.zeros((len(pf), 1)), np.ones((len(pf), 1))], axis=1) @ r2c.T
    p = p[:, :3] / p[:, 3:4]
    d = p / np.linalg.norm(p, axis=1, keepdims=True)
    lxy = lens.radius * _disk64(u) if lens is not None else np.zeros((len(pf), 2))
    f = d * (lens.focal_distance / d[:, 2:3]) if lens is not None else d
    o_cam = np.concatenate([lxy, np.zeros((len(pf), 1))], axis=1)
    dc = f - o_cam
    dc /= np.linalg.norm(dc, axis=1, keepdims=True)
    o = o_cam @ c2w[:3, :3].T + c2w[:3, 3]
    dw = dc @ c2w[:3, :3].T
    t = (-z - o[:, 2]) / dw[:, 2]
    return o + dw * t[:, None], lxy


@pytest.mark.gpu
@pytest.mark.parametrize("depth", ["F", "F/2", "2F"])
def test_uv_of_each_pixel_follows_the_float64_thin_lens(gpu_ctx, xf, depth):
    lens = D.ThinLens(0.25, 2.0)
    z = {"F": 2.0, "F/2": 1.0, "2F": 4.0}[depth]
    cam = D.CameraParameters((0.0, 0.0, 0.0), (0.0, 0.0, -1.0), fov_axis=D.FOV_X, fov_deg=40.0)
    film, smp = D.FilmSettings((48, 32), 16), D.SamplerType.uniform(1)
    dev = api.Scene(gpu_ctx, _quad_scene(xf, z))
    integ = D.IntegratorType.debug(D.INTEGRATOR_SHADING_UVS)
    r = _render(gpu_ctx, dev, cam, film, smp, integ, lens=lens)
    pin = _render(gpu_ctx, dev, cam, film, smp, integ)
    dev.close()
    ys, xs = np.mgrid[0:film.res[1], 0:film.res[0]]
    idx = np.stack([xs.ravel(), ys.ravel(), np.zeros(xs.size, int)], axis=1).astype(np.uint32)
    draws = api.sampler_draws(gpu_ctx, smp, idx, [2, 2]).reshape(-1, 4).astype(np.float64)
    pf = idx[:, :2].astype(np.float64) + draws[:, :2]
    cm = api.make_camera(cam, film)
    c2w, r2c = np.array(cm.camera_to_world[:], np.float64).reshape(4, 4), np.array(cm.raster_to_camera[:], np.float64).reshape(4, 4)
    p_lens, lxy = _hits64(c2w, r2c, pf, draws[:, 2:4], lens, z)
    p_pin, _ = _hits64(c2w, r2c, pf, None, None, z)
    uv = r.film.reshape(-1, 3)[:, :2].astype(np.float64)
    uv_pin = pin.film.reshape(-1, 3)[:, :2].astype(np.float64)
    tol = 1e-6
    assert np.abs(uv - (p_lens[:, :2] / (2 * QUAD_HALF) + 0.5)).max() < tol
    assert np.abs(uv_pin - (p_pin[:, :2] / (2 * QUAD_HALF) + 0.5)).max() < tol
    # the circle of confusion: the hit moves by (1 - z / F) * (lx, ly), in world axes
    shift = (1.0 - z / lens.focal_distance) * (np.concatenate([lxy, np.zeros((len(lxy), 1))], axis=1) @ c2w[:3, :3].T)
    assert np.abs((p_lens - p_pin) - shift).max() < 1e-9
    if depth == "F":   # the plane of focus is sharp
        assert np.abs(uv - uv_pin).max() < tol
    else:
        assert np.abs(uv - uv_pin).max() > 0.25 * lens.radius / (2 * QUAD_HALF) * abs(1.0 - z / lens.focal_distance)


# ---- GPU: several GPUs ----------------------------------------------------------------------------------------------
def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:  # noqa: BLE001
        return 0


def _check_multi(gpu_ctx_or_none, xf, device_ids):
    scene, cam = _scenes(xf)["glass-cornell-rect"]()
    film = D.FilmSettings((150, 100), 16)
    lens = LENSES["r0.02-f1.1-tall-box"]
    single = gpu_ctx_or_none or api.Context(device_ids[0])
    mctx = api.MultiContext(device_ids)
    try:
        dev = api.Scene(single, scene)
        ms = api.MultiScene(mctx, scene)
        for integ in (D.IntegratorType.path(4), D.IntegratorType.whitted(4)):
            ref = _render(single, dev, cam, film, S44, integ, want_hit_ids=True, lens=lens)
            r, per = api.multi_render(mctx, ms, cam, film, S44, integ, want_hit_ids=True, lens=lens)
            _assert_same(r, ref, (device_ids, integ))
        ms.close(); dev.close()
    finally:
        mctx.close()
        if gpu_ctx_or_none is None:
            single.close()


@pytest.mark.gpu
def test_multi_render_with_a_lens_on_one_gpu_equals_yk_render(gpu_ctx, xf, monkeypatch):
    monkeypatch.setenv("YK_MULTI_FORCE_CURSOR", "1")
    monkeypatch.setenv("YK_MULTI_RUN_TILES", "5")
    _check_multi(gpu_ctx, xf, [0])


@pytest.mark.gpu
@pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("no_peer", [False, True], ids=["peer-stores", "no-peer"])
def test_multi_render_with_a_lens_on_two_gpus_equals_yk_render(xf, monkeypatch, no_peer):
    if no_peer:
        monkeypatch.setenv("YK_MULTI_NO_PEER", "1")
    _check_multi(None, xf, [0, 1])


# ---- GPU: refusals and the CLI ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refusals_leave_the_context_usable(gpu_ctx, scene_cache, xf):
    scene, cam, dev = scene_cache("glass-cornell-rect")
    film = D.FilmSettings((16, 16), 8)
    ok = _render(gpu_ctx, dev, cam, film, S44, P8, lens=LENSES["r0.06-f0.6"])
    camc, tiles = api.make_camera(cam, film), api.film_tiles(film)
    fs, sm, ig = capi.film_settings(film), capi.sampler(S44), capi.integrator(P8)
    out = np.zeros((16, 16, 3), np.float32)
    bad = [None, (-0.1, 1.0), (float("nan"), 1.0), (float("inf"), 1.0), (0.1, 0.0), (0.1, -1.0), (0.1, float("nan")), (0.1, float("inf"))]
    mctx = api.MultiContext([0])
    ms = api.MultiScene(mctx, scene)
    try:
        for b in bad:
            opts = capi.RenderOpts()
            opts.flags = capi.RENDER_THIN_LENS
            if b is not None:
                opts.lens = C.pointer(capi.ThinLens(*b))
            rc = capi.lib().yk_render(gpu_ctx._h, dev._h, C.byref(camc), C.byref(fs), C.byref(sm), C.byref(ig),
                                      C.c_void_p(tiles.ctypes.data), len(tiles), C.byref(opts), C.c_void_p(out.ctypes.data), None)
            assert rc == -1 and (b"lens" in capi.lib().yk_last_error() or b"focal" in capi.lib().yk_last_error()), b
            rc = capi.lib().yk_multi_render(mctx._h, ms._h, C.byref(camc), C.byref(fs), C.byref(sm), C.byref(ig),
                                            C.c_void_p(tiles.ctypes.data), len(tiles), C.byref(opts), C.c_void_p(out.ctypes.data), None, None)
            assert rc == -1, b
            again = _render(gpu_ctx, dev, cam, film, S44, P8, lens=LENSES["r0.06-f0.6"])
            assert np.array_equal(_bits(again.film), _bits(ok.film))
    finally:
        ms.close(); mctx.close()


@pytest.mark.gpu
def test_headless_thin_lens_renders_the_files_lens(tmp_path, oracle, olens):
    from oracle import post
    from test_pbrt import cornell_pbrt
    path, _, _ = cornell_pbrt(tmp_path)
    text = path.read_text().replace('Camera "perspective" "float fov" [40.0]',
                                    'Camera "perspective" "float fov" [40.0] "float lensradius" [0.02] "float focaldistance" [1.1]')
    assert "lensradius" in text
    path.write_text(text)
    sc, cam, _, lens = api.load_pbrt(str(path), with_lens=True)
    assert lens == D.ThinLens(float(np.float32(0.02)), float(np.float32(1.1)))   # the file's values, as float32
    film, smp, integ = D.FilmSettings((64, 64), 16), D.SamplerType.stratified(2, 2), D.IntegratorType.whitted(3)
    common = ["--scene", str(path), "--integrator", "whitted", "--max-depth", "3", "--sampler", "stratified", "2", "2", "--res", "64", "64",
              "--tone-map", "raw"]
    log = io.StringIO()
    headless.render(headless.parse_args(common + ["--out", str(tmp_path / "lens.exr"), "--thin-lens"]), out=log)
    assert "Thin lens: radius 0.02, focal distance 1.1" in log.getvalue()
    o_img, _, _ = olens(sc).render(cam, film, smp, integ, lens)
    assert np.array_equal(post.read_exr_rgb(str(tmp_path / "lens.exr")).view(np.uint32), o_img.view(np.uint32))
    # without the flag the file renders pinhole, as the reference does
    headless.render(headless.parse_args(common + ["--out", str(tmp_path / "pin.exr")]), out=io.StringIO())
    o_img, _, _ = oracle.OracleScene(sc).render(cam, film, smp, integ)
    assert np.array_equal(post.read_exr_rgb(str(tmp_path / "pin.exr")).view(np.uint32), o_img.view(np.uint32))
    # --lens-radius with the file's focal distance
    headless.render(headless.parse_args(common + ["--out", str(tmp_path / "r.exr"), "--lens-radius", "0.04"]), out=io.StringIO())
    o_img, _, _ = olens(sc).render(cam, film, smp, integ, D.ThinLens(0.04, 1.1))
    assert np.array_equal(post.read_exr_rgb(str(tmp_path / "r.exr")).view(np.uint32), o_img.view(np.uint32))
