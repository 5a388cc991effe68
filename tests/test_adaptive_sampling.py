"""Adaptive sampling (`yk_render_opts.adaptive`, `Renderer.render(adaptive=...)`).

A pixel stops at a check point n (min_samples, min_samples + step, ... below spp) once, in all three channels, the squared
standard error of its mean, computed in float32 from S = sum li and Q = sum li * li in ascending sample order, is at most
(rel * mean + abs)^2. Every GPU test compares bits: the oracle gives each sample's li on its own (`_per_sample_films`), the
numpy float32 restatement of the rule (`adaptive_counts`) must give the GPU's count of every pixel, the film must be the
float32 S / n, and the companion films their own sums / n. The ray and traversal counters must equal those of an oracle
accumulating render over exactly the (pixel, sample) pairs traced, whose film divided by the counts is the same film again.
"""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from test_render_aovs import ALL, VIEWS, _bits, _debug_integrator, _per_sample_films, _scenes, SCENE_IDS
from test_render_limits import COUNTERS
from yuki_b200 import api, capi, desc as D, headless

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
S44, U16 = D.SamplerType.stratified(4, 4), D.SamplerType.uniform(16)
P8, W5 = D.IntegratorType.path(8), D.IntegratorType.whitted(5)
FILM = D.FilmSettings((24, 16), 8)
# (min_samples, step, rel_error, abs_error): checks at 4, 8, 12 / at 2, 5, 8, 11, 14 of 16 samples
SETTINGS = {"min4-step4-rel0.2": D.Adaptive(4, 4, 0.2, 0.0), "min2-step3-rel0.15-abs0.01": D.Adaptive(2, 3, 0.15, 0.01)}
MIN_PIXELS = 2   # each case has at least this many pixels at min_samples, strictly between, and at spp (on the oracle)
STATS = COUNTERS + ("samples", "primary_hit_hash")


def check_points(a: D.Adaptive, spp: int):
    return list(range(a.min_samples, spp, a.step))


def adaptive_counts(lis, a: D.Adaptive):
    """The stopping rule in numpy float32 over per-sample films li_k (k ascending): each pixel's sample count."""
    spp = len(lis)
    shape = lis[0].shape[:2]
    s, q = np.zeros_like(lis[0]), np.zeros_like(lis[0])
    counts = np.full(shape, spp, np.uint32)
    active = np.ones(shape, bool)
    rel, abs_err = np.float32(a.rel_error), np.float32(a.abs_error)
    checks = set(check_points(a, spp))
    for k, li in enumerate(lis):
        s = s + li
        q = q + li * li
        n = k + 1
        if n in checks:
            nf = np.float32(n)
            m = s / nf
            v = q / nf - m * m
            v = np.where(v < 0, np.float32(0), v)
            e2 = v / (nf - np.float32(1))
            t = rel * m + abs_err
            stop = active & (e2 <= t * t).all(axis=2)
            counts[stop] = n
            active &= ~stop
    return counts


def sums_over_counts(lis, counts, square=False):
    """Per pixel, the float32 sum of li_k (or li_k * li_k) over k < count in ascending k, / count."""
    acc = np.zeros_like(lis[0])
    out = np.zeros_like(lis[0])
    for k, li in enumerate(lis):
        acc = acc + (li * li if square else li)
        done = counts == k + 1
        out[done] = acc[done] / np.float32(k + 1)
    return out


def traced_tiles(counts):
    """1x1 tiles (pixel, k) for every k < the pixel's count, in ascending k (row-major pixels within one k)."""
    ys, xs = np.nonzero(np.ones_like(counts, bool))
    parts = []
    for k in range(int(counts.max())):
        sel = counts[ys, xs] > k
        t = np.zeros(int(sel.sum()), dtype=capi.TILE_DTYPE)
        t["x0"], t["y0"], t["x1"], t["y1"] = xs[sel], ys[sel], xs[sel] + 1, ys[sel] + 1
        t["sample"] = k
        parts.append(t)
    return np.concatenate(parts)


# ---- CPU: the rule, ABI layout, refusals, CLI, and the oracle's count mix -------------------------------------------
def test_rule_on_synthetic_streams():
    spp = 16
    rng = np.random.default_rng(3)
    a = D.Adaptive(4, 5, 0.05, 0.0)
    assert check_points(a, spp) == [4, 9, 14]
    lis = [np.zeros((3, 4, 3), np.float32) for _ in range(spp)]
    for k, li in enumerate(lis):
        li[0, :] = 0.0                                  # black
        li[1, :] = np.float32(0.37)                     # constant
        li[2, :2] = rng.random((2, 3), dtype=np.float32) * 4.0   # noisy
        li[2, 2] = np.nan if k == 1 else 0.5            # a NaN sample before the first check: never stops
        li[2, 3] = 1.0 if k < 9 else 100.0              # constant up to the first check: stops there, blind to what follows
    c = adaptive_counts(lis, a)
    assert (c[0] == 4).all() and (c[1] == 4).all()
    assert c[2, 2] == spp and c[2, 3] == 4 and (c[2, :2] == spp).all()
    # a NaN from the first sample on: the rule never stops it, whatever the tolerance
    nan = [np.full((1, 1, 3), np.nan, np.float32) for _ in range(spp)]
    assert adaptive_counts(nan, D.Adaptive(2, 1, 1e30, 1e30))[0, 0] == spp
    # a pixel that converges at the second check: constant until the first, then the spread shrinks under the tolerance
    a2 = D.Adaptive(2, 2, 0.3, 0.0)
    assert check_points(a2, 9) == [2, 4, 6, 8]
    s = [np.full((1, 1, 3), v, np.float32) for v in (1.0, 2.0, 1.5, 1.5, 1.5, 1.5, 1.5, 1.5, 1.5)]
    assert adaptive_counts(s, a2)[0, 0] == 4
    # min_samples >= spp: no check, every pixel runs to spp
    assert check_points(D.Adaptive(16, 1, 1.0, 1.0), 16) == [] and (adaptive_counts(lis, D.Adaptive(16, 1, 1.0, 1.0)) == spp).all()


LAYOUT_C = r"""
#include <stddef.h>
#include <stdio.h>
#include "yuki_gpu.h"
int main(void) {
    printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(yk_render_opts), offsetof(yk_render_opts, aovs),
           offsetof(yk_render_opts, adaptive), sizeof(yk_adaptive), offsetof(yk_adaptive, min_samples), offsetof(yk_adaptive, step),
           offsetof(yk_adaptive, rel_error), offsetof(yk_adaptive, abs_error), offsetof(yk_adaptive, sample_counts));
    printf("%u\n", (unsigned)YK_RENDER_ADAPTIVE);
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
    A, R = capi.Adaptive, capi.RenderOpts
    assert got == [C.sizeof(R), R.aovs.offset, R.adaptive.offset, C.sizeof(A), A.min_samples.offset, A.step.offset,
                   A.rel_error.offset, A.abs_error.offset, A.sample_counts.offset]
    assert int(lines[1]) == capi.RENDER_ADAPTIVE
    # appended after `aovs`, which keeps its offset
    assert R.aovs.offset == R._reserved.offset + 4 and R.adaptive.offset == R.aovs.offset + C.sizeof(C.c_void_p)


def test_python_refusals_before_the_library():
    rn = api.Renderer(None)   # no context: every refusal must happen before anything touches the library
    bad = [D.Adaptive(1, 4, 0.1), D.Adaptive(4, 0, 0.1), D.Adaptive(4, 4, -0.1), D.Adaptive(4, 4, 0.1, -1.0),
           D.Adaptive(4, 4, float("nan")), D.Adaptive(4, 4, 0.1, float("inf")), D.Adaptive(4, 4, 1e39)]
    for a in bad:
        with pytest.raises(ValueError):
            rn.render(None, None, FILM, S44, P8, adaptive=a)
    ok = D.Adaptive()
    acc = D.FilmSettings((24, 16), 8, accumulate=True)
    with pytest.raises(ValueError, match="averaging film"):
        rn.render(None, None, acc, S44, P8, adaptive=ok)
    for integ in [_debug_integrator(n) for n in VIEWS]:
        with pytest.raises(ValueError, match="Path or Whitted"):
            rn.render(None, None, FILM, S44, integ, adaptive=ok)
    with pytest.raises(ValueError, match="needs adaptive"):
        rn.render(None, None, FILM, S44, P8, sample_counts_out=np.zeros((16, 24), np.uint32))
    with pytest.raises(ValueError):
        rn.launch(None, None, api.Film(FILM), S44, P8, adaptive=D.Adaptive(1, 1, 0.1))
    with pytest.raises(ValueError):
        rn.render_progressive(None, None, api.Film(acc), S44, P8, adaptive=ok)


def test_headless_adaptive_arguments():
    a = headless.parse_args(["--out", "x.exr", "--adaptive", "0.05", "--adaptive-abs", "0.001", "--adaptive-min", "8",
                             "--adaptive-step", "4", "--sample-counts", "n.exr"])
    assert headless.adaptive_from_args(a) == D.Adaptive(8, 4, 0.05, 0.001) and a.sample_counts == "n.exr"
    b = headless.parse_args(["--out", "x.exr", "--adaptive", "0.1"])
    assert headless.adaptive_from_args(b) == D.Adaptive(16, 16, 0.1, 0.0) and b.sample_counts is None
    assert headless.adaptive_from_args(headless.parse_args(["--out", "x.exr"])) is None
    with pytest.raises(SystemExit):
        headless.parse_args(["--out", "x.exr", "--sample-counts", "n.exr"])


CASES = [(s, i, m, k) for s in SCENE_IDS for i in ("path-8", "whitted-5") for m in ("stratified-4x4", "uniform-16") for k in SETTINGS]
INTEG = {"path-8": P8, "whitted-5": W5}
SAMPLER = {"stratified-4x4": S44, "uniform-16": U16}


@pytest.mark.parametrize("scene_id,integ_id,smp_id,setting", CASES)
def test_oracle_counts_are_a_real_mix(oracle, xf, scene_id, integ_id, smp_id, setting):
    """The GPU case of the same parameters tests what it claims: pixels at min_samples, in between, and at spp."""
    scene, cam = _scenes(xf)[scene_id]()
    a = SETTINGS[setting]
    c = adaptive_counts(_per_sample_films(oracle, scene, cam, FILM, SAMPLER[smp_id], INTEG[integ_id]), a)
    spp = SAMPLER[smp_id].samples_per_pixel()
    assert int((c == a.min_samples).sum()) >= MIN_PIXELS
    assert int(((c > a.min_samples) & (c < spp)).sum()) >= MIN_PIXELS
    assert int((c == spp).sum()) >= MIN_PIXELS


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


def _render(ctx, dev, cam, film, smp, integ, **kw):
    return api.Renderer(ctx).render(dev, cam, film, smp, integ, **kw)


def _assert_same(r, ref, what=""):
    """Film, counts, companion films, hit ids and every counter of `r` equal those of `ref`."""
    assert np.array_equal(_bits(r.film), _bits(ref.film)), what
    assert np.array_equal(r.sample_counts, ref.sample_counts), what
    for n in ref.aovs:
        assert np.array_equal(_bits(r.aovs[n]), _bits(ref.aovs[n])), (what, n)
    if ref.hit_ids is not None:
        assert np.array_equal(r.hit_ids, ref.hit_ids), what
    for k in STATS:
        assert getattr(r.stats, k) == getattr(ref.stats, k), (what, k)


@pytest.mark.gpu
@pytest.mark.parametrize("scene_id,integ_id,smp_id,setting", CASES)
def test_counts_film_and_views_equal_the_oracle(gpu_ctx, scene_cache, oracle, scene_id, integ_id, smp_id, setting):
    scene, cam, dev = scene_cache(scene_id)
    smp, integ, a = SAMPLER[smp_id], INTEG[integ_id], SETTINGS[setting]
    lis = _per_sample_films(oracle, scene, cam, FILM, smp, integ)
    want = adaptive_counts(lis, a)
    r = _render(gpu_ctx, dev, cam, FILM, smp, integ, adaptive=a, aovs=ALL)
    assert r.sample_counts.shape == (16, 24) and r.sample_counts.dtype == np.uint32
    assert np.array_equal(r.sample_counts, want)
    assert r.stats.samples == int(want.sum())
    assert np.array_equal(_bits(r.film), _bits(sums_over_counts(lis, want)))
    assert np.array_equal(_bits(r.aovs["radiance_sq"]), _bits(sums_over_counts(lis, want, square=True)))
    osc = oracle.OracleScene(scene)
    for name in VIEWS:
        views = _per_sample_films(oracle, scene, cam, FILM, smp, _debug_integrator(name))
        assert np.array_equal(_bits(r.aovs[name]), _bits(sums_over_counts(views, want))), name
    # the second route: the oracle traces exactly the (pixel, sample) pairs the counts name
    acc = D.FilmSettings(tuple(FILM.res), FILM.tile_dim, accumulate=True)
    o_img, _, o_st = osc.render(cam, acc, smp, integ, tiles=traced_tiles(want), threads=1)
    assert np.array_equal(_bits(o_img / want[:, :, None].astype(np.float32)), _bits(r.film))
    for k in STATS:
        assert getattr(r.stats, k) == getattr(o_st, k), k
    # without the companion films: the same film, counts and counters
    _assert_same(r, _render(gpu_ctx, dev, cam, FILM, smp, integ, adaptive=a))


@pytest.mark.gpu
def test_independent_of_the_batch_shape(gpu_ctx, scene_cache, monkeypatch):
    """Batch samples 1 / 3 / 7, 200-path batches, one or two pipes and the ray sorts all give the same bits."""
    scene, cam, dev = scene_cache("material-room")
    a = SETTINGS["min2-step3-rel0.15-abs0.01"]
    for integ in (P8, W5):
        ref = _render(gpu_ctx, dev, cam, FILM, S44, integ, adaptive=a, aovs=["radiance_sq"], want_hit_ids=True, pipes=1)
        assert len(np.unique(ref.sample_counts)) >= 3
        runs = [dict(pipes=2), dict(wavefront_paths=200), dict(wavefront_paths=200, pipes=2), dict(wavefront_paths=1000, pipes=2)]
        if integ is P8:
            runs += [dict(ray_sort=1), dict(ray_sort=2), dict(ray_sort=3)]
        for kw in runs:
            _assert_same(_render(gpu_ctx, dev, cam, FILM, S44, integ, adaptive=a, aovs=["radiance_sq"], want_hit_ids=True, **kw), ref, kw)
        for mb in ("1", "3", "7"):
            monkeypatch.setenv("YK_MAX_BATCH_SAMPLES", mb)
            for kw in (dict(pipes=1), dict(pipes=2, wavefront_paths=300)):
                _assert_same(_render(gpu_ctx, dev, cam, FILM, S44, integ, adaptive=a, aovs=["radiance_sq"], want_hit_ids=True, **kw),
                             ref, (mb, kw))
            monkeypatch.delenv("YK_MAX_BATCH_SAMPLES")


@pytest.mark.gpu
def test_independent_of_the_shadow_mode(gpu_ctx, xf):
    scene, cam = _scenes(xf)["leaves-40"]()
    scene.lights.append(D.Light(D.LIGHT_POINT, xf.translation((2.0, 3.0, -1.0)), (100.0, 100.0, 100.0)))
    a = SETTINGS["min4-step4-rel0.2"]
    ctxs = {}
    try:
        with pytest.MonkeyPatch.context() as mp:
            for mode in ("0", "1"):
                mp.setenv("YK_SHADOW_MODE", mode)
                ctxs[mode] = api.Context(0)
        res = {}
        for mode, ctx in ctxs.items():
            d = api.Scene(ctx, scene)
            res[mode] = _render(ctx, d, cam, FILM, S44, P8, adaptive=a, want_hit_ids=True, pipes=2, wavefront_paths=500)
            d.close()
        _assert_same(res["1"], res["0"])
        assert len(np.unique(res["0"].sample_counts)) >= 2
    finally:
        for c in ctxs.values():
            c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("integ", [P8, W5], ids=["path-8", "whitted-5"])
def test_min_samples_at_spp_is_the_plain_render(gpu_ctx, scene_cache, integ):
    scene, cam, dev = scene_cache("glass-cornell-rect")
    plain = _render(gpu_ctx, dev, cam, FILM, S44, integ, want_hit_ids=True, aovs=ALL)
    for a in (D.Adaptive(16, 1, 0.0, 0.0), D.Adaptive(40, 7, 1.0, 1.0)):
        r = _render(gpu_ctx, dev, cam, FILM, S44, integ, want_hit_ids=True, aovs=ALL, adaptive=a)
        assert (r.sample_counts == 16).all()
        assert np.array_equal(_bits(r.film), _bits(plain.film)) and np.array_equal(r.hit_ids, plain.hit_ids)
        for n in ALL:
            assert np.array_equal(_bits(r.aovs[n]), _bits(plain.aovs[n])), n
        for k in STATS:
            assert getattr(r.stats, k) == getattr(plain.stats, k), k


@pytest.mark.gpu
def test_more_than_1024_spp(gpu_ctx, scene_cache, oracle):
    """Checks at 600 and 900 of 1100 samples: the first lies inside what would be one 1024-sample batch."""
    scene, cam, dev = scene_cache("glass-cornell-rect")
    film = D.FilmSettings((8, 4), 8)
    smp, a = D.SamplerType.uniform(1100), D.Adaptive(600, 300, 0.08, 0.0)
    lis = _per_sample_films(oracle, scene, cam, film, smp, P8)
    want = adaptive_counts(lis, a)
    assert set(np.unique(want)) == {600, 900, 1100}
    r = _render(gpu_ctx, dev, cam, film, smp, P8, adaptive=a, aovs=["radiance_sq"])
    assert np.array_equal(r.sample_counts, want) and r.stats.samples == int(want.sum())
    assert np.array_equal(_bits(r.film), _bits(sums_over_counts(lis, want)))
    assert np.array_equal(_bits(r.aovs["radiance_sq"]), _bits(sums_over_counts(lis, want, square=True)))
    _assert_same(_render(gpu_ctx, dev, cam, film, smp, P8, adaptive=a, aovs=["radiance_sq"], wavefront_paths=200, pipes=2), r)


@pytest.mark.gpu
def test_partial_tiles_device_buffers_and_hit_ids(gpu_ctx, scene_cache):
    import torch
    scene, cam, dev = scene_cache("sphere-field")
    a = SETTINGS["min4-step4-rel0.2"]
    full = _render(gpu_ctx, dev, cam, FILM, S44, P8, adaptive=a, want_hit_ids=True, aux_sample=9)
    # hit ids of sample 9: -1 where the pixel stopped at 4 or 8, the plain render's id elsewhere
    plain = _render(gpu_ctx, dev, cam, FILM, S44, P8, want_hit_ids=True, aux_sample=9)
    early = full.sample_counts <= 9
    assert early.any() and (~early).any()
    assert (full.hit_ids[early] == -1).all() and np.array_equal(full.hit_ids[~early], plain.hit_ids[~early])
    assert (plain.hit_ids[early] >= 0).any()
    tiles = api.film_tiles(FILM)
    tiles = tiles[: len(tiles) // 2]
    inside = np.zeros((16, 24), bool)
    for t in tiles:
        inside[t["y0"]:t["y1"], t["x0"]:t["x1"]] = True
    assert inside.any() and not inside.all()
    sentinel = np.float32(-7.25)
    counts = np.full((16, 24), 12345, np.uint32)
    r = _render(gpu_ctx, dev, cam, FILM, S44, P8, tiles=tiles, adaptive=a, film_out=np.full((16, 24, 3), sentinel, np.float32),
                sample_counts_out=counts)
    assert r.sample_counts is counts
    assert (counts[~inside] == 12345).all() and np.array_equal(counts[inside], full.sample_counts[inside])
    assert (r.film[~inside] == sentinel).all() and np.array_equal(_bits(r.film[inside]), _bits(full.film[inside]))
    assert r.stats.samples == int(full.sample_counts[inside].sum())
    film_t = torch.full((16, 24, 3), float(sentinel), dtype=torch.float32, device="cuda")
    counts_t = torch.full((16, 24), 12345, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    rd = _render(gpu_ctx, dev, cam, FILM, S44, P8, tiles=tiles, adaptive=a, device_film_ptr=film_t.data_ptr(),
                 sample_counts_out=counts_t.data_ptr())
    assert rd.sample_counts == counts_t.data_ptr()
    assert np.array_equal(_bits(film_t.cpu().numpy()), _bits(r.film))
    assert np.array_equal(counts_t.cpu().numpy().view(np.uint32), counts)
    # device film without counts
    film_t.zero_()
    torch.cuda.synchronize()
    rd = _render(gpu_ctx, dev, cam, FILM, S44, P8, adaptive=a, device_film_ptr=film_t.data_ptr())
    assert rd.sample_counts is None and np.array_equal(_bits(film_t.cpu().numpy()), _bits(full.film))


@pytest.mark.gpu
def test_progress_reports_the_maximum_then_the_total(gpu_ctx, scene_cache):
    scene, cam, dev = scene_cache("glass-cornell-rect")
    calls = []
    r = _render(gpu_ctx, dev, cam, FILM, S44, P8, adaptive=SETTINGS["min4-step4-rel0.2"], wavefront_paths=400,
                progress=lambda done, total: calls.append((done, total)) and False)
    total = int(r.sample_counts.sum())
    assert total < 16 * 24 * 16 and r.stats.samples == total
    assert calls[-1] == (total, total)
    assert len(calls) > 2 and all(t == 16 * 24 * 16 and d <= total for d, t in calls[:-1])


@pytest.mark.gpu
def test_refusals_leave_the_context_usable(gpu_ctx, scene_cache):
    scene, cam, dev = scene_cache("glass-cornell-rect")
    film = D.FilmSettings((16, 8), 8)
    a = D.Adaptive(4, 4, 0.2, 0.0)
    ref = _render(gpu_ctx, dev, cam, film, S44, P8, adaptive=a)
    L = capi.lib()
    cam_c = api.make_camera(cam, film)
    sm = capi.sampler(S44)
    img = np.zeros((8, 16, 3), np.float32)
    counts = np.full((8, 16), 77, np.uint32)

    def call(integ, opts, fsd=film):
        fs = capi.film_settings(fsd)
        tiles = api.film_tiles(fsd)
        ig = capi.integrator(integ)
        stats = capi.Stats()
        return L.yk_render(gpu_ctx._h, dev._h, C.byref(cam_c), C.byref(fs), C.byref(sm), C.byref(ig), C.c_void_p(tiles.ctypes.data),
                           len(tiles), C.byref(opts), C.c_void_p(img.ctypes.data), C.byref(stats))

    opts = capi.RenderOpts()
    opts.flags = capi.RENDER_ADAPTIVE   # adaptive NULL
    assert call(P8, opts) == -1 and b"adaptive" in L.yk_last_error()
    for bad in [(1, 4, 0.1, 0.0), (4, 0, 0.1, 0.0), (4, 4, -0.1, 0.0), (4, 4, 0.1, -0.5), (4, 4, float("nan"), 0.0), (4, 4, 0.1, float("inf"))]:
        ad = capi.Adaptive(*bad)
        ad.sample_counts = counts.ctypes.data
        opts.adaptive = C.pointer(ad)
        assert call(P8, opts) == -1, bad
    ad = capi.Adaptive(4, 4, 0.2, 0.0)
    ad.sample_counts = counts.ctypes.data
    opts.adaptive = C.pointer(ad)
    assert call(P8, opts, D.FilmSettings((16, 8), 8, accumulate=True)) == -1
    for integ in [_debug_integrator(n) for n in VIEWS]:
        assert call(integ, opts) == -1, integ
    assert (counts == 77).all() and not img.any()   # nothing launched, nothing written
    mctx = api.MultiContext([0])
    try:
        ms = api.MultiScene(mctx, scene)
        ig = capi.integrator(P8)
        fs, tiles = capi.film_settings(film), api.film_tiles(film)
        stats, per = capi.Stats(), (capi.Stats * 1)()
        rc = L.yk_multi_render(mctx._h, ms._h, C.byref(cam_c), C.byref(fs), C.byref(sm), C.byref(ig), C.c_void_p(tiles.ctypes.data),
                               len(tiles), C.byref(opts), C.c_void_p(img.ctypes.data), C.byref(stats), per)
        assert rc == -1 and b"yk_multi_render" in L.yk_last_error()
        ms.close()
    finally:
        mctx.close()
    assert (counts == 77).all() and not img.any()
    assert call(P8, opts) == 0 and np.array_equal(_bits(img), _bits(ref.film)) and np.array_equal(counts, ref.sample_counts)


@pytest.mark.gpu
def test_headless_writes_the_sample_counts(tmp_path):
    import io
    from oracle import post
    out, cnt = tmp_path / "box.exr", tmp_path / "counts.exr"
    argv = ["--out", str(out), "--integrator", "path", "--max-depth", "8", "--sampler", "stratified", "4", "4", "--res", "48", "32",
            "--tone-map", "raw", "--adaptive", "0.2", "--adaptive-min", "4", "--adaptive-step", "4", "--sample-counts", str(cnt)]
    log = io.StringIO()
    headless.render(headless.parse_args(argv), out=log)
    scene, cam, _ = headless.try_load_scene("")
    ctx = api.Context(0)
    dev = api.Scene(ctx, scene)
    try:
        r = _render(ctx, dev, cam, D.FilmSettings((48, 32), 16), S44, P8, adaptive=D.Adaptive(4, 4, 0.2, 0.0))
    finally:
        dev.close()
        ctx.close()
    assert np.array_equal(_bits(post.read_exr_rgb(str(out))), _bits(r.film))
    c = post.read_exr_rgb(str(cnt))
    assert np.array_equal(c, np.repeat(r.sample_counts.astype(np.float32)[:, :, None], 3, axis=2))
    assert f"wrote sample counts to {cnt}" in log.getvalue()
