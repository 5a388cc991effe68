"""Denoising a render's film (`yk_denoise`, `api.denoise`, `headless --denoise`): the edge-avoiding a-trous filter guided by
the render's own variance (`radiance_sq` and the sample counts) and, optionally, a normal companion film.

The rule uses only un-fused float32 + - * /, sqrtf and comparisons in a fixed order, so every GPU test compares bits with
the numpy restatement `denoise_reference.denoise`. The CPU tests check the restatement itself: its quality on the Cornell box
against a 4096-spp reference, edges kept by the normal guide, and a constant film coming back as itself.
"""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import denoise_reference as ref_denoise
from oracle import post
from yuki_b200 import api, capi, desc as D, headless, scenes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_REF = os.path.join(ROOT, "tests", "golden", "denoise_cornell_4096spp.npz")
ERR_INVALID = -1   # YK_ERR_INVALID
S44, U16 = D.SamplerType.stratified(4, 4), D.SamplerType.uniform(16)
P8, W5 = D.IntegratorType.path(8), D.IntegratorType.whitted(5)
FILM = D.FilmSettings((40, 24), 8)
VIEWS = ["radiance_sq", "geometry_normals", "shading_normals"]


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _same_bits(a, b):
    """Equal bit patterns, except that any NaN equals any NaN."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    both_nan = np.isnan(a) & np.isnan(b)
    return bool(np.array_equal(np.where(both_nan, 0, _bits(a)), np.where(both_nan, 0, _bits(b))))


def _noisy_film(h, w, seed, spp=16):
    """A seeded film with plausible statistics: mean, mean of squares and a normal film with two facing directions."""
    rng = np.random.default_rng(seed)
    film = rng.gamma(2.0, 0.5, (h, w, 3)).astype(np.float32)
    sq = (film * film + rng.gamma(1.0, 0.3, (h, w, 3)).astype(np.float32)).astype(np.float32)
    nrm = np.where((np.arange(w) < w // 2)[None, :, None], np.float32([0.5, 0.5, 1.0]), np.float32([1.0, 0.5, 0.5]))
    nrm = np.broadcast_to(nrm, (h, w, 3)).astype(np.float32)
    return film, sq, nrm


# ---- CPU: parameters, argument checks, ABI layout ----------------------------------------------------------------------
def test_denoise_settings_are_validated_on_construction():
    d = D.Denoise()
    assert (d.iterations, d.sigma, d.eps) == (5, 2.0, 1e-4)
    D.Denoise(1, 0.5, 1e-6)
    D.Denoise(10)
    for bad in [dict(iterations=0), dict(iterations=11), dict(iterations=2.5), dict(iterations=True), dict(sigma=0.0),
                dict(sigma=-1.0), dict(sigma=float("inf")), dict(sigma=float("nan")), dict(sigma=1e39), dict(eps=0.0),
                dict(eps=1e-50), dict(eps=float("nan"))]:
        with pytest.raises(ValueError):
            D.Denoise(**bad)


def test_bad_arguments_raise_before_the_library():
    film, sq, nrm = _noisy_film(6, 5, 0)
    for kw in [dict(), dict(spp=1), dict(spp=4, normals=nrm[:, :4]), dict(spp=4, out=np.zeros((5, 6, 3), np.float32)),
               dict(sample_counts=np.zeros((6, 4), np.uint32)), dict(spp=4, params=(5, 2.0, 1e-4)),
               dict(spp=4, out=np.zeros((6, 5, 3), np.float64))]:
        with pytest.raises(ValueError):
            api.denoise(None, film, sq, **kw)   # no context: these must fail before anything reaches the library
    with pytest.raises(ValueError):
        api.denoise(None, film, sq[:, :, :2], spp=4)
    with pytest.raises(ValueError):
        api.denoise(None, film[:, :, 0], sq[:, :, 0], spp=4)


def test_headless_denoise_arguments():
    a = headless.parse_args(["--out", "x.exr", "--integrator", "path", "--sampler", "uniform", "4", "--denoise",
                             "--denoise-sigma", "3", "--denoise-iterations", "4"])
    assert headless.denoise_from_args(a) == D.Denoise(4, 3.0)
    assert headless.denoise_from_args(headless.parse_args(["--out", "x.exr"])) is None
    assert headless.denoise_from_args(headless.parse_args(["--out", "x.exr", "--sampler", "uniform", "4", "--denoise"])) == D.Denoise()
    for bad in (["--integrator", "shading-normals", "--sampler", "uniform", "4", "--denoise"],
                ["--integrator", "bvh-intersections", "--sampler", "uniform", "4", "--denoise"],
                ["--sampler", "uniform", "1", "--denoise"],
                ["--sampler", "uniform", "4", "--denoise", "--denoise-iterations", "11"],
                ["--sampler", "uniform", "4", "--denoise", "--denoise-sigma", "0"]):
        with pytest.raises(SystemExit):
            headless.parse_args(["--out", "x.exr"] + bad)


LAYOUT_C = r"""
#include <stddef.h>
#include <stdio.h>
#include "yuki_gpu.h"
int main(void) {
    printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(yk_denoise_params), offsetof(yk_denoise_params, flags),
           offsetof(yk_denoise_params, iterations), offsetof(yk_denoise_params, sigma), offsetof(yk_denoise_params, eps),
           offsetof(yk_denoise_params, samples_per_pixel), offsetof(yk_denoise_params, _reserved),
           offsetof(yk_denoise_params, sample_counts), offsetof(yk_denoise_params, normals), offsetof(yk_denoise_params, stream));
    printf("%u\n", (unsigned)YK_DENOISE_ON_DEVICE);
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
    P = capi.DenoiseParams
    assert [int(v) for v in lines[0].split()] == [C.sizeof(P)] + [getattr(P, n).offset for n, _ in P._fields_]
    assert int(lines[1]) == capi.DENOISE_ON_DEVICE


# ---- CPU: the restatement ------------------------------------------------------------------------------------------------
QUALITY_RES, QUALITY_INTEG = (128, 96), D.IntegratorType.path(10, indirect_clamp=2.0)


def _quality_scene(xf):
    return scenes.cornell(xf, light="rect", tall_box="glass", sphere=True, split_method=D.SPLIT_MIDDLE)


def _sample_sums(oracle, scene, cam, film, smp, integ, threads=8):
    """The float32 mean and mean of li * li over the samples in ascending order, from the oracle's per-sample films: what a
    render's film and radiance_sq companion film hold."""
    acc = D.FilmSettings(tuple(film.res), film.tile_dim, accumulate=True)
    base = api.film_tiles(acc)
    osc = oracle.OracleScene(scene)
    s = q = np.zeros((film.res[1], film.res[0], 3), np.float32)
    for k in range(smp.samples_per_pixel()):
        t = base.copy()
        t["sample"] = k
        li = osc.render(cam, acc, smp, integ, tiles=t, film_out=np.zeros_like(s), threads=threads)[0]
        s, q = s + li, q + li * li
    n = np.float32(smp.samples_per_pixel())
    return s / n, q / n


def make_golden(xf, oracle):
    """The 4096-spp oracle render of the quality test's scene (tests/golden/make_denoise_golden.py)."""
    scene, cam = _quality_scene(xf)
    ref = oracle.OracleScene(scene).render(cam, D.FilmSettings(QUALITY_RES, 16), D.SamplerType.uniform(4096), QUALITY_INTEG, threads=8)[0]
    np.savez_compressed(GOLDEN_REF, ref=ref)


def test_denoised_16spp_film_is_as_close_as_64spp(xf, oracle):
    scene, cam = _quality_scene(xf)
    film = D.FilmSettings(QUALITY_RES, 16)
    mean, sq = _sample_sums(oracle, scene, cam, film, D.SamplerType.uniform(16), QUALITY_INTEG)
    osc = oracle.OracleScene(scene)
    assert _same_bits(mean, osc.render(cam, film, D.SamplerType.uniform(16), QUALITY_INTEG, threads=8)[0])
    nrm = osc.render(cam, film, D.SamplerType.uniform(16), D.IntegratorType.debug(D.INTEGRATOR_SHADING_NORMALS), threads=8)[0]
    raw64 = osc.render(cam, film, D.SamplerType.uniform(64), QUALITY_INTEG, threads=8)[0]
    ref = np.load(GOLDEN_REF)["ref"].astype(np.float64)
    guided = ref_denoise.denoise(mean, sq, spp=16, normals=nrm)
    plain = ref_denoise.denoise(mean, sq, spp=16)

    def mae(a):
        return float(np.mean(np.abs(a.astype(np.float64) - ref)))

    def tm_rmse(a):
        a = a.astype(np.float64)
        return float(np.sqrt(np.mean((a / (1 + a) - ref / (1 + ref)) ** 2)))
    assert mae(guided) <= 0.6 * mae(mean), (mae(guided), mae(mean))
    assert mae(guided) <= 1.1 * mae(raw64), (mae(guided), mae(raw64))
    assert tm_rmse(guided) <= 0.75 * tm_rmse(plain), (tm_rmse(guided), tm_rmse(plain))


def test_the_normal_guide_keeps_an_edge_the_unguided_filter_blurs():
    """Two planes facing different ways, colours 0.5 and 0.8, with seeded noise whose spread matches the variance the
    film's statistics give (per-sample variance 0.36 at 16 spp)."""
    h, w = 32, 32
    rng = np.random.default_rng(3)
    left = np.arange(w) < w // 2
    clean = np.broadcast_to(np.where(left[None, :, None], np.float32(0.5), np.float32(0.8)), (h, w, 3)).astype(np.float32)
    film = (clean + rng.normal(0.0, 0.15, (h, w, 3)).astype(np.float32)).astype(np.float32)
    sq = (film * film + np.float32(0.36)).astype(np.float32)
    nrm = np.where(left[None, :, None], np.float32([0.5, 0.5, 1.0]), np.float32([1.0, 0.5, 0.5]))
    nrm = np.broadcast_to(nrm, (h, w, 3)).astype(np.float32)
    guided = ref_denoise.denoise(film, sq, spp=16, normals=nrm)
    plain = ref_denoise.denoise(film, sq, spp=16)

    def edge(a):   # the mean of the two columns either side of the edge
        return float(a[:, w // 2 - 1].mean()), float(a[:, w // 2].mean())
    gl, gr = edge(guided)
    pl, pr = edge(plain)
    assert abs(gl - 0.5) < 0.03 and abs(gr - 0.8) < 0.03 and gr - gl > 0.27, (gl, gr)
    assert pr - pl < 0.22, (pl, pr)
    for out in (guided, plain):   # both remove noise inside the planes
        assert np.std(out[:, 2:8]) < 0.3 * np.std(film[:, 2:8])


def test_a_constant_film_comes_back_as_itself():
    c = np.broadcast_to(np.float32([0.75, 1.25, 3.0]), (21, 17, 3)).astype(np.float32)
    sq = (c * c + np.float32(0.01)).astype(np.float32)
    nrm = np.full((21, 17, 3), 0.5, np.float32)
    nrm[..., 2] = 1.0
    for normals in (None, nrm):
        out = ref_denoise.denoise(c, sq, spp=8, normals=normals, iterations=5)
        np.testing.assert_allclose(out, c, rtol=4 * np.finfo(np.float32).eps, atol=0)


def test_restatement_keeps_nan_and_inf_to_their_own_pixel_and_copies_pixels_without_two_samples():
    film, sq, nrm = _noisy_film(23, 37, 4)
    film[5, 7] = np.nan
    film[11, 20, 1] = np.inf
    sq[17, 3, 2] = np.nan
    counts = np.full((23, 37), 16, np.uint32)
    counts[:, 30:] = 0
    counts[2, 2] = 1
    out = ref_denoise.denoise(film, sq, sample_counts=counts, normals=nrm, iterations=4)
    bad = np.zeros((23, 37), bool)
    bad[5, 7] = bad[11, 20] = True
    assert np.isnan(out[5, 7]).all() and not np.isfinite(out[11, 20]).all()
    assert np.isfinite(out[~bad]).all()
    assert _same_bits(out[:, 30:], film[:, 30:]) and _same_bits(out[2, 2], film[2, 2])


# ---- GPU ---------------------------------------------------------------------------------------------------------------------
def _device_denoise(ctx, film, sq, **kw):
    """api.denoise on host arrays, checked bit for bit against the restatement with the same arguments."""
    params = kw.pop("params", D.Denoise())
    out = api.denoise(ctx, film, sq, params=params, **kw)
    ref = ref_denoise.denoise(film, sq, spp=kw.get("spp"), sample_counts=kw.get("sample_counts"), normals=kw.get("normals"),
                       iterations=params.iterations, sigma=params.sigma, eps=params.eps)
    assert out.shape == film.shape and out.dtype == np.float32
    assert _same_bits(out, ref), float(np.nanmax(np.abs(out.astype(np.float64) - ref)))
    return out


@pytest.fixture(scope="module")
def renders(gpu_ctx, xf):
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass", sphere=True, split_method=D.SPLIT_MIDDLE)
    dev = api.Scene(gpu_ctx, scene)
    made = {}

    def get(integ, smp):
        key = (integ.kind, smp.kind)
        if key not in made:
            made[key] = api.Renderer(gpu_ctx).render(dev, cam, FILM, smp, integ, aovs=VIEWS)
        return made[key]
    yield get
    dev.close()


SETTINGS = [D.Denoise(), D.Denoise(3, 0.5, 1e-2)]


@pytest.mark.gpu
@pytest.mark.parametrize("settings", SETTINGS, ids=["defaults", "sigma0.5-eps1e-2-k3"])
@pytest.mark.parametrize("guide", [None, "geometry_normals", "shading_normals"])
@pytest.mark.parametrize("smp", [S44, U16], ids=["stratified-4x4", "uniform-16"])
@pytest.mark.parametrize("integ", [P8, W5], ids=["path-8", "whitted-5"])
def test_rendered_films_match_the_restatement(gpu_ctx, renders, integ, smp, guide, settings):
    r = renders(integ, smp)
    normals = None if guide is None else r.aovs[guide]
    out = _device_denoise(gpu_ctx, r.film, r.aovs["radiance_sq"], spp=16, normals=normals, params=settings)
    assert not np.array_equal(out, r.film) and np.isfinite(out).all()


@pytest.mark.gpu
@pytest.mark.parametrize("iterations", [1, 3, 5, 10])
def test_iterations_including_steps_past_the_film(gpu_ctx, renders, iterations):
    r = renders(P8, U16)
    for normals in (None, r.aovs["shading_normals"]):
        _device_denoise(gpu_ctx, r.film, r.aovs["radiance_sq"], spp=16, normals=normals, params=D.Denoise(iterations))


@pytest.mark.gpu
@pytest.mark.parametrize("partial", [False, True], ids=["all-tiles", "partial-tiles"])
def test_adaptive_render_with_its_sample_counts(gpu_ctx, xf, partial):
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    dev = api.Scene(gpu_ctx, scene)
    tiles = api.film_tiles(FILM)
    if partial:
        tiles = tiles[: len(tiles) // 2]
    counts = np.zeros((24, 40), np.uint32)   # pixels outside the tiles keep count 0: copied through, never a tap
    r = api.Renderer(gpu_ctx).render(dev, cam, FILM, D.SamplerType.uniform(64), P8, tiles=tiles, aovs=VIEWS,
                                     adaptive=D.Adaptive(4, 4, 0.1), sample_counts_out=counts)
    dev.close()
    assert len(np.unique(counts[counts > 0])) > 2 and ((counts == 0).any() == partial)
    for normals in (None, r.aovs["shading_normals"]):
        out = _device_denoise(gpu_ctx, r.film, r.aovs["radiance_sq"], sample_counts=counts, normals=normals)
        assert _same_bits(out[counts < 2], r.film[counts < 2])
    # sample_counts take precedence over spp
    out = api.denoise(gpu_ctx, r.film, r.aovs["radiance_sq"], spp=64, sample_counts=counts)
    assert _same_bits(out, ref_denoise.denoise(r.film, r.aovs["radiance_sq"], sample_counts=counts))


@pytest.mark.gpu
@pytest.mark.parametrize("hw", [(1, 1), (1, 37), (37, 23), (23, 37), (1080, 1920)], ids=lambda s: f"{s[1]}x{s[0]}")
def test_film_sizes(gpu_ctx, hw):
    h, w = hw
    film, sq, nrm = _noisy_film(h, w, h * 1000 + w)
    k = 2 if h * w > 100000 else 5   # (the numpy restatement takes ~3 s per iteration at 1080p)
    _device_denoise(gpu_ctx, film, sq, spp=16, normals=nrm, params=D.Denoise(k))
    if h * w <= 100000:
        _device_denoise(gpu_ctx, film, sq, spp=3, params=D.Denoise(k))


@pytest.mark.gpu
def test_nan_and_inf_pixels_do_not_spread(gpu_ctx, renders):
    r = renders(P8, U16)
    film, sq = r.film.copy(), r.aovs["radiance_sq"].copy()
    film[5, 7] = np.nan
    film[11, 20, 1] = np.inf
    film[3, 30, 0] = -np.inf
    sq[17, 3, 2] = np.nan
    sq[20, 35, 0] = np.inf
    bad = np.zeros((24, 40), bool)
    bad[5, 7] = bad[11, 20] = bad[3, 30] = True
    for normals in (None, r.aovs["shading_normals"]):
        out = _device_denoise(gpu_ctx, film, sq, spp=16, normals=normals, params=D.Denoise(4))
        assert np.isnan(out[5, 7]).all()
        assert np.isfinite(out[~bad]).all()


@pytest.mark.gpu
def test_output_may_be_the_film(gpu_ctx, renders):
    r = renders(W5, S44)
    film = r.film.copy()
    ref = ref_denoise.denoise(film, r.aovs["radiance_sq"], spp=16, normals=r.aovs["geometry_normals"])
    got = api.denoise(gpu_ctx, film, r.aovs["radiance_sq"], spp=16, normals=r.aovs["geometry_normals"], out=film)
    assert got is film and _same_bits(film, ref)


@pytest.mark.gpu
def test_torch_tensors_after_a_long_op_on_the_callers_stream(gpu_ctx, renders):
    torch = pytest.importorskip("torch")
    r = renders(P8, S44)
    dev = torch.device("cuda", gpu_ctx.device_id)
    src = {k: torch.from_numpy(v).to(dev) for k, v in (("film", r.film), ("sq", r.aovs["radiance_sq"]),
                                                      ("nrm", r.aovs["shading_normals"]))}
    counts = np.full((24, 40), 16, np.uint32)
    counts[:3] = 1
    counts_t = torch.from_numpy(counts.view(np.int32)).to(dev)
    side = torch.cuda.Stream(dev)
    torch.cuda.synchronize(dev)
    with torch.cuda.stream(side):
        film, sq, nrm = (torch.zeros_like(src[k]) for k in ("film", "sq", "nrm"))
        torch.cuda._sleep(200_000_000)   # a long op queued before the inputs are written on the caller's stream
        film.copy_(src["film"])
        sq.copy_(src["sq"])
        nrm.copy_(src["nrm"])
        out = api.denoise(gpu_ctx, film, sq, sample_counts=counts_t, normals=nrm)
        assert isinstance(out, torch.Tensor) and out.device == dev and out.dtype == torch.float32
        got = out.cpu().numpy()
        # in place on the film tensor
        out2 = api.denoise(gpu_ctx, film, sq, sample_counts=counts_t, normals=nrm, out=film)
        assert out2 is film
        got2 = film.cpu().numpy()
    ref = ref_denoise.denoise(r.film, r.aovs["radiance_sq"], sample_counts=counts, normals=r.aovs["shading_normals"])
    assert _same_bits(got, ref) and _same_bits(got2, ref)
    with pytest.raises(ValueError, match="mixes"):
        api.denoise(gpu_ctx, src["film"], r.aovs["radiance_sq"], spp=16)
    with pytest.raises(ValueError):
        api.denoise(gpu_ctx, src["film"], src["sq"].double(), spp=16)


@pytest.mark.gpu
def test_every_refusal_leaves_the_context_usable(gpu_ctx, renders):
    r = renders(P8, U16)
    film, sq = np.ascontiguousarray(r.film), np.ascontiguousarray(r.aovs["radiance_sq"])
    out = np.full_like(film, 7.0)
    L = capi.lib()

    def call(prm, h=24, w=40, f=film, s=sq, o=out, ctx=gpu_ctx._h):
        return L.yk_denoise(ctx, w, h, None if f is None else f.ctypes.data, None if s is None else s.ctypes.data,
                            None if prm is None else C.byref(prm), None if o is None else o.ctypes.data)

    def prm(**kw):
        p = capi.DenoiseParams(0, 5, 2.0, 1e-4, 16, 0)
        for k, v in kw.items():
            setattr(p, k, v)
        return p
    bad = [call(prm(), ctx=None), call(prm(), f=None), call(prm(), s=None), call(prm(), o=None), call(None),
           call(prm(), h=0), call(prm(), w=0), call(prm(iterations=0)), call(prm(iterations=11)),
           call(prm(sigma=0.0)), call(prm(sigma=-2.0)), call(prm(sigma=float("inf"))), call(prm(sigma=float("nan"))),
           call(prm(eps=0.0)), call(prm(eps=float("inf"))), call(prm(eps=float("nan"))), call(prm(samples_per_pixel=1)),
           call(prm(samples_per_pixel=0)), call(prm(flags=2))]
    assert bad == [ERR_INVALID] * len(bad)
    assert (out == 7.0).all()   # nothing was written
    # device flag with host arrays: refused before anything is launched
    assert call(prm(flags=capi.DENOISE_ON_DEVICE)) == ERR_INVALID
    assert "device memory" in L.yk_last_error().decode()
    assert call(prm()) == 0
    assert _same_bits(out, ref_denoise.denoise(film, sq, spp=16))


@pytest.mark.gpu
@pytest.mark.parametrize("adaptive", [False, True], ids=["uniform", "adaptive"])
def test_headless_denoise(tmp_path, xf, gpu_ctx, adaptive):
    out, rsq, nrm, cnt = (tmp_path / f"{n}.exr" for n in ("out", "rsq", "nrm", "cnt"))
    extra = ["--adaptive", "0.1", "--adaptive-min", "4", "--adaptive-step", "4", "--sample-counts", str(cnt)] if adaptive else []
    argv = ["--out", str(out), "--integrator", "path", "--max-depth", "5", "--sampler", "uniform", "16", "--res", "48", "32",
            "--tone-map", "raw", "--denoise", "--denoise-sigma", "1.5", "--denoise-iterations", "3",
            "--aov", f"radiance_sq={rsq}", "--aov", f"shading_normals={nrm}"] + extra
    log = tmp_path / "log.txt"
    with open(log, "w") as f:
        headless.render(headless.parse_args(argv), out=f)
    assert "Denoised: 3 iterations" in log.read_text()
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass", sphere=True, split_method=D.SPLIT_MIDDLE)
    dev = api.Scene(gpu_ctx, scene)
    counts = np.zeros((32, 48), np.uint32) if adaptive else None
    r = api.Renderer(gpu_ctx).render(dev, cam, D.FilmSettings((48, 32), 16), D.SamplerType.uniform(16), D.IntegratorType.path(5),
                                     adaptive=D.Adaptive(4, 4, 0.1) if adaptive else None, sample_counts_out=counts)
    dev.close()
    if adaptive:
        assert np.array_equal(post.read_exr_rgb(str(cnt))[..., 0], counts.astype(np.float32))
    ref = ref_denoise.denoise(r.film, post.read_exr_rgb(str(rsq)), spp=16, sample_counts=counts, normals=post.read_exr_rgb(str(nrm)),
                       iterations=3, sigma=1.5)
    assert _same_bits(post.read_exr_rgb(str(out)), ref)
