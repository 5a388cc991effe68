"""`launch_debug_ray` + `Integrator::li_debug` (app/window.rs:812-905, integrators/mod.rs:76-118, path.rs:71-153,
whitted.rs:89-170): the ray list of one path.

The reference has no test for it ("parity unpinned"): the CPU tests below pin the oracle's restatement to the structure the
source prescribes, the GPU tests compare `yk_debug_ray` with the oracle bit for bit.
"""
import numpy as np
import pytest

from test_render_limits import white_box
from yuki_b200 import api, capi, desc as D, scenes

DIRECT, REFLECTION, REFRACTION, NORMAL, SHADOW = range(5)
FILM = D.FilmSettings((96, 96), 16)
PIXELS = [(48, 48), (10, 80), (70, 30), (95, 0), (33, 61), (52, 70)]


def _cases(xf):
    cornell = scenes.cornell(xf, light="rect", tall_box="glass")
    room = scenes.material_room(xf)
    point = scenes.cornell(xf, light="point")
    return [
        # the deepest settings yk_render admits: Path's bounce counter full, Whitted's largest tree depth
        ("white-box-path-255", *white_box(xf), D.SamplerType.uniform(8), D.IntegratorType.path(255)),
        ("cornell-whitted-24", *cornell, D.SamplerType.stratified(2, 2), D.IntegratorType.whitted(24)),
        ("cornell-path", *cornell, D.SamplerType.stratified(4, 4), D.IntegratorType.path(8)),
        ("cornell-path-uniform", *cornell, D.SamplerType.uniform(16), D.IntegratorType.path(6)),
        ("room-path", *room, D.SamplerType.stratified(3, 3), D.IntegratorType.path(8)),
        ("cornell-whitted", *cornell, D.SamplerType.stratified(2, 2), D.IntegratorType.whitted(5)),
        ("point-whitted", *point, D.SamplerType.uniform(4), D.IntegratorType.whitted(3)),
    ]


def test_oracle_debug_rays_follow_the_reference_structure(oracle, xf):
    saw_refraction = saw_shadow = False
    for name, scene, cam, smp, integ in _cases(xf):
        osc = oracle.OracleScene(scene)
        bounds = osc.nodes()[0]
        extent = np.asarray(bounds["p_max"], np.float32) - np.asarray(bounds["p_min"], np.float32)
        min_len = np.float32(extent.max()) / np.float32(10.0)
        for px in PIXELS:
            rays, li, count = osc.debug_ray(cam, FILM, smp, integ, px)
            t = rays["ray_type"]
            assert len(rays) >= 1 and t[0] == DIRECT, name
            # one bounce ray per traced ray (path.rs:87, whitted.rs:108,174); only the camera ray is "direct"
            bounce = np.isin(t, (DIRECT, REFLECTION, REFRACTION))
            assert int(bounce.sum()) == count, name
            assert int((t == DIRECT).sum()) == 1, name
            assert np.all(np.isfinite(li)) and np.all(li >= 0)
            for i in np.flatnonzero(t == NORMAL):
                # a normal follows the bounce ray that hit, starts at the hit point and has the fixed debug length
                assert bounce[i - 1], name
                hit = rays["o"][i - 1] + rays["d"][i - 1] * rays["t_max"][i - 1]
                assert np.allclose(hit, rays["o"][i], atol=2e-4), name
                assert rays["t_max"][i] == min_len, name
                assert abs(np.linalg.norm(rays["d"][i]) - 1.0) < 1e-5, name
            for i in np.flatnonzero(t == SHADOW):
                assert rays["t_max"][i] == np.float32(0.9999), name  # interaction.rs:57-58
                j = i - 1
                while t[j] == SHADOW:
                    j -= 1
                assert t[j] == NORMAL, name  # shadow rays are collected right after the hit's normal
            saw_refraction |= bool((t == REFRACTION).any())
            saw_shadow |= bool((t == SHADOW).any())
    assert saw_refraction and saw_shadow


def test_oracle_debug_ray_uses_the_fresh_sampler_and_the_clicked_pixel(oracle, xf):
    """window.rs:884-888: the sampler is a fresh clone (pixel (0,0), sample 0, dimension 0, `Pcg32::new(seed, 0)`, never
    seeked), the camera sample is film_px + get_2d(). The first get_2d is recomputed here from the PCG / SipHash /
    permutation primitives and the camera ray must equal Camera::ray at that film position."""
    import struct
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    osc = oracle.OracleScene(scene)
    px = (40, 20)
    for smp in (D.SamplerType.uniform(4, seed=99), D.SamplerType.stratified(3, 2, seed=5), D.SamplerType.stratified(3, 2, jitter=False, seed=5)):
        u = (oracle.pcg32_sequence(smp.seed, 0, 0, 2) >> 8).astype(np.float32) * np.float32(2.0 ** -24)
        if smp.kind == D.SAMPLER_STRATIFIED:
            h = oracle.siphash13(struct.pack("=HHIQ", 0, 0, 0, smp.seed))  # hash_values!(pixel, dimension, seed), stratified.rs:122
            stratum = oracle.permutation_element(0, smp.nx * smp.ny, h & 0xFFFFFFFF)
            sx, sy = stratum % smp.nx, stratum // smp.ny   # (the reference divides by pixel_samples.y, stratified.rs:128)
            d = u if smp.jitter else np.float32([0.5, 0.5])
            u = np.float32([(np.float32(sx) + d[0]) / np.float32(smp.nx), (np.float32(sy) + d[1]) / np.float32(smp.ny)])
        rays, _, _ = osc.debug_ray(cam, FILM, smp, D.IntegratorType.path(3), px)
        o, d = oracle.camera_rays(cam, FILM, np.float32([[np.float32(px[0]) + u[0], np.float32(px[1]) + u[1]]]))
        assert np.array_equal(rays["o"][0], o[0]) and np.array_equal(rays["d"][0], d[0]), smp
        # a different pixel gives a different ray from the same origin
        other, _, _ = osc.debug_ray(cam, FILM, smp, D.IntegratorType.path(3), (41, 20))
        assert np.array_equal(rays["o"][0], other["o"][0]) and not np.array_equal(rays["d"][0], other["d"][0])


def test_oracle_debug_integrators_collect_nothing(oracle, xf):
    """integrators/mod.rs:103-118: the trait's default li_debug returns zero radiance, zero rays."""
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    osc = oracle.OracleScene(scene)
    for integ in (D.IntegratorType.bvh_intersections(), D.IntegratorType.debug(D.INTEGRATOR_GEOMETRY_NORMALS)):
        rays, li, count = osc.debug_ray(cam, FILM, D.SamplerType.uniform(1), integ, (48, 48))
        assert len(rays) == 0 and count == 0 and not li.any()


def test_debug_ray_symbol_rejects_null_arguments():
    L = capi.lib()
    assert L.yk_debug_ray(None, None, None, None, None, 0, 0, None, 0, None, None, None) == -1
    assert b"yk_debug_ray" in L.yk_last_error()


@pytest.mark.gpu
def test_gpu_debug_rays_match_the_oracle_bit_for_bit(gpu_ctx, oracle, xf):
    rn = api.Renderer(gpu_ctx)
    for name, scene, cam, smp, integ in _cases(xf):
        dev = api.Scene(gpu_ctx, scene)
        osc = oracle.OracleScene(scene)
        for px in PIXELS:
            g_rays, g_li, g_count = rn.debug_ray(dev, cam, FILM, smp, integ, px)
            o_rays, o_li, o_count = osc.debug_ray(cam, FILM, smp, integ, px)
            assert len(g_rays) == len(o_rays) and g_count == o_count, (name, px)
            assert g_rays.tobytes() == o_rays.tobytes(), (name, px)
            if integ.kind == D.INTEGRATOR_PATH:
                assert np.array_equal(g_li.view(np.uint32), o_li.view(np.uint32)), (name, px)
            else:  # Whitted: top-down pre-multiplied weights, a documented rounding difference (DESIGN.md §2)
                assert np.allclose(g_li, o_li, rtol=1e-5, atol=1e-7), (name, px)
        dev.close()


@pytest.mark.gpu
def test_gpu_debug_ray_edge_cases(gpu_ctx, oracle, xf):
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    dev = api.Scene(gpu_ctx, scene)
    rn = api.Renderer(gpu_ctx)
    smp, integ = D.SamplerType.stratified(4, 4), D.IntegratorType.path(8)
    # outside the film: no ray is launched (window.rs:866-869)
    assert rn.debug_ray(dev, cam, FILM, smp, integ, (96, 10)) is None
    assert rn.debug_ray(dev, cam, FILM, smp, integ, (-1, 10)) is None
    # the debug integrators keep the default li_debug
    rays, li, count = rn.debug_ray(dev, cam, FILM, smp, D.IntegratorType.bvh_intersections(), (48, 48))
    assert len(rays) == 0 and count == 0 and not li.any()
    # a short buffer reports the full count and fills what fits; the wrapper then retries with room for all
    full, _, _ = rn.debug_ray(dev, cam, FILM, smp, integ, (48, 48))
    short, _, _ = rn.debug_ray(dev, cam, FILM, smp, integ, (48, 48), max_rays=2)
    assert len(full) > 2 and short.tobytes() == full.tobytes()
    # a render after a debug ray is unaffected (the debug path runs on the context's own wavefront state)
    a = rn.render(dev, cam, D.FilmSettings((64, 64), 16), smp, integ).film
    rn.debug_ray(dev, cam, FILM, smp, integ, (5, 5))
    b = rn.render(dev, cam, D.FilmSettings((64, 64), 16), smp, integ).film
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    # a ray that leaves the scene: an open scene (heightfield) seen from above the horizon
    hf, hcam = scenes.heightfield(xf, 32, 32, seed=2)
    hdev = api.Scene(gpu_ctx, hf)
    hosc = oracle.OracleScene(hf)
    for px in [(0, 0), (95, 95), (48, 5), (48, 60)]:
        g = rn.debug_ray(hdev, hcam, FILM, smp, integ, px)
        o = hosc.debug_ray(hcam, FILM, smp, integ, px)
        assert g[0].tobytes() == o[0].tobytes() and g[2] == o[2]
    hdev.close()
    dev.close()
