"""Oracle self-consistency (the reference ships no renderer tests, SURVEY.md §8c) and the committed golden fixtures."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import rel_rmse
from yuki_b200 import desc as D, scenes

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_renders.json")


def golden_cases(xf):
    c_point, cam = scenes.cornell(xf, light="point", tall_box="glass")
    c_rect, _ = scenes.cornell(xf, light="rect", tall_box="glass", textured_back_wall=True)
    room, rcam = scenes.material_room(xf)
    hf, hcam = scenes.heightfield(xf, 48, 48, seed=3)
    film = D.FilmSettings((48, 48), 16)
    c_sphere, _ = scenes.cornell(xf, light="rect", tall_box="glass", sphere=True, split_method=D.SPLIT_MIDDLE)
    sky, scam = scenes.open_scene(xf)
    return {
        "cornell_sphere_path6_s2x2": (c_sphere, cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.path(6)),
        "cornell_sphere_whitted4_s2x2": (c_sphere, cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.whitted(4)),
        "open_scene_distant_path6_s3x3": (sky, scam, D.FilmSettings((60, 40), 16), D.SamplerType.stratified(3, 3), D.IntegratorType.path(6)),
        "room_whitted5_s2x2": (room, rcam, D.FilmSettings((64, 36), 16), D.SamplerType.stratified(2, 2), D.IntegratorType.whitted(5)),
        "cornell_point_whitted3_s2x2": (c_point, cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.whitted(3)),
        "cornell_rect_path8_s2x2": (c_rect, cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.path(8)),
        "cornell_rect_path8_uniform3": (c_rect, cam, film, D.SamplerType.uniform(3), D.IntegratorType.path(8)),
        "room_path8_s2x2": (room, rcam, D.FilmSettings((64, 36), 16), D.SamplerType.stratified(2, 2), D.IntegratorType.path(8)),
        "heightfield_bvh_counts": (hf, hcam, D.FilmSettings((80, 60), 16), D.SamplerType.uniform(1), D.IntegratorType.bvh_intersections()),
        "room_shading_normals": (room, rcam, D.FilmSettings((64, 36), 16), D.SamplerType.uniform(1), D.IntegratorType.debug(D.INTEGRATOR_SHADING_NORMALS)),
    }


def roulette_draw_of_one_case(xf):
    """Two samples of the benchmark render (Cornell box 1024x1024, Path 8, stratified 32x32) whose paths lose their green
    throughput on the red wall, so that Russian roulette's q is 1 at the fifth vertex, and whose roulette draw rounds up to
    exactly 1.0f: an accumulating one-pixel tile each. Found by rendering every sample of the pixels that were NaN in the
    benchmark film one at a time. Returns (scene, camera, film, sampler, integrator, tiles)."""
    from yuki_b200 import capi
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    tiles = np.zeros(2, capi.TILE_DTYPE)
    tiles[0] = (448, 246, 449, 247, 265, 0, 0)
    tiles[1] = (630, 673, 631, 674, 424, 0, 1)
    return (scene, cam, D.FilmSettings((1024, 1024), 16, accumulate=True), D.SamplerType.stratified(32, 32, jitter=True),
            D.IntegratorType.path(8), tiles)


def digest(img, ids, st):
    return {"film_sha256": hashlib.sha256(np.ascontiguousarray(img).tobytes()).hexdigest(),
            "ids_sha256": hashlib.sha256(np.ascontiguousarray(ids).tobytes()).hexdigest(),
            "ray_count": int(st.ray_count), "shadow_rays": int(st.shadow_rays), "closest_nodes": int(st.closest_nodes),
            "primary_hit_hash": int(st.primary_hit_hash), "film_mean": float(np.mean(img, dtype=np.float64))}


def test_golden_fixtures(oracle, xf):
    """tests/golden/oracle_renders.json was produced by tests/golden/make_golden.py with this oracle on this image
    (the Rust reference cannot run here): it pins the oracle against silent change, not against the reference."""
    want = json.load(open(GOLDEN))
    for name, (scene, cam, film, smp, integ) in golden_cases(xf).items():
        img, ids, st = oracle.OracleScene(scene).render(cam, film, smp, integ, want_hit_ids=True)
        got = digest(img, ids, st)
        assert got == want[name], name


def test_thread_count_does_not_change_the_film(oracle, xf):
    """integrators/mod.rs:135-142: the sampler is re-cloned per tile so results do not depend on thread assignment."""
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    film = D.FilmSettings((40, 40), 8)
    osc = oracle.OracleScene(scene)
    a, _, sa = osc.render(cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.path(6), threads=1)
    b, _, sb = osc.render(cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.path(6), threads=5)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and sa.ray_count == sb.ray_count


def test_whitted_equals_path_depth_one_on_diffuse_scene(oracle, xf):
    """Direct lighting only: Whitted(max_depth 1) and Path(max_depth 1) evaluate the same light fold with the same draws."""
    scene, cam = scenes.cornell(xf, light="point", tall_box="matte")
    film = D.FilmSettings((32, 32), 16)
    osc = oracle.OracleScene(scene)
    w, _, _ = osc.render(cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.whitted(1))
    p, _, _ = osc.render(cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.path(1))
    assert np.array_equal(w.view(np.uint32), p.view(np.uint32))


def test_accumulate_mode(oracle, xf):
    """film.rs:260-272 + render_manager.rs:135-143: accumulate mode adds one sample per tile pass; the sum over samples
    divided by spp is the averaged render (up to summation order)."""
    scene, cam = scenes.cornell(xf, light="point", tall_box="matte")
    osc = oracle.OracleScene(scene)
    smp = D.SamplerType.stratified(2, 2)
    avg, _, _ = osc.render(cam, D.FilmSettings((32, 32), 16), smp, D.IntegratorType.whitted(3), threads=1)
    acc, _, st = osc.render(cam, D.FilmSettings((32, 32), 16, accumulate=True), smp, D.IntegratorType.whitted(3), threads=1)
    assert st.samples == 32 * 32 * 4
    assert np.allclose(acc / 4.0, avg, rtol=1e-5, atol=1e-6)


def test_white_furnace_energy_bound(oracle, xf):
    """A closed grey box around a point light cannot return more radiance per bounce than it receives: deeper paths add
    energy monotonically and the series stays bounded."""
    scene, cam = scenes.cornell(xf, light="point", tall_box=None)
    osc = oracle.OracleScene(scene)
    film = D.FilmSettings((24, 24), 8)
    means = [float(osc.render(cam, film, D.SamplerType.stratified(4, 4), D.IntegratorType.path(d))[0].mean()) for d in (1, 2, 4, 8)]
    assert means[0] > 0 and all(b >= a * 0.98 for a, b in zip(means, means[1:])) and means[-1] < 4 * means[0]


def test_ray_counts(oracle, xf):
    """Mrays/s counts closest-hit rays only (path.rs:87): a depth-1 path traces exactly one ray per sample."""
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    osc = oracle.OracleScene(scene)
    _, _, st = osc.render(cam, D.FilmSettings((16, 16), 16), D.SamplerType.uniform(2), D.IntegratorType.path(1))
    assert st.ray_count == 16 * 16 * 2 and st.samples == 16 * 16 * 2
    _, _, st = osc.render(cam, D.FilmSettings((16, 16), 16), D.SamplerType.uniform(2), D.IntegratorType.path(0))
    assert st.ray_count == 0


def test_roulette_ends_a_path_whose_continuation_probability_is_zero(oracle, xf):
    """q == 1 ends the path whatever the draw: a draw of exactly 1.0f used to go on with beta * 1 / 0 and make the pixel NaN."""
    scene, cam, film, smp, integ, tiles = roulette_draw_of_one_case(xf)
    # draws up to the first roulette: the camera jitter, then per vertex one get_2d per light (one light) and the BSDF's
    # get_2d, five vertices (bounces 0..4), then roulette's get_1d
    assert len(scene.lights) == 1
    for t in tiles:
        draws = oracle.sampler_draws(smp, int(t["x0"]), int(t["y0"]), int(t["sample"]), [2] + [2, 2] * 5 + [1])
        assert draws[-1] == np.float32(1.0)
    img, _, st = oracle.OracleScene(scene).render(cam, film, smp, integ, tiles=tiles)
    px = img[tiles["y0"], tiles["x0"]]
    assert st.samples == 2 and np.isfinite(px).all() and (px >= 0).all()
