"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs.

Gates (SURVEY.md §8d): BVH-intersection counter images and primary-hit triangle ids bit-exact; radiance within
per-image relative RMSE <= 1e-3; closest-hit ray counts within 0.1 %. The CUDA path in fact reproduces the oracle's
films bit for bit (un-fused IEEE arithmetic in the reference's association, glibc-exact libm restatements, Whitted's tree
summed bottom-up) and the *_bit_identical_* tests assert that.
"""
import numpy as np
import pytest

from conftest import rel_rmse
from yuki_b200 import api, desc as D, scenes

pytestmark = pytest.mark.gpu

RMSE_TOL = 1e-3


def _both(gpu_ctx, oracle, xf, scene, cam, film, sampler, integ, **kw):
    dev = api.Scene(gpu_ctx, scene)
    r = api.Renderer(gpu_ctx).render(dev, cam, film, sampler, integ, want_hit_ids=True, **kw)
    osc = oracle.OracleScene(scene)
    o_img, o_ids, o_st = osc.render(cam, film, sampler, integ, want_hit_ids=True)
    dev.close()
    return r, o_img, o_ids, o_st


@pytest.mark.parametrize("split", [D.SPLIT_SAH, D.SPLIT_MIDDLE, D.SPLIT_EQUAL_COUNTS])
def test_bvh_intersections_bit_exact(gpu_ctx, oracle, xf, split):
    scene, cam = scenes.heightfield(xf, 96, 96, seed=3, split_method=split)
    film = D.FilmSettings((160, 120), 16)
    r, o_img, o_ids, o_st = _both(gpu_ctx, oracle, xf, scene, cam, film, D.SamplerType.uniform(1), D.IntegratorType.bvh_intersections())
    assert np.array_equal(r.hit_ids, o_ids)
    assert np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32))
    assert r.stats.closest_nodes == o_st.closest_nodes == int(o_img[..., 0].sum())
    assert r.stats.closest_tris == o_st.closest_tris
    assert r.stats.primary_hit_hash == o_st.primary_hit_hash
    assert r.stats.ray_count == o_st.ray_count == 160 * 120


@pytest.mark.parametrize("kind", [D.INTEGRATOR_GEOMETRY_NORMALS, D.INTEGRATOR_SHADING_NORMALS, D.INTEGRATOR_SHADING_UVS])
def test_debug_integrators_bit_exact(gpu_ctx, oracle, xf, kind):
    scene, cam = scenes.material_room(xf)
    film = D.FilmSettings((96, 64), 16)
    r, o_img, o_ids, _ = _both(gpu_ctx, oracle, xf, scene, cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.debug(kind))
    assert np.array_equal(r.hit_ids, o_ids)
    assert np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32))


def test_whitted_cornell_point_light(gpu_ctx, oracle, xf):
    scene, cam = scenes.cornell(xf, light="point", tall_box="glass")
    film = D.FilmSettings((128, 128), 16)
    r, o_img, o_ids, o_st = _both(gpu_ctx, oracle, xf, scene, cam, film, D.SamplerType.stratified(4, 4), D.IntegratorType.whitted(3))
    assert np.array_equal(r.hit_ids, o_ids)
    assert r.stats.primary_hit_hash == o_st.primary_hit_hash
    assert abs(int(r.stats.ray_count) - int(o_st.ray_count)) <= 1e-3 * o_st.ray_count
    assert rel_rmse(r.film, o_img) <= RMSE_TOL


def test_whitted_deep_recursion(gpu_ctx, oracle, xf):
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    film = D.FilmSettings((96, 96), 32)
    r, o_img, o_ids, o_st = _both(gpu_ctx, oracle, xf, scene, cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.whitted(6))
    assert np.array_equal(r.hit_ids, o_ids)
    assert abs(int(r.stats.ray_count) - int(o_st.ray_count)) <= 1e-3 * o_st.ray_count
    assert rel_rmse(r.film, o_img) <= RMSE_TOL


@pytest.mark.parametrize("sampler", [D.SamplerType.stratified(4, 4), D.SamplerType.uniform(8), D.SamplerType.stratified(3, 2, jitter=False)])
def test_path_cornell_area_light(gpu_ctx, oracle, xf, sampler):
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass", textured_back_wall=True)
    film = D.FilmSettings((128, 128), 16)
    r, o_img, o_ids, o_st = _both(gpu_ctx, oracle, xf, scene, cam, film, sampler, D.IntegratorType.path(8))
    assert np.array_equal(r.hit_ids, o_ids)
    assert r.stats.primary_hit_hash == o_st.primary_hit_hash
    assert abs(int(r.stats.ray_count) - int(o_st.ray_count)) <= 1e-3 * o_st.ray_count
    assert abs(int(r.stats.shadow_rays) - int(o_st.shadow_rays)) <= 1e-3 * o_st.shadow_rays
    assert rel_rmse(r.film, o_img) <= RMSE_TOL


def test_path_material_room_all_materials_and_lights(gpu_ctx, oracle, xf):
    scene, cam = scenes.material_room(xf)
    film = D.FilmSettings((160, 90), 16)
    r, o_img, o_ids, o_st = _both(gpu_ctx, oracle, xf, scene, cam, film, D.SamplerType.stratified(4, 4), D.IntegratorType.path(8))
    assert np.array_equal(r.hit_ids, o_ids)
    assert abs(int(r.stats.ray_count) - int(o_st.ray_count)) <= 1e-3 * o_st.ray_count
    assert rel_rmse(r.film, o_img) <= RMSE_TOL


def test_path_indirect_clamp(gpu_ctx, oracle, xf):
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    film = D.FilmSettings((64, 64), 16)
    r, o_img, _, _ = _both(gpu_ctx, oracle, xf, scene, cam, film, D.SamplerType.stratified(4, 4), D.IntegratorType.path(6, indirect_clamp=2.0))
    assert rel_rmse(r.film, o_img) <= RMSE_TOL


def test_small_wavefront_batches_match_single_batch(gpu_ctx, xf):
    """Batching is invisible: many small batches give the same film bits as one large batch."""
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    film = D.FilmSettings((64, 48), 16)
    dev = api.Scene(gpu_ctx, scene)
    rn = api.Renderer(gpu_ctx)
    a = rn.render(dev, cam, film, D.SamplerType.stratified(4, 4), D.IntegratorType.path(8))
    b = rn.render(dev, cam, film, D.SamplerType.stratified(4, 4), D.IntegratorType.path(8), wavefront_paths=4096)
    assert np.array_equal(a.film.view(np.uint32), b.film.view(np.uint32))
    assert a.stats.ray_count == b.stats.ray_count


def test_tile_subset_and_ragged_film(gpu_ctx, oracle, xf):
    """Film not a multiple of the tile size, and only every other spiral tile rendered (a 2-rank share)."""
    scene, cam = scenes.cornell(xf, light="point", tall_box="matte")
    film = D.FilmSettings((70, 50), 16)
    tiles = api.film_tiles(film)[::2]
    dev = api.Scene(gpu_ctx, scene)
    r = api.Renderer(gpu_ctx).render(dev, cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.whitted(3), tiles=tiles)
    o_img, _, _ = oracle.OracleScene(scene).render(cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.whitted(3), tiles=tiles)
    covered = np.zeros((50, 70), bool)
    for t in tiles:
        covered[t["y0"]:t["y1"], t["x0"]:t["x1"]] = True
    assert np.all(r.film[~covered] == 0.0)
    assert rel_rmse(r.film, o_img) <= RMSE_TOL


def test_accumulate_mode_sums_samples(gpu_ctx, oracle, xf):
    """film.rs:260-272: accumulating tiles add one sample each; the sum over samples / spp equals the averaged render."""
    scene, cam = scenes.cornell(xf, light="point", tall_box="matte")
    film = D.FilmSettings((48, 48), 16)
    acc = D.FilmSettings((48, 48), 16, accumulate=True)
    smp = D.SamplerType.stratified(2, 2)
    dev = api.Scene(gpu_ctx, scene)
    rn = api.Renderer(gpu_ctx)
    avg = rn.render(dev, cam, film, smp, D.IntegratorType.whitted(3)).film
    tiles = api.film_tiles(film)
    out = np.zeros((48, 48, 3), np.float32)
    for s in range(4):
        t = tiles.copy()
        t["sample"] = s
        rn.render(dev, cam, acc, smp, D.IntegratorType.whitted(3), tiles=t, film_out=out)
    assert np.allclose(out / 4.0, avg, rtol=1e-5, atol=1e-6)


def test_empty_tile_list_and_bad_arguments(gpu_ctx, xf):
    from yuki_b200 import capi
    scene, cam = scenes.cornell(xf, light="point", tall_box=None)
    film = D.FilmSettings((32, 32), 16)
    dev = api.Scene(gpu_ctx, scene)
    rn = api.Renderer(gpu_ctx)
    r = rn.render(dev, cam, film, D.SamplerType.uniform(1), D.IntegratorType.whitted(3), tiles=np.zeros(0, capi.TILE_DTYPE))
    assert r.stats.samples == 0 and np.all(r.film == 0)
    bad = np.zeros(1, capi.TILE_DTYPE)
    bad[0] = (0, 0, 64, 16, 0, 0, 0)
    with pytest.raises(capi.YukiGpuError):
        rn.render(dev, cam, film, D.SamplerType.uniform(1), D.IntegratorType.whitted(3), tiles=bad)
    with pytest.raises(capi.YukiGpuError):
        rn.render(dev, cam, film, D.SamplerType.uniform(0), D.IntegratorType.whitted(3))


def test_gpu_matches_committed_golden_fixtures(gpu_ctx, xf):
    """The GPU box has no reference checkout: compare against tests/golden/oracle_renders.json (made by
    tests/golden/make_golden.py). Every film — Path, Whitted, debug integrators — is bit-identical."""
    import hashlib
    import json
    from test_oracle_render import GOLDEN, golden_cases
    want = json.load(open(GOLDEN))
    for name, (scene, cam, film, smp, integ) in golden_cases(xf).items():
        dev = api.Scene(gpu_ctx, scene)
        r = api.Renderer(gpu_ctx).render(dev, cam, film, smp, integ, want_hit_ids=True)
        dev.close()
        g = want[name]
        assert hashlib.sha256(r.hit_ids.tobytes()).hexdigest() == g["ids_sha256"], name
        assert r.stats.primary_hit_hash == g["primary_hit_hash"] and r.stats.ray_count == g["ray_count"], name
        assert r.stats.closest_nodes == g["closest_nodes"] and r.stats.shadow_rays == g["shadow_rays"], name
        assert abs(float(np.mean(r.film, dtype=np.float64)) - g["film_mean"]) <= 1e-6 * g["film_mean"], name
        assert hashlib.sha256(r.film.tobytes()).hexdigest() == g["film_sha256"], name


def test_roulette_with_zero_continuation_probability_matches_the_oracle(gpu_ctx, oracle, xf):
    """The two benchmark samples whose roulette draw is exactly 1.0f at q == 1 (test_oracle_render.py): finite and bit-identical."""
    from test_oracle_render import roulette_draw_of_one_case
    scene, cam, film, smp, integ, tiles = roulette_draw_of_one_case(xf)
    dev = api.Scene(gpu_ctx, scene)
    r = api.Renderer(gpu_ctx).render(dev, cam, film, smp, integ, tiles=tiles)
    dev.close()
    o_img, _, o_st = oracle.OracleScene(scene).render(cam, film, smp, integ, tiles=tiles)
    assert np.isfinite(r.film).all() and np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32))
    assert r.stats.ray_count == o_st.ray_count


def test_path_is_bit_identical_to_the_oracle(gpu_ctx, oracle, xf):
    """Stronger than the RMSE gate: with un-fused IEEE arithmetic and glibc-exact sinf/cosf the Path film has no
    differing bit, for every material and light kind."""
    for scene, cam, film in [(*scenes.material_room(xf), D.FilmSettings((96, 54), 16)),
                             (*scenes.cornell(xf, light="rect", tall_box="glass", textured_back_wall=True), D.FilmSettings((64, 64), 16))]:
        r, o_img, o_ids, o_st = _both(gpu_ctx, oracle, xf, scene, cam, film, D.SamplerType.stratified(3, 3), D.IntegratorType.path(8))
        assert np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32))
        assert r.stats.ray_count == o_st.ray_count and r.stats.shadow_rays == o_st.shadow_rays
        assert r.stats.any_nodes == o_st.any_nodes and r.stats.any_tris == o_st.any_tris


def test_whitted_is_bit_identical_to_the_oracle(gpu_ctx, oracle, xf):
    """The recursion tree is summed bottom-up like whitted.rs:132-170 does (k_tree_return), so the Whitted film has no
    differing bit either: nested glass (reflection + transmission subtrees), every material, deep recursion."""
    for scene, cam, film, depth in [(*scenes.cornell(xf, light="rect", tall_box="glass"), D.FilmSettings((96, 96), 32), 6),
                                    (*scenes.cornell(xf, light="point", tall_box="glass"), D.FilmSettings((64, 64), 16), 3),
                                    (*scenes.material_room(xf), D.FilmSettings((96, 54), 16), 5),
                                    (*scenes.cornell(xf, light="rect", tall_box="glass"), D.FilmSettings((32, 32), 16), 1)]:
        r, o_img, o_ids, o_st = _both(gpu_ctx, oracle, xf, scene, cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.whitted(depth))
        assert np.array_equal(r.hit_ids, o_ids)
        assert np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32))
        assert r.stats.ray_count == o_st.ray_count and r.stats.shadow_rays == o_st.shadow_rays


@pytest.mark.parametrize("integ", [D.IntegratorType.path(6), D.IntegratorType.whitted(4)])
def test_distant_light_and_background_in_an_open_scene(gpu_ctx, oracle, xf, integ):
    scene, cam = scenes.open_scene(xf)
    film = D.FilmSettings((120, 80), 16)
    r, o_img, o_ids, o_st = _both(gpu_ctx, oracle, xf, scene, cam, film, D.SamplerType.stratified(3, 3), integ)
    assert np.array_equal(r.hit_ids, o_ids)
    assert (o_ids < 0).any() and (o_ids >= 0).any()
    assert np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32))
    assert r.stats.ray_count == o_st.ray_count and r.stats.shadow_rays == o_st.shadow_rays


def test_many_lights_and_the_light_limit(gpu_ctx, oracle, xf):
    """32 lights (the shadow-ray mask's width) of every kind, folded in light order; a 33rd is refused at scene creation."""
    scene, cam = scenes.material_room(xf)
    rng = np.random.default_rng(4)
    while len(scene.lights) < 32:
        k = len(scene.lights)
        pos = tuple(float(v) for v in rng.uniform((-1.0, 0.3, -1.0), (1.0, 1.1, 1.0)))
        if k % 3 == 0:
            scene.lights.append(D.Light(D.LIGHT_DISTANT, xf.identity(), (0.05, 0.05, 0.06), direction=tuple(float(v) for v in rng.uniform(-1, 1, 3))))
        elif k % 3 == 1:
            scene.lights.append(D.Light(D.LIGHT_POINT, xf.translation(pos), tuple(float(v) for v in rng.uniform(0.02, 0.1, 3))))
        else:
            spot = xf.mul(xf.translation(pos), xf.rotation(float(rng.uniform(0.5, 2.5)), (1.0, 0.2, 0.0)))
            scene.lights.append(D.Light(D.LIGHT_SPOT, spot, (0.4, 0.4, 0.3), total_width_deg=40.0, falloff_start_deg=25.0))
    film = D.FilmSettings((64, 36), 16)
    for integ in (D.IntegratorType.path(4), D.IntegratorType.whitted(3)):
        r, o_img, o_ids, o_st = _both(gpu_ctx, oracle, xf, scene, cam, film, D.SamplerType.stratified(2, 2), integ)
        assert np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32))
        assert r.stats.shadow_rays == o_st.shadow_rays and r.stats.any_nodes == o_st.any_nodes
    scene.lights.append(D.Light(D.LIGHT_POINT, xf.translation((0.0, 1.0, 0.0)), (0.1, 0.1, 0.1)))
    with pytest.raises(RuntimeError, match="32 lights"):
        api.Scene(gpu_ctx, scene)


@pytest.mark.parametrize("integ", [D.IntegratorType.path(0), D.IntegratorType.path(1), D.IntegratorType.whitted(0), D.IntegratorType.whitted(1),
                                   D.IntegratorType.bvh_intersections()])
def test_degenerate_settings(gpu_ctx, oracle, xf, integ):
    """max_depth 0 / 1 (path.rs:66: the loop body never / once runs), a 1x1 film, a tile larger than the film, one sample."""
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    for film, smp in ((D.FilmSettings((1, 1), 16), D.SamplerType.uniform(1)),
                      (D.FilmSettings((23, 9), 64), D.SamplerType.stratified(1, 1)),
                      (D.FilmSettings((17, 31), 7), D.SamplerType.stratified(2, 3, jitter=False))):
        r, o_img, o_ids, o_st = _both(gpu_ctx, oracle, xf, scene, cam, film, smp, integ)
        assert np.array_equal(r.hit_ids, o_ids)
        assert np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32))
        assert r.stats.ray_count == o_st.ray_count and r.stats.shadow_rays == o_st.shadow_rays
        assert r.stats.samples == film.res[0] * film.res[1] * smp.samples_per_pixel()


def test_image_textured_roughness_is_remapped_with_glibc_logf(gpu_ctx, oracle, xf):
    """Metal / Glossy roughness from an image texture with remap_roughness: roughness_to_alpha (trowbridge_reitz.rs:22-30)
    runs per hit on the device, through the restated glibc logf (constant roughness is converted on the host)."""
    scene, cam = scenes.material_room(xf)
    rng = np.random.default_rng(8)
    rough = np.repeat(rng.uniform(0.0, 0.95, (32, 32, 1)).astype(np.float32), 3, axis=2)   # includes values below the 1e-3 floor
    rough[0, :4] = 0.0
    t = scene.add_texture(D.Texture.from_image(rough))
    n_mapped = 0
    for i, m in enumerate(scene.materials):
        if m.kind == D.MAT_METAL:
            scene.materials[i] = D.Material(D.MAT_METAL, (m.tex[0], m.tex[1], t), remap_roughness=True)
            n_mapped += 1
        elif m.kind == D.MAT_GLOSSY:
            scene.materials[i] = D.Material(D.MAT_GLOSSY, (m.tex[0], t), remap_roughness=True)
            n_mapped += 1
    assert n_mapped == 2
    film = D.FilmSettings((160, 90), 16)
    for integ in (D.IntegratorType.path(6), D.IntegratorType.whitted(3)):
        r, o_img, o_ids, o_st = _both(gpu_ctx, oracle, xf, scene, cam, film, D.SamplerType.stratified(3, 3), integ)
        assert np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32))
        assert r.stats.ray_count == o_st.ray_count and r.stats.shadow_rays == o_st.shadow_rays


def test_round_trip_properties_at_full_size(gpu_ctx, xf):
    """Size-independent properties on the benchmark-size film (the oracle would take minutes here): rendering the two
    interleaved halves of the tile list separately and summing equals rendering all tiles; re-rendering is idempotent;
    every pixel is finite and non-negative."""
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    film = D.FilmSettings((1024, 1024), 16)
    smp, integ = D.SamplerType.stratified(2, 2), D.IntegratorType.path(8)
    dev = api.Scene(gpu_ctx, scene)
    rn = api.Renderer(gpu_ctx)
    tiles = api.film_tiles(film)
    full = rn.render(dev, cam, film, smp, integ)
    again = rn.render(dev, cam, film, smp, integ)
    a = rn.render(dev, cam, film, smp, integ, tiles=tiles[0::2])
    b = rn.render(dev, cam, film, smp, integ, tiles=tiles[1::2])
    assert np.array_equal(full.film.view(np.uint32), again.film.view(np.uint32))
    assert np.array_equal((a.film + b.film).view(np.uint32), full.film.view(np.uint32))
    assert a.stats.ray_count + b.stats.ray_count == full.stats.ray_count
    assert np.isfinite(full.film).all() and (full.film >= 0).all()
    assert full.stats.samples == 1024 * 1024 * 4
    dev.close()


def test_async_renderer_launch_check_status_kill(gpu_ctx, xf):
    """renderer/mod.rs:53-177: launch() returns at once, check_status() reports progress and then Finished{ray_count},
    kill() stops a running task; the film equals the blocking render's."""
    import time
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    fs = D.FilmSettings((96, 96), 16)
    smp, integ = D.SamplerType.stratified(4, 4), D.IntegratorType.path(6)
    dev = api.Scene(gpu_ctx, scene)
    rn = api.Renderer(gpu_ctx)
    ref = rn.render(dev, cam, fs, smp, integ)
    film = api.Film(fs)
    rn.launch(dev, cam, film, smp, integ)
    assert rn.is_active()
    finished, deadline = None, time.time() + 60
    while finished is None and time.time() < deadline:
        st = rn.check_status()
        if isinstance(st, api.RenderFinished):
            finished = st
        elif isinstance(st, api.RenderProgress):
            assert 0 <= st.tiles_done <= st.tiles_total == 36
        time.sleep(0.001)
    assert finished is not None and not rn.is_active()
    assert finished.ray_count == ref.stats.ray_count
    assert np.array_equal(film.pixels.view(np.uint32), ref.film.view(np.uint32)) and film.dirty
    # a long render is cut short by kill() (polled between wavefront batches)
    big = D.FilmSettings((512, 512), 16)
    film2 = api.Film(big)
    t0 = time.time()
    rn.launch(dev, cam, film2, D.SamplerType.stratified(32, 32), D.IntegratorType.path(8), wavefront_paths=1 << 18)
    time.sleep(0.05)
    rn.kill()
    assert not rn.is_active() and rn.check_status() is None
    assert time.time() - t0 < 20.0


def test_accumulating_launch_counts_samples_and_matches_the_mean(gpu_ctx, xf):
    """render_manager.rs:135-143 + film.rs:260-272: an accumulating launch renders one tile list per sample index and adds
    them in order; pixels / samples[tile] is then bit-identical to the averaging render (same ascending-sample sums)."""
    import time
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    fs = D.FilmSettings((80, 48), 16)
    acc = D.FilmSettings((80, 48), 16, accumulate=True)
    smp, integ = D.SamplerType.stratified(3, 3), D.IntegratorType.path(5)
    dev = api.Scene(gpu_ctx, scene)
    rn = api.Renderer(gpu_ctx)
    ref = rn.render(dev, cam, fs, smp, integ).film
    film = api.Film(acc)
    rn.launch(dev, cam, film, smp, integ)
    deadline = time.time() + 60
    while rn.is_active() and time.time() < deadline:
        rn.check_status()
        time.sleep(0.001)
    assert not rn.is_active() and rn.last_error is None
    assert np.all(film.samples == 9)
    mean = (film.pixels / np.float32(9.0)).astype(np.float32)
    assert np.array_equal(mean.view(np.uint32), ref.view(np.uint32))
    # a single forced sample (force_single_sample, sampling/mod.rs:21-42) adds exactly one more
    rn.launch(dev, cam, film, smp, integ, force_single_sample=True)
    while rn.is_active() and time.time() < deadline:
        rn.check_status()
        time.sleep(0.001)
    assert np.all(film.samples == 10)


@pytest.mark.parametrize("split,max_shapes", [(D.SPLIT_EQUAL_COUNTS, 40), (D.SPLIT_MIDDLE, 40), (D.SPLIT_SAH, 7), (D.SPLIT_EQUAL_COUNTS, 60000)])
def test_leaf_sizes_counters_and_path_bit_exact(gpu_ctx, oracle, xf, split, max_shapes):
    """Leaves of many shapes: above 16 shapes the device leaf refs go through the leaf table instead of the packed form
    (DESIGN.md §3); with max_shapes above the triangle count the root itself is a leaf (no interior record at all).
    Counter images, hit ids, shadow-ray counters and the Path film stay bit-exact."""
    scene, cam = scenes.heightfield(xf, 40, 40, seed=5, split_method=split, max_shapes_in_node=max_shapes)
    film = D.FilmSettings((96, 72), 16)
    r, o_img, o_ids, o_st = _both(gpu_ctx, oracle, xf, scene, cam, film, D.SamplerType.uniform(1), D.IntegratorType.bvh_intersections())
    assert np.array_equal(r.hit_ids, o_ids)
    assert np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32))
    assert r.stats.closest_nodes == o_st.closest_nodes and r.stats.closest_tris == o_st.closest_tris
    r, o_img, o_ids, o_st = _both(gpu_ctx, oracle, xf, scene, cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.path(5))
    assert np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32))
    assert r.stats.closest_nodes == o_st.closest_nodes and r.stats.closest_tris == o_st.closest_tris
    assert r.stats.any_nodes == o_st.any_nodes and r.stats.any_tris == o_st.any_tris and r.stats.shadow_rays == o_st.shadow_rays


def test_deep_traversal_stack_spills_bit_exact(gpu_ctx, oracle, xf):
    """A degenerate (list-like) hierarchy drives the traversal stack beyond its shared-memory levels into the spill
    arrays: Middle splits of a geometrically graded strip of tilted quads give a one-sided tree, and rays along the strip
    pass through every nested box (up to 69 passed box tests per ray, > 30 pending far children)."""
    import numpy as np_
    n = 60
    xs = np_.concatenate([[0.0], np_.cumsum(1.7 ** np_.arange(n))]).astype(np_.float32)
    xs = xs / xs[-1] * 8.0 - 4.0
    pts, idx = [], []
    for i in range(n):
        b = len(pts)
        pts += [(xs[i], -0.5, 0.0), (xs[i + 1], -0.5, 0.0), (xs[i + 1], 0.5, 1.0), (xs[i], 0.5, 1.0)]
        idx += [b, b + 1, b + 2, b, b + 2, b + 3]
    s = D.SceneDesc(split_method=D.SPLIT_MIDDLE, max_shapes_in_node=1)
    m = s.add_material(D.Material(D.MAT_MATTE, (s.add_texture(D.Texture.constant(0.7, 0.6, 0.5)), s.add_texture(D.Texture.constant(0.0)))))
    s.meshes.append(D.Mesh(xf.identity(), np_.asarray(pts, np_.float32), np_.asarray(idx, np_.uint32), m))
    s.lights.append(D.Light(D.LIGHT_POINT, xf.translation((-6.0, 0.3, 0.2)), (30.0, 30.0, 30.0)))
    cam = D.CameraParameters((-6.0, 0.1, 0.45), (4.0, 0.1, 0.5), fov_axis=D.FOV_X, fov_deg=12.0)  # looks along the strip
    film = D.FilmSettings((80, 60), 16)
    r, o_img, o_ids, o_st = _both(gpu_ctx, oracle, xf, s, cam, film, D.SamplerType.uniform(1), D.IntegratorType.bvh_intersections())
    assert np.array_equal(r.hit_ids, o_ids)
    assert np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32))
    assert o_img[..., 1].max() > 40
    r, o_img, o_ids, o_st = _both(gpu_ctx, oracle, xf, s, cam, film, D.SamplerType.stratified(2, 2), D.IntegratorType.path(4))
    assert np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32))
    assert r.stats.any_nodes == o_st.any_nodes and r.stats.closest_nodes == o_st.closest_nodes


def test_maximum_film_coordinates_and_sample_indices(gpu_ctx, oracle, xf):
    """The limits the reference asserts (integrators/mod.rs:140-141): pixel coordinates and sample indices up to 0xFFFF.
    A 65535-pixel-wide film rendered at its two ends, and the last sample index (65535) of a 256x256-strata sampler in
    accumulate mode, both bit-identical to the oracle (the sampler seek distance is 65535 * 65536 there)."""
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    film = D.FilmSettings((65535, 20), 16)
    all_tiles = api.film_tiles(film)
    assert len(all_tiles) == 4096 * 2 and int(all_tiles["x1"].max()) == 65535
    pick = all_tiles[(all_tiles["x0"] < 32) | (all_tiles["x1"] > 65535 - 32) | ((all_tiles["x0"] >= 32768 - 16) & (all_tiles["x0"] < 32768 + 16))]
    smp, integ = D.SamplerType.stratified(2, 2), D.IntegratorType.path(5)
    dev = api.Scene(gpu_ctx, scene)
    rn = api.Renderer(gpu_ctx)
    r = rn.render(dev, cam, film, smp, integ, tiles=pick)
    o_img, _, o_st = oracle.OracleScene(scene).render(cam, film, smp, integ, tiles=pick)
    assert np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32))
    assert r.stats.ray_count == o_st.ray_count and r.stats.samples == sum(int(t["x1"] - t["x0"]) * int(t["y1"] - t["y0"]) for t in pick) * 4
    # last sample index of the largest sampler the interface admits
    film2 = D.FilmSettings((64, 48), 16, accumulate=True)
    big = D.SamplerType.stratified(256, 256)
    tiles = api.film_tiles(film2).copy()
    tiles["sample"] = 65535
    out = np.zeros((48, 64, 3), np.float32)
    r2 = rn.render(dev, cam, film2, big, integ, tiles=tiles, film_out=out)
    o2, _, o2_st = oracle.OracleScene(scene).render(cam, film2, big, integ, tiles=tiles)
    dev.close()
    assert np.array_equal(out.view(np.uint32), o2.view(np.uint32)) and float(o2.max()) > 0.0
    assert r2.stats.ray_count == o2_st.ray_count


@pytest.mark.parametrize("scene_name", ["room", "heightfield", "sphere_room"])
def test_ray_sort_is_invisible_in_the_results(gpu_ctx, oracle, xf, scene_name):
    """The ray-queue sort between bounces (csrc/wf_sort.cuh) only changes the order rays are processed in: film bits,
    ray counts and traversal counters equal the unsorted render's (and the oracle's) for both keys and both orders."""
    if scene_name == "room":
        scene, cam = scenes.material_room(xf)
    elif scene_name == "heightfield":
        scene, cam = scenes.heightfield(xf, 64, 64, seed=5)
    else:
        scene, cam = scenes.cornell(xf, light="rect", tall_box="glass", sphere=True)
    film = D.FilmSettings((96, 64), 16)
    smp, integ = D.SamplerType.stratified(3, 2), D.IntegratorType.path(8)
    dev = api.Scene(gpu_ctx, scene)
    rn = api.Renderer(gpu_ctx)
    base = rn.render(dev, cam, film, smp, integ, ray_sort=1)
    o_img, _, o_st = oracle.OracleScene(scene).render(cam, film, smp, integ)
    assert np.array_equal(base.film.view(np.uint32), o_img.view(np.uint32))
    for mode in (2, 3, 2 | 16, 3 | 16):
        for kw in ({}, {"wavefront_paths": 2048}, {"pipes": 1}):
            r = rn.render(dev, cam, film, smp, integ, ray_sort=mode, **kw)
            assert np.array_equal(r.film.view(np.uint32), base.film.view(np.uint32)), (mode, kw)
            for k in ("ray_count", "shadow_rays", "closest_nodes", "closest_tris", "any_nodes", "any_tris", "primary_hit_hash"):
                assert getattr(r.stats, k) == getattr(base.stats, k), (mode, kw, k)
    assert base.stats.ray_count == o_st.ray_count and base.stats.closest_nodes == o_st.closest_nodes
    dev.close()
