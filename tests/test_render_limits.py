"""Renders at the limits `yk_render` admits (render.cu: Path max_depth 255, Whitted 24, 32 lights, 65536 spp), compared
with the oracle bit for bit.

Each case comes in two parts. The CPU part runs on the oracle and checks that the scene really reaches the limit it is
meant to test, so that a later change to a scene cannot make the GPU part pass vacuously. The GPU part compares film bits,
hit ids, ray counts, shadow rays and the traversal counters with the oracle.

Ends of the device code these cases reach and no other test does:
* Path's 8-bit bounce counter full at bounce 255, with roulette continuing at 0.95 (an albedo-1 box).
* The per-group table of stratified hashes (render.cu) ending inside a path: at the 4096-dimension cap (32 lights, bounce
  62), and at 2^26 / jobs-in-group dimensions for a large pixel group.
* Whitted trees of more than 2^15 nodes with 32 lights, whose sampler dimensions pass 2^21, and trees that outgrow the
  8 levels the hash table covers for Whitted.
* More than 1024 samples per pixel: a pixel's samples split over several batches (kMaxBatchSamples, wf_raygen.cuh).
"""
import numpy as np
import pytest

from yuki_b200 import api, capi, desc as D, scenes

COUNTERS = ("ray_count", "shadow_rays", "closest_nodes", "closest_tris", "any_nodes", "any_tris")

# ---- scenes ------------------------------------------------------------------------------------------------
# The six walls of the cube [-1, 1]^3: inward normal and the two axes spanning the wall.
WALLS = [((0, -1, 0), 0, 2), ((0, 1, 0), 0, 2), ((-1, 0, 0), 1, 2), ((1, 0, 0), 1, 2), ((0, 0, -1), 0, 1), ((0, 0, 1), 0, 1)]


def _wall(n, a, b, half=(1.0, 1.0, 1.0)):
    """The wall of the box [-half, half] with inward normal n, wound so that its geometric normal is n."""
    pts = []
    for sa, sb in ((-1, -1), (1, -1), (1, 1), (-1, 1)):
        p = -np.asarray(n, np.float32)
        p[a], p[b] = sa, sb
        pts.append(p * np.float32(half))
    pts = np.array(pts, np.float32)
    idx = (0, 1, 2, 0, 2, 3) if np.dot(np.cross(pts[0] - pts[2], pts[1] - pts[2]), n) > 0 else (0, 2, 1, 0, 3, 2)
    return pts, np.array(idx, np.uint32)


def _wall_light(xf, n):
    """Light-to-world of a 2 x 2 rect light (light space: the xz plane, emitting along -y) on the cube wall with inward normal n."""
    half = float(np.float32(np.pi / 2))
    for r in (xf.identity(), xf.rotation(float(np.float32(np.pi)), (1.0, 0.0, 0.0)), xf.rotation(half, (0.0, 0.0, 1.0)),
              xf.rotation(-half, (0.0, 0.0, 1.0)), xf.rotation(half, (1.0, 0.0, 0.0)), xf.rotation(-half, (1.0, 0.0, 0.0))):
        if np.allclose(xf.vec(r, (0.0, -1.0, 0.0)), n, atol=1e-6):
            return xf.mul(xf.translation(tuple(float(-v) for v in n)), r)
    raise AssertionError(n)


def closed_box(xf, albedo, le=None, lights=(), half=(1.0, 1.0, 1.0)):
    """Six Matte walls of the given albedo. With `le`, every wall is also an inward-facing rect light of radiance le
    (only for the unit cube)."""
    s = D.SceneDesc()
    zero = s.add_texture(D.Texture.constant(0.0))
    m = s.add_material(D.Material(D.MAT_MATTE, (s.add_texture(D.Texture.constant(albedo)), zero)))
    for n, a, b in WALLS:
        pts, idx = _wall(n, a, b, half)
        al = -1
        if le is not None:
            al = len(s.lights)
            s.lights.append(D.Light(D.LIGHT_RECT, _wall_light(xf, n), (le,) * 3, size=(2.0, 2.0)))
        s.meshes.append(D.Mesh(xf.identity(), pts, idx, m, area_light=al))
    s.lights += list(lights)
    return s


def white_box(xf, n_lights=1):
    """An albedo-1 box with point lights inside: Lambert with cosine sampling keeps beta.g at 1, so from bounce 4 on
    roulette continues with probability 0.95."""
    rng = np.random.default_rng(7)
    lights = [D.Light(D.LIGHT_POINT, xf.translation((0.3, 0.5, -0.2)), (1.0, 1.0, 1.0))]
    while len(lights) < n_lights:
        pos = tuple(float(v) for v in rng.uniform(-0.8, 0.8, 3))
        lights.append(D.Light(D.LIGHT_POINT, xf.translation(pos), tuple(float(v) for v in rng.uniform(0.02, 0.1, 3))))
    cam = D.CameraParameters((0.0, 0.0, 0.5), (0.0, 0.0, -1.0), fov_deg=60.0)
    return closed_box(xf, 1.0, lights=lights), cam


def glass_plates(xf, n_plates=6, n_lights=32):
    """Parallel glass plates seen near normal incidence inside an 8 x 4 x 8 Matte room: both specular children exist at
    every face, so a Whitted tree grows like a power of the depth; the rays that leave the stack end on Matte walls lit by
    `n_lights` rect lights under the ceiling."""
    s = closed_box(xf, 0.6, half=(4.0, 2.0, 4.0))
    one = s.add_texture(D.Texture.constant(1.0))
    glass = s.add_material(D.Material(D.MAT_GLASS, (one, one), eta=1.5))
    for k in range(n_plates):
        z = np.float32(-1.0 - 0.1 * k)
        pts = np.array([(-1.5, -1.5, z), (1.5, -1.5, z), (1.5, 1.5, z), (-1.5, 1.5, z)], np.float32)
        s.meshes.append(D.Mesh(xf.identity(), pts, np.array((0, 1, 2, 0, 2, 3), np.uint32), glass))
    for k in range(n_lights):
        x, z = -3.0 + 6.0 * ((k % 8) + 0.5) / 8, -3.5 + 7.0 * ((k // 8) + 0.5) / 4
        s.lights.append(D.Light(D.LIGHT_RECT, xf.translation((x, 1.95, z)), (0.5, 0.5, 0.5), size=(0.3, 0.3)))
    cam = D.CameraParameters((0.05, 0.03, 1.5), (0.0, 0.0, -1.0), fov_deg=10.0)
    return s, cam


def one_pixel_tiles(film, picks):
    """Accumulate-mode tiles of one pixel each: (x, y, sample index)."""
    t = np.zeros(len(picks), capi.TILE_DTYPE)
    for k, (x, y, si) in enumerate(picks):
        t[k]["x0"], t[k]["y0"], t[k]["x1"], t[k]["y1"], t[k]["sample"] = x, y, x + 1, y + 1, si
    return t


# ---- pinned inputs ------------------------------------------------------------------------------------------
# (pixel x, pixel y, sample index) of white_box's 512 x 512 film at uniform(8) whose paths trace their 255th ray at
# max_depth 255. Found once by searching the oracle's ray counts (0.95^251: about 3 in 10^6 paths get that far).
DEEP_FILM = D.FilmSettings((512, 512), 16, accumulate=True)
DEEP_SAMPLER = D.SamplerType.uniform(8)
DEEP_PINS = [(322, 172, 1), (456, 337, 4), (251, 452, 2), (36, 88, 3), (481, 451, 4)]

WHITTED_CHAIN_DEPTHS = (7, 9, 16, 24)
LARGE_TREE_DEPTH = 19          # glass_plates: ~54 k nodes in one sample's tree
SMALL_TABLE_TREE_DEPTH = 14    # glass_plates with one light: ~2.9 k nodes, past the 255 nodes of Whitted's 8-level table


def _render_both(gpu_ctx, oracle, scene, cam, film, smp, integ, tiles=None, **kw):
    dev = api.Scene(gpu_ctx, scene)
    try:
        if film.accumulate:
            out = np.zeros((film.res[1], film.res[0], 3), np.float32)
            r = api.Renderer(gpu_ctx).render(dev, cam, film, smp, integ, tiles=tiles, film_out=out, **kw)
            o = oracle.OracleScene(scene).render(cam, film, smp, integ, tiles=tiles)
        else:
            r = api.Renderer(gpu_ctx).render(dev, cam, film, smp, integ, tiles=tiles, want_hit_ids=True, **kw)
            o = oracle.OracleScene(scene).render(cam, film, smp, integ, tiles=tiles, want_hit_ids=True)
    finally:
        dev.close()
    return r, o


def _assert_parity(r, o, what=""):
    o_img, o_ids, o_st = o
    assert np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32)), what
    if o_ids is not None:
        assert np.array_equal(r.hit_ids, o_ids), what
    for k in COUNTERS:
        assert getattr(r.stats, k) == getattr(o_st, k), (what, k)
    assert r.stats.samples == o_st.samples, what


def _oracle_rays(oracle, scene, cam, film, smp, integ, tiles=None):
    return oracle.OracleScene(scene).render(cam, film, smp, integ, tiles=tiles)[2].ray_count


# ---- 1. Path at max_depth 255 -------------------------------------------------------------------------------
def test_deep_path_pins_reach_bounce_255(oracle, xf):
    scene, cam = white_box(xf)
    osc = oracle.OracleScene(scene)
    for pin in DEEP_PINS:
        tiles = one_pixel_tiles(DEEP_FILM, [pin])
        assert osc.render(cam, DEEP_FILM, DEEP_SAMPLER, D.IntegratorType.path(255), tiles=tiles)[2].ray_count == 255, pin
        assert osc.render(cam, DEEP_FILM, DEEP_SAMPLER, D.IntegratorType.path(254), tiles=tiles)[2].ray_count == 254, pin


def test_deep_path_with_32_lights_crosses_the_4096_dimension_table(oracle, xf):
    """A Path bounce draws 2 * 32 + 3 dimensions after the camera's 2, so bounce 62 draws dimensions past
    2 + 61 * 67 = 4089 .. 4156: the hash table, at most 4096 dimensions, ends inside these paths whatever the film size."""
    scene, cam = white_box(xf, n_lights=32)
    film, smp = D.FilmSettings((24, 24), 16), D.SamplerType.stratified(2, 2)
    assert _oracle_rays(oracle, scene, cam, film, smp, D.IntegratorType.path(80)) > _oracle_rays(oracle, scene, cam, film, smp, D.IntegratorType.path(62))


@pytest.mark.gpu
def test_gpu_deep_path_matches_the_oracle(gpu_ctx, oracle, xf):
    scene, cam = white_box(xf)
    r, o = _render_both(gpu_ctx, oracle, scene, cam, DEEP_FILM, DEEP_SAMPLER, D.IntegratorType.path(255),
                        tiles=one_pixel_tiles(DEEP_FILM, DEEP_PINS))
    assert o[2].ray_count >= 255 * len(DEEP_PINS) and float(o[0].max()) > 0.0
    _assert_parity(r, o, "pinned deep paths")
    r, o = _render_both(gpu_ctx, oracle, scene, cam, D.FilmSettings((64, 48), 16), D.SamplerType.stratified(2, 2), D.IntegratorType.path(255))
    _assert_parity(r, o, "full film at depth 255")
    scene, cam = white_box(xf, n_lights=32)
    r, o = _render_both(gpu_ctx, oracle, scene, cam, D.FilmSettings((24, 24), 16), D.SamplerType.stratified(2, 2), D.IntegratorType.path(80))
    _assert_parity(r, o, "32 lights at depth 80")


# ---- 2. hash table bounded by the group size ----------------------------------------------------------------
TABLE_FILM = D.FilmSettings((1024, 1024), 16)
TABLE_SAMPLER = D.SamplerType.stratified(2, 1)
TABLE_DEPTH = 16


def _table_case(xf):
    """1024 x 1024 pixels at 2 spp with wavefront_paths = 2^21 and one pipe: 2 samples per batch, one group of 2^20 jobs,
    so the table holds 2^26 / 2^20 = 64 dimensions. white_box has one light, so a Path bounce draws 2 + 3 dimensions and
    bounce 12 draws dimensions 62 .. 66: every path that gets that far crosses from the table to the hash. (Depth 16 needs
    2 + 16 * 5 = 82 dimensions; the comparison render with groups of 2^16 jobs tabulates all of them.)"""
    scene, cam = white_box(xf)
    return scene, cam, api.film_tiles(TABLE_FILM)[::64]


def test_table_case_paths_reach_bounce_12(oracle, xf):
    scene, cam, tiles = _table_case(xf)
    deep = _oracle_rays(oracle, scene, cam, TABLE_FILM, TABLE_SAMPLER, D.IntegratorType.path(TABLE_DEPTH), tiles)
    assert deep > _oracle_rays(oracle, scene, cam, TABLE_FILM, TABLE_SAMPLER, D.IntegratorType.path(12), tiles)


@pytest.mark.gpu
def test_gpu_hash_table_edge_inside_a_path(gpu_ctx, oracle, xf):
    scene, cam, tiles = _table_case(xf)
    integ = D.IntegratorType.path(TABLE_DEPTH)
    dev = api.Scene(gpu_ctx, scene)
    rn = api.Renderer(gpu_ctx)
    big = rn.render(dev, cam, TABLE_FILM, TABLE_SAMPLER, integ, wavefront_paths=1 << 21, pipes=1)
    small = rn.render(dev, cam, TABLE_FILM, TABLE_SAMPLER, integ, wavefront_paths=1 << 16, pipes=1)
    dev.close()
    assert np.array_equal(big.film.view(np.uint32), small.film.view(np.uint32))
    for k in COUNTERS:
        assert getattr(big.stats, k) == getattr(small.stats, k), k
    o_img, _, _ = oracle.OracleScene(scene).render(cam, TABLE_FILM, TABLE_SAMPLER, integ, tiles=tiles)
    covered = np.zeros((1024, 1024), bool)
    for t in tiles:
        covered[t["y0"]:t["y1"], t["x0"]:t["x1"]] = True
    assert np.array_equal(big.film[covered].view(np.uint32), o_img[covered].view(np.uint32))


# ---- 3. deep Whitted chains ---------------------------------------------------------------------------------
WHITTED_FILM = D.FilmSettings((48, 48), 16)


def test_whitted_chains_reach_depth_24(oracle, xf):
    """Inside the glass box the reflection child goes on until the depth limit: depth 24 traces more rays than 23."""
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    smp = D.SamplerType.stratified(2, 2)
    assert _oracle_rays(oracle, scene, cam, WHITTED_FILM, smp, D.IntegratorType.whitted(24)) > \
        _oracle_rays(oracle, scene, cam, WHITTED_FILM, smp, D.IntegratorType.whitted(23))


@pytest.mark.gpu
@pytest.mark.parametrize("depth", WHITTED_CHAIN_DEPTHS)
def test_gpu_deep_whitted_chains_match_the_oracle(gpu_ctx, oracle, xf, depth):
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    r, o = _render_both(gpu_ctx, oracle, scene, cam, WHITTED_FILM, D.SamplerType.stratified(2, 2), D.IntegratorType.whitted(depth))
    _assert_parity(r, o, depth)


# ---- 4. large Whitted trees ---------------------------------------------------------------------------------
LARGE_TREE_FILM = D.FilmSettings((1, 1), 16)


def test_large_whitted_tree_passes_2_to_the_21_dimensions(oracle, xf):
    """Every node draws one get_2d per light: with 32 lights node n starts at dimension 2 + 64 n, past 2^21 from node
    32768 on. One sample's tree (one closest-hit ray per node) is larger than that."""
    scene, cam = glass_plates(xf)
    acc = D.FilmSettings((1, 1), 16, accumulate=True)
    rays = _oracle_rays(oracle, scene, cam, acc, D.SamplerType.stratified(2, 2), D.IntegratorType.whitted(LARGE_TREE_DEPTH),
                        one_pixel_tiles(acc, [(0, 0, 0)]))
    assert 40000 < rays < 200000


def test_whitted_tree_outgrows_the_8_level_table(oracle, xf):
    """With one light the table covers 2 + 2 * 255 dimensions (8 tree levels): a tree of more than 255 nodes crosses to
    the on-the-fly hash."""
    scene, cam = glass_plates(xf, n_lights=1)
    acc = D.FilmSettings((1, 1), 16, accumulate=True)
    rays = _oracle_rays(oracle, scene, cam, acc, D.SamplerType.stratified(2, 2), D.IntegratorType.whitted(SMALL_TABLE_TREE_DEPTH),
                        one_pixel_tiles(acc, [(0, 0, 0)]))
    assert rays > 255


@pytest.mark.gpu
@pytest.mark.parametrize("smp", [D.SamplerType.stratified(2, 2), D.SamplerType.uniform(4)], ids=["stratified", "uniform"])
def test_gpu_large_whitted_trees_match_the_oracle(gpu_ctx, oracle, xf, smp):
    scene, cam = glass_plates(xf)
    r, o = _render_both(gpu_ctx, oracle, scene, cam, LARGE_TREE_FILM, smp, D.IntegratorType.whitted(LARGE_TREE_DEPTH))
    _assert_parity(r, o, "32 lights")


@pytest.mark.gpu
def test_gpu_whitted_tree_past_the_8_level_table(gpu_ctx, oracle, xf):
    scene, cam = glass_plates(xf, n_lights=1)
    r, o = _render_both(gpu_ctx, oracle, scene, cam, D.FilmSettings((4, 4), 16), D.SamplerType.stratified(2, 2),
                        D.IntegratorType.whitted(SMALL_TABLE_TREE_DEPTH))
    _assert_parity(r, o, "1 light")


# ---- 5. more than 1024 samples per pixel --------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("res,smp", [((3, 2), D.SamplerType.uniform(1025)), ((2, 2), D.SamplerType.stratified(33, 32)),
                                     ((2, 2), D.SamplerType.stratified(33, 32, jitter=False)), ((2, 1), D.SamplerType.uniform(65536))],
                         ids=["uniform-1025", "stratified-33x32", "stratified-33x32-no-jitter", "uniform-65536"])
def test_gpu_samples_split_over_batches_match_the_oracle(gpu_ctx, oracle, xf, res, smp):
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    film = D.FilmSettings(res, 16)
    r, o = _render_both(gpu_ctx, oracle, scene, cam, film, smp, D.IntegratorType.path(5))
    _assert_parity(r, o, smp)
    assert r.stats.samples == res[0] * res[1] * smp.samples_per_pixel()


@pytest.mark.gpu
def test_gpu_batch_sample_override_leaves_the_film_unchanged(gpu_ctx, xf, monkeypatch):
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    film, smp, integ = D.FilmSettings((5, 3), 16), D.SamplerType.stratified(33, 32), D.IntegratorType.path(5)
    dev = api.Scene(gpu_ctx, scene)
    rn = api.Renderer(gpu_ctx)
    base = rn.render(dev, cam, film, smp, integ)
    for m in ("7", "1000"):
        monkeypatch.setenv("YK_MAX_BATCH_SAMPLES", m)
        r = rn.render(dev, cam, film, smp, integ)
        assert np.array_equal(r.film.view(np.uint32), base.film.view(np.uint32)), m
        assert r.stats.ray_count == base.stats.ray_count and r.stats.samples == base.stats.samples, m
    dev.close()


@pytest.mark.gpu
def test_gpu_many_groups_on_two_pipes_with_split_samples(gpu_ctx, oracle, xf):
    """512 x 288 pixels at 1056 spp with wavefront_paths = 2^20: 16 samples per batch (16 * 65536 <= 2^20), four groups
    of 36864 jobs that alternate between two pipes, 66 batches per group. Tiles from each group are compared with the
    oracle, the whole film with a one-pipe render."""
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    film, smp, integ = D.FilmSettings((512, 288), 16), D.SamplerType.stratified(33, 32), D.IntegratorType.path(3)
    tiles = api.film_tiles(film)
    pick = tiles[[0, 200, 400, len(tiles) - 1]]  # 144 tiles per group
    dev = api.Scene(gpu_ctx, scene)
    rn = api.Renderer(gpu_ctx)
    two = rn.render(dev, cam, film, smp, integ, wavefront_paths=1 << 20, pipes=2)
    one = rn.render(dev, cam, film, smp, integ, wavefront_paths=1 << 20, pipes=1)
    dev.close()
    assert two.stats.samples == 512 * 288 * 1056
    assert np.array_equal(two.film.view(np.uint32), one.film.view(np.uint32))
    for k in COUNTERS:
        assert getattr(two.stats, k) == getattr(one.stats, k), k
    o_img, _, _ = oracle.OracleScene(scene).render(cam, film, smp, integ, tiles=pick)
    for t in pick:
        sl = (slice(t["y0"], t["y1"]), slice(t["x0"], t["x1"]))
        assert np.array_equal(two.film[sl].view(np.uint32), o_img[sl].view(np.uint32)), t


# ---- 6. refusals --------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_depth_limits_are_enforced(gpu_ctx, xf):
    scene, cam = scenes.cornell(xf, light="rect", tall_box="glass")
    film, smp = D.FilmSettings((4, 4), 16), D.SamplerType.uniform(1)
    dev = api.Scene(gpu_ctx, scene)
    rn = api.Renderer(gpu_ctx)
    for integ in (D.IntegratorType.path(256), D.IntegratorType.whitted(25)):
        with pytest.raises(capi.YukiGpuError, match="max_depth"):
            rn.render(dev, cam, film, smp, integ)
    for integ in (D.IntegratorType.path(255), D.IntegratorType.whitted(24)):
        assert rn.render(dev, cam, film, smp, integ).stats.samples == 16
    dev.close()


# ---- 7. closed form ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("depth", [1, 2, 5, 40])
def test_oracle_path_matches_the_closed_form_in_an_emitting_box(oracle, xf, depth):
    """Six inward-facing rect lights of radiance Le that are also Matte walls of albedo a. Path counts emission at bounce 0
    only, and next-event estimation at each of the d vertices sees emitters over the whole hemisphere (a * Le in
    expectation), so a pixel's expected value is Le * (1 + a * (1 - a^d) / (1 - a)). The camera sees the middle of one
    wall, so the first vertex stays away from the edges, where area sampling of the neighbouring wall is heavy-tailed."""
    a, le = 0.5, 1.5
    scene = closed_box(xf, a, le=le)
    cam = D.CameraParameters((0.0, 0.0, 0.0), (0.0, 0.0, -1.0), fov_deg=60.0)
    img, _, _ = oracle.OracleScene(scene).render(cam, D.FilmSettings((128, 128), 16), D.SamplerType.stratified(4, 4),
                                                 D.IntegratorType.path(depth))
    px = np.asarray(img, np.float64)
    assert np.all(px[..., 0] == px[..., 1]) and np.all(px[..., 1] == px[..., 2])
    px = px[..., 0].ravel()
    want = le * (1.0 + a * (1.0 - a ** depth) / (1.0 - a))
    tol = 6.0 * px.std() / np.sqrt(px.size)
    assert abs(px.mean() - want) <= tol, (px.mean(), want, tol)
