"""Both shadow-ray stages (DESIGN.md §4, "Shadow rays") against the oracle and float64 references.

* One path per lane (`k_trace_shadow`): a lane traces its path's lights one after another, the fold fused in.
* One ray per lane (`k_trace_shadow_rays` + `k_shadow_fold`): (shading position, light) pairs, light-major in chunks of 64
  positions; an occluded ray clears its bit in `sh_mask`, and the fold adds the surviving lights in light order.

`yk_render` takes one ray per lane on scenes with >= 2 lights and >= 2^18 shapes, else one path per lane; `yk_occluded` and
`yk_query_occluded` take the per-ray kernel. `YK_SHADOW_MODE` (read when a context is created) forces 1 = one ray per lane or
0 = one path per lane. Every GPU test here renders in both forced modes and requires the oracle's bits from each, so the
two kernels are pinned to each other and to the reference.

As in test_render_limits.py, every case has a CPU part that checks on the oracle that the scene reaches what it is meant to
exercise (a later change to a scene must not make the GPU part pass vacuously), and a GPU part.
"""
import numpy as np
import pytest

from test_oracle_geometry import _pixel_centre_hits, _quad_scene
from test_ray_queries import _grid_scene, _random_rays, corner_case_rays
from test_render_limits import _assert_parity, closed_box, glass_plates, white_box
from test_sphere import sphere_field, sphere_scene
from yuki_b200 import api, desc as D, scenes

PER_RAY, PER_PATH, DEFAULT = 1, 0, -1
FORCED = (PER_RAY, PER_PATH)


@pytest.fixture(scope="module")
def mode_ctx():
    """One context per shadow mode: YK_SHADOW_MODE=1, =0 and unset. A context keeps the mode it was created with."""
    ctxs = {}
    try:
        with pytest.MonkeyPatch.context() as mp:
            for mode in (PER_RAY, PER_PATH, DEFAULT):
                if mode == DEFAULT:
                    mp.delenv("YK_SHADOW_MODE", raising=False)
                else:
                    mp.setenv("YK_SHADOW_MODE", str(mode))
                ctxs[mode] = api.Context(0)
        yield ctxs
    finally:
        for c in ctxs.values():
            c.close()


# ---- rendering in several modes ----------------------------------------------------------------------------------
def _render(ctx, scene, cam, film, smp, integ, tiles=None, film_in=None, host=None, **kw):
    dev = api.Scene(ctx, scene, host=host)
    try:
        rn = api.Renderer(ctx)
        if film.accumulate:
            out = np.zeros((film.res[1], film.res[0], 3), np.float32) if film_in is None else film_in.copy()
            return rn.render(dev, cam, film, smp, integ, tiles=tiles, film_out=out, **kw)
        return rn.render(dev, cam, film, smp, integ, tiles=tiles, want_hit_ids=True, **kw)
    finally:
        dev.close()


def _oracle(oracle, scene, cam, film, smp, integ, tiles=None, film_in=None):
    if film.accumulate:
        # one thread: a pixel's samples are added in tile-list order, as the library does; worker threads would add a
        # tile's copies at different sample indices in whatever order they finish
        out = np.zeros((film.res[1], film.res[0], 3), np.float32) if film_in is None else film_in.copy()
        return oracle.OracleScene(scene).render(cam, film, smp, integ, tiles=tiles, film_out=out, threads=1)
    return oracle.OracleScene(scene).render(cam, film, smp, integ, tiles=tiles, want_hit_ids=True)


def _assert_ran_both_kernels(r1, r0, scene, what=""):
    """The per-ray mode launches one more kernel (the fold) per bounce iteration than the per-path mode, and only when the
    scene has lights (render.cu: the shadow stage). A forced mode that did not take effect fails here."""
    assert r1.stats.trace_closest_launches == r0.stats.trace_closest_launches > 0, what
    extra = r1.stats.trace_closest_launches if scene.lights else 0
    assert r1.stats.kernel_launches - r0.stats.kernel_launches == extra, what


def _both_modes(mode_ctx, oracle, scene, cam, film, smp, integ, tiles=None, film_in=None, what="", **kw):
    """Renders in both forced modes; each must equal the oracle in film bits, hit ids and every counter."""
    o = _oracle(oracle, scene, cam, film, smp, integ, tiles, film_in)
    rs = {m: _render(mode_ctx[m], scene, cam, film, smp, integ, tiles, film_in, **kw) for m in FORCED}
    for m, r in rs.items():
        _assert_parity(r, o, (what, "mode", m))
    _assert_ran_both_kernels(rs[PER_RAY], rs[PER_PATH], scene, what)
    return rs, o


# ---- scenes --------------------------------------------------------------------------------------------------------
def _plus_point_light(scene_cam, pos=(-0.4, 0.5, 0.3), intensity=(0.2, 0.25, 0.3)):
    from yuki_b200 import transforms as xf
    scene, cam = scene_cam
    scene.lights.append(D.Light(D.LIGHT_POINT, xf.translation(pos), intensity))
    return scene, cam


def _sky_camera(scene_cam):
    """open_scene seen looking up into the sky: every camera ray misses, so every bounce's shading queue is empty."""
    scene, _ = scene_cam
    return scene, D.CameraParameters((0.0, 0.9, 2.6), (0.0, 5.0, 2.7), fov_axis=D.FOV_X, fov_deg=30.0)


def _leaf_counts(scene):
    from oracle import oracle as O
    nodes = O.OracleScene(scene).nodes()
    return nodes["shape_count"][nodes["is_leaf"] != 0]


# ---- the cases: (id, scene builder, film, sampler, integrator, GPU render options, CPU claim) --------------------------
# A claim gets (scene, oracle film, oracle ids, oracle stats) and checks that the case exercises what its id says.
def _claim_lit(scene, img, ids, st):
    assert st.shadow_rays > 0 and float(img.max()) > 0.0


def _claim_rect_light(scene, img, ids, st):
    _claim_lit(scene, img, ids, st)
    assert any(l.kind == D.LIGHT_RECT for l in scene.lights) and any(m.area_light >= 0 for m in scene.meshes)


def _claim_room(scene, img, ids, st):
    _claim_lit(scene, img, ids, st)
    assert {l.kind for l in scene.lights} == {D.LIGHT_POINT, D.LIGHT_SPOT, D.LIGHT_RECT}
    assert {m.kind for m in scene.materials} == {D.MAT_MATTE, D.MAT_GLASS, D.MAT_METAL, D.MAT_GLOSSY}
    assert any(t.kind == D.TEX_IMAGE for t in scene.textures)


def _claim_open(scene, img, ids, st):
    _claim_lit(scene, img, ids, st)
    assert any(l.kind == D.LIGHT_DISTANT for l in scene.lights) and (ids < 0).any() and any(scene.background)


def _claim_spheres(scene, img, ids, st):
    _claim_lit(scene, img, ids, st)
    assert (ids >= scene.n_triangles()).sum() > 20   # pixels whose camera ray hits a sphere


def _claim_leaf_7(scene, img, ids, st):
    _claim_lit(scene, img, ids, st)
    counts = _leaf_counts(scene)
    assert counts.max() == 7 and len(scene.lights) == 2   # packed leaf refs (at most 16 shapes), two lights


def _claim_leaf_40(scene, img, ids, st):
    _claim_lit(scene, img, ids, st)
    assert _leaf_counts(scene).max() > 16 and not scene.spheres   # the leaf table alone selects the generic kernels


def _claim_32_lights(scene, img, ids, st):
    _claim_lit(scene, img, ids, st)
    assert len(scene.lights) == 32


def _claim_emitting_walls(scene, img, ids, st):
    """Every wall is a rect light and that light's emissive triangles: each shadow ray's target light has triangles."""
    _claim_lit(scene, img, ids, st)
    assert len(scene.lights) == 6 and sorted(m.area_light for m in scene.meshes) == list(range(6))


def _claim_few_thousand_nodes(scene, img, ids, st):
    _claim_lit(scene, img, ids, st)
    assert len(scene.lights) == 32 and 1000 < st.ray_count / st.samples < 10000   # closest rays = tree nodes per sample


def _claim_nothing_seen(scene, img, ids, st):
    assert (ids < 0).all() and st.shadow_rays == 0 and st.ray_count == st.samples
    assert np.all(img == np.float32(scene.background))


def _claim_small_queue(scene, img, ids, st):
    _claim_lit(scene, img, ids, st)
    assert 0 < (ids >= 0).sum() < 64 and (ids >= 0).sum() % 64 != 0   # one sample per pixel: the first queue is below 64


def _claim_ragged_queue(scene, img, ids, st):
    _claim_lit(scene, img, ids, st)
    assert (ids >= 0).sum() > 64 and (ids >= 0).sum() % 64 != 0 and len(scene.lights) == 3


def _cases():
    from yuki_b200 import transforms as xf
    S2, S3 = D.SamplerType.stratified(2, 2), D.SamplerType.stratified(3, 3)
    P, W = D.IntegratorType.path, D.IntegratorType.whitted
    room_film = D.FilmSettings((96, 54), 16)
    return [
        # Path
        ("path-cornell-rect", lambda: scenes.cornell(xf, light="rect", tall_box="glass"), D.FilmSettings((64, 48), 16), S2, P(8), {}, _claim_rect_light),
        ("path-material-room", lambda: scenes.material_room(xf), room_film, S2, P(8), {}, _claim_room),
        ("path-open-scene", lambda: scenes.open_scene(xf), D.FilmSettings((96, 64), 16), S2, P(6), {}, _claim_open),
        ("path-sphere-scene", lambda: sphere_scene(xf), D.FilmSettings((64, 48), 16), S2, P(6), {}, _claim_spheres),
        ("path-sphere-field", lambda: sphere_field(xf, 40), D.FilmSettings((80, 48), 16), S2, P(6), {}, _claim_spheres),
        ("path-leaves-7", lambda: _plus_point_light(scenes.heightfield(xf, 40, 40, seed=5, split_method=D.SPLIT_SAH, max_shapes_in_node=7), (-3.0, 4.0, 2.0), (300.0, 250.0, 200.0)),
         D.FilmSettings((64, 48), 16), S2, P(5), {}, _claim_leaf_7),
        ("path-leaves-40", lambda: _plus_point_light(scenes.heightfield(xf, 40, 40, seed=5, split_method=D.SPLIT_EQUAL_COUNTS, max_shapes_in_node=40), (-3.0, 4.0, 2.0), (300.0, 250.0, 200.0)),
         D.FilmSettings((64, 48), 16), S2, P(5), {}, _claim_leaf_40),
        ("path-indirect-clamp", lambda: _plus_point_light(scenes.cornell(xf, light="rect", tall_box="glass"), (0.4, 0.3, -0.3), (0.05, 0.05, 0.05)),
         D.FilmSettings((64, 64), 16), D.SamplerType.stratified(4, 4), P(6, indirect_clamp=2.0), {}, _claim_rect_light),
        ("path-32-lights-depth-12", lambda: white_box(xf, n_lights=32), D.FilmSettings((32, 24), 16), S2, P(12), {}, _claim_32_lights),
        ("path-emitting-walls", lambda: (closed_box(xf, 0.5, le=1.5), D.CameraParameters((0.3, 0.2, 0.1), (-0.5, -0.3, -1.0), fov_deg=80.0)),
         D.FilmSettings((48, 32), 16), S2, P(5), {}, _claim_emitting_walls),
        # Whitted
        ("whitted-glass-cornell-point", lambda: scenes.cornell(xf, light="point", tall_box="glass"), D.FilmSettings((64, 64), 16), S2, W(3), {}, _claim_lit),
        ("whitted-glass-plates-32-lights", lambda: glass_plates(xf), D.FilmSettings((2, 2), 16), S2, W(14), {}, _claim_few_thousand_nodes),
        ("whitted-sphere-scene", lambda: sphere_scene(xf), D.FilmSettings((64, 48), 16), S2, W(3), {}, _claim_spheres),
        ("whitted-open-scene", lambda: scenes.open_scene(xf), D.FilmSettings((96, 64), 16), S2, W(4), {}, _claim_open),
        # shapes of the shading queue
        ("path-queue-below-64", lambda: scenes.cornell(xf, light="rect", tall_box="glass"), D.FilmSettings((5, 3), 16), D.SamplerType.uniform(1), P(8), {}, _claim_small_queue),
        ("path-queue-ragged", lambda: scenes.material_room(xf), D.FilmSettings((13, 11), 16), D.SamplerType.uniform(1), P(8), {}, _claim_ragged_queue),
        ("whitted-queue-ragged", lambda: scenes.material_room(xf), D.FilmSettings((13, 11), 16), D.SamplerType.uniform(1), W(5), {}, _claim_ragged_queue),
        ("path-many-batches", lambda: scenes.material_room(xf), D.FilmSettings((48, 32), 16), S2, P(8), {"wavefront_paths": 200}, _claim_room),
        ("whitted-many-batches", lambda: scenes.material_room(xf), D.FilmSettings((48, 32), 16), S2, W(5), {"wavefront_paths": 200}, _claim_room),
        ("path-empty-queue", lambda: _sky_camera(scenes.open_scene(xf)), D.FilmSettings((24, 16), 16), S2, P(4), {}, _claim_nothing_seen),
        ("whitted-empty-queue", lambda: _sky_camera(scenes.open_scene(xf)), D.FilmSettings((24, 16), 16), S2, W(4), {}, _claim_nothing_seen),
        # ordering: two pipes over many batches, shading positions in sorted order
        ("path-two-pipes-sort-2", lambda: scenes.material_room(xf), room_film, D.SamplerType.stratified(3, 2), P(8), {"pipes": 2, "ray_sort": 2, "wavefront_paths": 4096}, _claim_room),
        ("path-two-pipes-sort-3", lambda: scenes.material_room(xf), room_film, D.SamplerType.stratified(3, 2), P(8), {"pipes": 2, "ray_sort": 3, "wavefront_paths": 4096}, _claim_room),
        ("path-two-pipes-sort-3-trace-only", lambda: scenes.material_room(xf), room_film, D.SamplerType.stratified(3, 2), P(8), {"pipes": 2, "ray_sort": 3 | 16, "wavefront_paths": 4096}, _claim_room),
    ]


CASES = {c[0]: c[1:] for c in _cases()}


@pytest.mark.parametrize("case", list(CASES))
def test_case_exercises_what_it_names(oracle, case):
    build, film, smp, integ, _, claim = CASES[case]
    scene, cam = build()
    img, ids, st = _oracle(oracle, scene, cam, film, smp, integ)
    claim(scene, img, ids, st)
    if case == "path-indirect-clamp":   # the clamp bites: the unclamped film differs
        free, _, _ = _oracle(oracle, scene, cam, film, smp, D.IntegratorType.path(integ.max_depth))
        assert not np.array_equal(free.view(np.uint32), img.view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_gpu_both_modes_match_the_oracle(mode_ctx, oracle, case):
    build, film, smp, integ, kw, _ = CASES[case]
    scene, cam = build()
    _both_modes(mode_ctx, oracle, scene, cam, film, smp, integ, what=case, **kw)


# ---- 1. which kernel ran -------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_forced_modes_launch_the_kernels_they_name(mode_ctx, xf):
    film, smp = D.FilmSettings((32, 32), 16), D.SamplerType.stratified(2, 2)
    lit = scenes.cornell(xf, light="rect", tall_box="glass")
    dark = scenes.cornell(xf, light=None, tall_box="glass")
    for integ in (D.IntegratorType.path(6), D.IntegratorType.whitted(4)):
        for scene, cam in (lit, dark):
            r1, r0 = (_render(mode_ctx[m], scene, cam, film, smp, integ) for m in FORCED)
            assert r1.stats.trace_closest_launches == r0.stats.trace_closest_launches > 1
            want = r1.stats.trace_closest_launches if scene.lights else 0
            assert r1.stats.kernel_launches - r0.stats.kernel_launches == want, (integ.kind, len(scene.lights))
            assert np.array_equal(r1.film.view(np.uint32), r0.film.view(np.uint32))


# ---- 2. accumulating film, debug rays, queries ------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("integ", [D.IntegratorType.path(6), D.IntegratorType.whitted(4)], ids=["path", "whitted"])
def test_gpu_accumulating_film_in_both_modes(mode_ctx, oracle, xf, integ):
    """Sample indices 0 .. 3 added into a non-zero film, as the progressive renderer does."""
    scene, cam = scenes.material_room(xf)
    acc = D.FilmSettings((48, 32), 16, accumulate=True)
    smp = D.SamplerType.stratified(2, 2)
    base = api.film_tiles(acc)
    tiles = np.concatenate([base] * 4)
    tiles["sample"] = np.repeat(np.arange(4, dtype=np.uint16), len(base))
    film_in = np.random.default_rng(2).uniform(0.0, 1.0, (32, 48, 3)).astype(np.float32)
    rs, o = _both_modes(mode_ctx, oracle, scene, cam, acc, smp, integ, tiles=tiles, film_in=film_in, what="accumulate")
    assert not np.array_equal(o[0], film_in) and rs[PER_RAY].stats.shadow_rays > 0


DEBUG_FILM = D.FilmSettings((96, 96), 16)
DEBUG_PIXELS = [(48, 48), (10, 80), (70, 30), (95, 0), (33, 61), (52, 70)]


@pytest.mark.gpu
@pytest.mark.parametrize("smp,integ", [(D.SamplerType.stratified(3, 3), D.IntegratorType.path(8)),
                                       (D.SamplerType.stratified(2, 2), D.IntegratorType.whitted(5))], ids=["path", "whitted"])
def test_gpu_debug_rays_in_both_modes(mode_ctx, oracle, xf, smp, integ):
    scene, cam = scenes.material_room(xf)
    osc = oracle.OracleScene(scene)
    devs = {m: api.Scene(mode_ctx[m], scene) for m in FORCED}
    shadow = 0
    try:
        for px in DEBUG_PIXELS:
            o_rays, o_li, o_count = osc.debug_ray(cam, DEBUG_FILM, smp, integ, px)
            shadow += int((o_rays["ray_type"] == 4).sum())
            got = {m: api.Renderer(mode_ctx[m]).debug_ray(devs[m], cam, DEBUG_FILM, smp, integ, px) for m in FORCED}
            for m, (g_rays, g_li, g_count) in got.items():
                assert g_count == o_count and g_rays.tobytes() == o_rays.tobytes(), (px, m)
                if integ.kind == D.INTEGRATOR_PATH:
                    assert np.array_equal(g_li.view(np.uint32), o_li.view(np.uint32)), (px, m)
                else:  # Whitted: top-down pre-multiplied weights, the rounding difference documented in DESIGN.md §2
                    assert np.allclose(g_li, o_li, rtol=1e-5, atol=1e-7), (px, m)
            assert np.array_equal(got[PER_RAY][1].view(np.uint32), got[PER_PATH][1].view(np.uint32)), px
    finally:
        for d in devs.values():
            d.close()
    assert shadow > 0


def _query_cases(xf):
    rng = np.random.default_rng(21)
    hf = scenes.heightfield(xf, 64, 64, seed=9)[0]
    leaf_table = scenes.cornell(xf, light="rect", tall_box="glass", sphere=True, max_shapes_in_node=40)[0]
    out = [("heightfield", hf, *_random_rays(rng, 60000, (-0.7, -0.4, -0.7), (0.7, 0.6, 0.7))),
           ("sphere-field", sphere_field(xf, 60)[0], *_random_rays(rng, 30000, (-2.0, 0.0, -2.0), (2.0, 1.5, 2.0))),
           ("leaf-table", leaf_table, *_random_rays(rng, 30000, (0.0, 0.0, -0.56), (0.555, 0.55, 0.0)))]
    o, d, _ = corner_case_rays(6)
    out.append(("corner-cases", _grid_scene(xf, 6), o, d))
    return out


@pytest.mark.gpu
def test_gpu_occlusion_queries_in_both_modes(mode_ctx, oracle, xf):
    """yk_occluded (host arrays) and yk_query_occluded (torch CUDA tensors): mode 1 reads the answer from sh_mask, mode 0
    from the fused fold's L.x (wf_query.cuh)."""
    import torch
    for name, scene, o, d in _query_cases(xf):
        want = oracle.OracleScene(scene).occluded(o, d, t_max=np.full(len(o), 0.9999, np.float32))
        assert 0 < int(want.sum()) < len(o), name
        to, td = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
        for m in FORCED:
            dev = api.Scene(mode_ctx[m], scene)
            try:
                assert np.array_equal(dev.occluded(o, d), want), (name, m)
                got = dev.occluded(to, td)
                torch.cuda.synchronize()
                assert np.array_equal(got.cpu().numpy(), want), (name, m)
            finally:
                dev.close()


# ---- 3. float64 references ---------------------------------------------------------------------------------------------
OCCLUDER_CENTRE, OCCLUDER_HALF = np.array([0.2, -0.1]), 0.25
PLANE_FILM = D.FilmSettings((96, 72), 16)
PLANE_SAMPLER = D.SamplerType.stratified(1, 1, jitter=False)   # pixel centres
LIGHT_COUNTS = (1, 2, 31, 32)
# One term kd/pi * I * cos / d^2 evaluated in float32 from float32 inputs: about ten roundings of at most 2^-24 each
# (6e-7). The shading point is the float32 hit o + t*d, a few ulp (~1e-6 absolute) off the plane point computed here in
# float64; with d >= 1.5 and cos >= 0.4 that moves d^2 and cos by at most ~1e-5 relative. A sum of up to 32 positive terms
# adds at most 31 * 2^-24 = 2e-6 relative. So a pixel is within ~2e-5 of the float64 value; 1e-4 leaves a margin.
PLANE_RTOL = 1e-4
EDGE = 2e-3   # pixels whose segment to some light passes within this of the occluder's outline are left out


def lit_plane(k):
    """test_oracle_geometry's plane under a square occluder, lit by k point lights. Light 0 (when k > 1) and every 7th
    light lie below the plane, so their bit is never set; the others sit in a cluster above the occluder, so their shadows
    overlap in a region no light reaches. Returns the scene, camera and the light positions (float32 values)."""
    from yuki_b200 import transforms as xf
    scene, cam = _quad_scene()
    zero = scene.add_texture(D.Texture.constant(0.0))
    black = scene.add_material(D.Material(D.MAT_MATTE, (zero, zero)))
    c, h = OCCLUDER_CENTRE, OCCLUDER_HALF
    oc = np.array([(c[0] - h, c[1] - h, 1), (c[0] + h, c[1] - h, 1), (c[0] + h, c[1] + h, 1), (c[0] - h, c[1] + h, 1)], np.float32)
    scene.meshes.append(D.Mesh(xf.identity(), oc, np.array([0, 1, 2, 0, 2, 3], np.uint32), black))
    rng = np.random.default_rng(31)
    pos, inten = [], []
    for i in range(k):
        if k > 1 and i % 7 == 0:
            p = (rng.uniform(-0.8, 0.8), rng.uniform(-0.8, 0.8), -rng.uniform(0.3, 1.0))
        else:
            p = (0.55 + rng.uniform(-0.08, 0.08), 0.45 + rng.uniform(-0.08, 0.08), rng.uniform(1.9, 2.4))
        p = tuple(float(np.float32(v)) for v in p)
        i_rgb = tuple(float(np.float32(v)) for v in rng.uniform(0.2, 1.0, 3) * (3.0 / k))
        scene.lights.append(D.Light(D.LIGHT_POINT, xf.translation(p), i_rgb))
        pos.append(p)
        inten.append(i_rgb)
    return scene, cam, np.array(pos, np.float64), np.array(inten, np.float64)


def lit_plane_reference(oracle, k, ids):
    """float64 radiance of every pixel centre, and masks: pixels that see the plane away from its outline and from every
    light's shadow outline (`clean`), and among them those no light reaches (`dark`); plus the per-light visibility."""
    scene, cam, pos, inten = lit_plane(k)
    _, _, _, p, inside = _pixel_centre_hits(oracle, cam, PLANE_FILM)
    on_plane = inside & (ids >= 0) & (ids < 2)
    clean = on_plane & (np.abs(np.abs(p[..., 0]) - 1) > 1e-2) & (np.abs(np.abs(p[..., 1]) - 1) > 1e-2)
    want = np.zeros(p.shape, np.float64)
    vis = np.zeros(p.shape[:2] + (k,), bool)
    for j in range(k):
        lp = pos[j]
        if lp[2] <= 0.0:
            continue   # below the plane: cos < 0, no shadow ray
        s = (1.0 - p[..., 2]) / (lp[2] - p[..., 2])   # the segment p -> light crosses z = 1 here
        q = p + s[..., None] * (lp - p)
        dx, dy = np.abs(q[..., 0] - OCCLUDER_CENTRE[0]), np.abs(q[..., 1] - OCCLUDER_CENTRE[1])
        inner = (dx < OCCLUDER_HALF - EDGE) & (dy < OCCLUDER_HALF - EDGE)
        outer = (dx > OCCLUDER_HALF + EDGE) | (dy > OCCLUDER_HALF + EDGE)
        clean &= inner | outer
        vis[..., j] = outer
        to = lp - p
        d2 = (to ** 2).sum(axis=-1)
        cos = to[..., 2] / np.sqrt(d2)
        want += np.where(outer, cos / d2, 0.0)[..., None] * (0.5 / np.pi) * inten[j]
    dark = clean & ~vis.any(axis=-1)
    return want, clean, dark, vis, on_plane


def _check_lit_plane(img, want, clean, dark):
    lit = clean & ~dark
    assert np.all(np.abs(img[lit] - want[lit]) <= PLANE_RTOL * want[lit])
    assert np.all(img[dark] == 0.0)


@pytest.mark.parametrize("k", LIGHT_COUNTS)
def test_lit_plane_reaches_its_lights_and_the_oracle_matches_float64(oracle, k):
    scene, cam, pos, _ = lit_plane(k)
    osc = oracle.OracleScene(scene)
    img, ids, st = osc.render(cam, PLANE_FILM, PLANE_SAMPLER, D.IntegratorType.path(1), want_hit_ids=True)
    img_w, _, _ = osc.render(cam, PLANE_FILM, PLANE_SAMPLER, D.IntegratorType.whitted(1))
    assert np.array_equal(img.view(np.uint32), img_w.view(np.uint32))
    want, clean, dark, vis, on_plane = lit_plane_reference(oracle, k, ids)
    above = pos[:, 2] > 0
    # one shadow ray per (plane hit, light above the plane); none towards the lights below, none from the black occluder
    assert st.shadow_rays == int(on_plane.sum()) * int(above.sum())
    assert clean.sum() > 1000 and dark.sum() > 50 and (clean & ~dark).sum() > 1000
    if k > 1:
        assert not above[0]
    if k == 32:   # light 31, the top bit of the mask, both lights some pixels and is blocked at others
        assert (clean & vis[..., 31]).sum() > 200 and (clean & ~vis[..., 31]).sum() > 200
    _check_lit_plane(img, want, clean, dark)


@pytest.mark.gpu
@pytest.mark.parametrize("k", LIGHT_COUNTS)
def test_gpu_lit_plane_matches_float64_and_the_oracle(mode_ctx, oracle, k):
    scene, cam, _, _ = lit_plane(k)
    for integ in (D.IntegratorType.path(1), D.IntegratorType.whitted(1)):
        rs, o = _both_modes(mode_ctx, oracle, scene, cam, PLANE_FILM, PLANE_SAMPLER, integ, what=("plane", k))
        want, clean, dark, _, _ = lit_plane_reference(oracle, k, o[1])
        for m in FORCED:
            _check_lit_plane(rs[m].film, want, clean, dark)


EMITTING_BOX_DEPTHS = (1, 2, 5, 40)


@pytest.mark.gpu
@pytest.mark.parametrize("depth", EMITTING_BOX_DEPTHS)
def test_gpu_emitting_box_matches_the_closed_form(mode_ctx, oracle, xf, depth):
    """test_render_limits' closed form Le * (1 + a * (1 - a^d) / (1 - a)) in the box whose six walls are rect lights."""
    a, le = 0.5, 1.5
    scene = closed_box(xf, a, le=le)
    cam = D.CameraParameters((0.0, 0.0, 0.0), (0.0, 0.0, -1.0), fov_deg=60.0)
    film, smp = D.FilmSettings((128, 128), 16), D.SamplerType.stratified(4, 4)
    rs, _ = _both_modes(mode_ctx, oracle, scene, cam, film, smp, D.IntegratorType.path(depth), what=("box", depth))
    px = np.asarray(rs[PER_RAY].film, np.float64)[..., 0].ravel()
    want = le * (1.0 + a * (1.0 - a ** depth) / (1.0 - a))
    assert abs(px.mean() - want) <= 6.0 * px.std() / np.sqrt(px.size), (px.mean(), want)


# ---- 4. the selection rule at its boundary -------------------------------------------------------------------------------
BOUNDARY_FILM = D.FilmSettings((32, 24), 16)


def boundary_scenes(xf):
    """scenes.heightfield at 256 x 512 quads: exactly 2^18 triangles. (scene, camera, the mode the default picks)."""
    def second_light(s):
        s.lights.append(D.Light(D.LIGHT_POINT, xf.translation((-4.0, 5.0, 2.0)), (300.0, 200.0, 250.0)))
        return s
    at, cam = scenes.heightfield(xf, 256, 512)
    below, _ = scenes.heightfield(xf, 256, 512)
    below.meshes[0].indices = below.meshes[0].indices[:-3]
    one_light, _ = scenes.heightfield(xf, 256, 512)
    return [("2^18-shapes-2-lights", second_light(at), cam, PER_RAY),
            ("2^18-1-shapes-2-lights", second_light(below), cam, PER_PATH),
            ("2^18-shapes-1-light", one_light, cam, PER_PATH)]


def test_boundary_scenes_sit_on_the_threshold(xf):
    counts = [(s.n_triangles(), len(s.lights)) for _, s, _, _ in boundary_scenes(xf)]
    assert counts == [(1 << 18, 2), ((1 << 18) - 1, 2), (1 << 18, 1)]


@pytest.mark.gpu
def test_gpu_default_mode_follows_the_rule_at_2_to_the_18_shapes(mode_ctx, oracle, xf):
    smp, integ = D.SamplerType.stratified(2, 2), D.IntegratorType.path(4)
    for name, scene, cam, picked in boundary_scenes(xf):
        host = api.HostScene(scene)
        try:
            rs = {m: _render(mode_ctx[m], scene, cam, BOUNDARY_FILM, smp, integ, host=host) for m in (PER_RAY, PER_PATH, DEFAULT)}
        finally:
            host.close()
        o = _oracle(oracle, scene, cam, BOUNDARY_FILM, smp, integ)
        for m, r in rs.items():
            _assert_parity(r, o, (name, m))
        _assert_ran_both_kernels(rs[PER_RAY], rs[PER_PATH], scene, name)
        assert rs[DEFAULT].stats.kernel_launches == rs[picked].stats.kernel_launches, name
        assert rs[DEFAULT].stats.shadow_rays > 0, name
