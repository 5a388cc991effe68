"""yk_trace / yk_occluded: BoundingVolumeHierarchy::intersect / any_intersect (bvh.rs:160-302) called directly on ray
batches, against the oracle's Scene::intersect / any_intersect on the same rays — hit distance bits, original shape ids
and the per-ray (tests, hits) node counters. Unlike camera rays these batches are incoherent and include the slab /
triangle tests' corner cases: zero direction components (infinite inv_dir, NaN products), negative zeros, origins on box
planes and mesh vertices, rays in a triangle's plane or through shared edges (the f64 edge-function fallback,
triangle.rs:98-105), t_max equal to the hit distance (accepted, triangle.rs:126-130), t_max = 0, huge and tiny scales."""
import ctypes as C

import numpy as np
import pytest

from yuki_b200 import api, capi, desc as D, scenes
from test_sphere import sphere_field

SPLITS = [D.SPLIT_SAH, D.SPLIT_MIDDLE, D.SPLIT_EQUAL_COUNTS]


def _same(dev, osc, o, d, t_max=None):
    t, ids, cnt = dev.intersect(o, d, t_max)
    ot, oids, ocnt = osc.trace(o, d, t_max)
    assert np.array_equal(ids, oids)
    # a NaN distance (a hit of a zero-length direction) has no defined payload: x86 produces 0xffc00000, the GPU 0x7fffffff
    assert np.array_equal(np.isnan(t), np.isnan(ot))
    assert np.array_equal(np.where(np.isnan(t), 0, t.view(np.uint32)), np.where(np.isnan(ot), 0, ot.view(np.uint32)))
    assert np.array_equal(cnt, ocnt)
    return t, ids


def _same_occluded(dev, osc, o, d):
    got = dev.occluded(o, d)
    want = osc.occluded(o, d, t_max=np.full(len(o), 0.9999, np.float32))
    assert np.array_equal(got, want)
    return got


def _random_rays(rng, n, lo, hi):
    o = rng.uniform(lo, hi, (n, 3)).astype(np.float32)
    tgt = rng.uniform(lo, hi, (n, 3)).astype(np.float32)
    return o, (tgt - o).astype(np.float32)


def test_query_symbols_reject_null_arguments():
    L = capi.lib()
    assert L.yk_trace(None, None, None, None, None, 4, None, None, None) != 0
    assert L.yk_occluded(None, None, None, None, 4, None) != 0
    assert b"null argument" in L.yk_last_error()


@pytest.mark.gpu
@pytest.mark.parametrize("split", SPLITS)
def test_incoherent_rays_on_a_mesh(gpu_ctx, oracle, xf, split):
    scene, _ = scenes.heightfield(xf, 64, 64, seed=9, split_method=split, max_shapes_in_node=1 + 3 * split)
    dev, osc = api.Scene(gpu_ctx, scene), oracle.OracleScene(scene)
    rng = np.random.default_rng(11 + split)
    o, d = _random_rays(rng, 60000, (-0.7, -0.4, -0.7), (0.7, 0.6, 0.7))
    t, ids = _same(dev, osc, o, d)
    assert (ids >= 0).sum() > 10000 and (ids < 0).sum() > 1000
    tm = rng.uniform(0.0, 1.5, len(o)).astype(np.float32)   # bounded rays: some hits now lie beyond t_max
    _same(dev, osc, o, d, tm)
    occ = _same_occluded(dev, osc, o, d)
    assert 0 < occ.sum() < len(occ)
    dev.close()


@pytest.mark.gpu
def test_incoherent_rays_on_spheres_and_large_leaves(gpu_ctx, oracle, xf):
    cases = [(sphere_field(xf, 60)[0], (-2.0, 0.0, -2.0), (2.0, 1.5, 2.0)),
             (scenes.cornell(xf, light="rect", tall_box="glass", sphere=True, max_shapes_in_node=7)[0], (0.0, 0.0, -0.56), (0.555, 0.55, 0.0))]
    for scene, lo, hi in cases:
        dev, osc = api.Scene(gpu_ctx, scene), oracle.OracleScene(scene)
        rng = np.random.default_rng(5)
        o, d = _random_rays(rng, 30000, lo, hi)
        _, ids = _same(dev, osc, o, d)
        assert (ids >= 0).sum() > 3000
        _same_occluded(dev, osc, o, d)
        dev.close()


def _grid_scene(xf, n=6):
    """An exact-coordinate mesh: an n x n grid of unit quads in the plane y = 0 plus a wall at x = n, all vertices on
    integers, so rays can be aimed exactly at vertices, shared edges and box planes."""
    s = D.SceneDesc(split_method=D.SPLIT_MIDDLE)
    zero = s.add_texture(D.Texture.constant(0.0))
    m = s.add_material(D.Material(D.MAT_MATTE, (s.add_texture(D.Texture.constant(0.5)), zero)))
    pts, idx = [], []
    for j in range(n + 1):
        for i in range(n + 1):
            pts.append((float(i), 0.0, float(j)))
    for j in range(n):
        for i in range(n):
            a, b, c, e = j * (n + 1) + i, j * (n + 1) + i + 1, (j + 1) * (n + 1) + i + 1, (j + 1) * (n + 1) + i
            idx += [a, b, c, a, c, e]
    s.meshes.append(D.Mesh(xf.identity(), np.array(pts, np.float32), np.array(idx, np.uint32), m))
    p, i = scenes._quad([(n, 0, 0), (n, 2, 0), (n, 2, n), (n, 0, n)])
    s.meshes.append(D.Mesh(xf.identity(), p, i, m))
    s.lights.append(D.Light(D.LIGHT_POINT, xf.translation((1.0, 3.0, 1.0)), (1.0, 1.0, 1.0)))
    return s


def corner_case_rays(n=6):
    """Rays at _grid_scene(xf, n)'s vertices, shared edges and box planes: (o, d, t_max) as float32 arrays."""
    o, d, tm = [], [], []
    inf = np.inf

    def add(oo, dd, t=inf):
        o.append(oo); d.append(dd); tm.append(t)

    for i in range(n + 1):
        for j in range(n + 1):
            add((i, 1.0, j), (0.0, -1.0, 0.0))            # straight down onto a vertex: two zero components, e == 0 fallback
            add((i, 1.0, j), (-0.0, -1.0, 0.0))           # the same with a negative zero (inv_dir = -inf)
            add((i + 0.5, 2.0, j), (0.0, -1.0, 0.0))      # onto a shared edge
            add((i, 1.0, j), (0.0, -1.0, 0.0), 1.0)       # t_max exactly the hit distance: accepted
            add((i, 1.0, j), (0.0, -1.0, 0.0), np.float32(1.0) - np.float32(2.0 ** -24))  # one ulp short: rejected
            add((i, -1.0, j), (0.0, 1.0, 0.0))            # from below (back face)
            add((i, 0.0, j), (1.0, 0.0, 0.0))             # in the plane of the grid, origin on a vertex, towards the wall
            add((i + 0.25, 0.0, j + 0.25), (0.0, 0.0, 1.0))   # in the plane, inside a triangle
            add((i, 0.5, j), (1.0, 0.0, 0.0))             # parallel to the grid, origin on box planes, hits the wall
            add((i, 0.5, j), (1.0, 0.0, 0.0), 0.0)        # t_max = 0
            add((i, 0.5, j), (1e-30, 0.0, 0.0))           # tiny direction: t is huge
            add((i, 0.5, j), (1e30, 0.0, 0.0))            # huge direction: t is tiny
            add((i, 0.5, j), (-1.0, 0.0, 0.0))            # leaves the scene along a box plane
            add((i, 1.0, j), (1.0, -1.0, 1.0))            # diagonal through vertices / along quad diagonals
            add((i, 1.0, j), (1.0, -1.0, 0.0))
            add((i - 1e30, 1.0, j), (1.0, 0.0, 0.0))      # origin far outside: o + t d cancels catastrophically
    add((3.0, 1.0, 3.0), (0.0, 0.0, 0.0))                 # degenerate direction: every product is NaN or inf; no hit, same counters
    add((n, 1.0, 3.0), (0.0, 0.0, 1.0))                   # inside the wall's plane
    add((n, 1.0, 3.0), (1.0, 0.0, 0.0))                   # starts on the wall
    add((n, 1.0, 3.0), (-1.0, 0.0, 0.0))
    return np.array(o, np.float32), np.array(d, np.float32), np.array(tm, np.float32)


@pytest.mark.gpu
def test_corner_case_rays(gpu_ctx, oracle, xf):
    n = 6
    scene = _grid_scene(xf, n)
    dev, osc = api.Scene(gpu_ctx, scene), oracle.OracleScene(scene)
    o, d, tm = corner_case_rays(n)
    t, ids = _same(dev, osc, o, d, tm)
    assert (ids >= 0).sum() > 100
    _same_occluded(dev, osc, o, d)
    # the ABI's own argument checks
    bad_tm = tm.copy()
    bad_tm[3] = np.nan
    with pytest.raises(RuntimeError):
        dev.intersect(o, d, bad_tm)
    e_t, e_ids, _ = dev.intersect(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32))
    assert e_t.shape == (0,) and e_ids.shape == (0,)
    assert dev.occluded(np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32)).shape == (0,)
    dev.close()


@pytest.mark.gpu
def test_degenerate_directions_on_sphere_scenes_and_leaf_tables(gpu_ctx, oracle, xf):
    """A zero-length or NaN direction gives every triangle a NaN determinant, which the triangle test accepts
    (triangle.rs:109-130: every comparison is false) — the same signature the NaN vertex lanes of a sphere slot produce. The
    generic kernels (sphere slots and / or a leaf table, i.e. leaves of more than 16 shapes) must still tell the two apart:
    a triangle stays a triangle hit with t = NaN, as in the reference; only tagged slots reach the sphere test."""
    cases = [scenes.cornell(xf, light="rect", tall_box="glass", sphere=True)[0],
             scenes.cornell(xf, light="rect", tall_box="glass", sphere=True, max_shapes_in_node=40)[0],   # root leaf, spheres, leaf table
             scenes.heightfield(xf, 24, 24, seed=4, max_shapes_in_node=40)[0]]                            # leaf table, no spheres
    nan = np.nan
    for scene in cases:
        dev, osc = api.Scene(gpu_ctx, scene), oracle.OracleScene(scene)
        rng = np.random.default_rng(8)
        o, d = _random_rays(rng, 4000, (-0.6, -0.4, -0.6), (0.6, 0.6, 0.6))
        d[0::8] = 0.0                       # zero-length directions
        d[1::8, 0] = nan                    # one NaN component
        d[2::8] = (nan, nan, nan)
        d[3::8] = (0.0, -0.0, 0.0)
        o[4::8] = (0.3, 0.3, -0.3)          # inside the Cornell box (and on the heightfield's side)
        t, ids = _same(dev, osc, o, d)
        _same_occluded(dev, osc, o, d)
        # the renderer still works on this context afterwards (no poisoned CUDA context)
        assert dev.intersect(o[5:6], d[5:6])[0].shape == (1,)
        dev.close()


@pytest.mark.gpu
def test_batches_above_one_chunk_equal_small_batches(gpu_ctx, oracle, xf):
    """More rays than one internal chunk (2^22): the result is independent of how the batch is cut, and the renderer
    still works afterwards (the query reuses / replaces the wavefront state of pipe 0)."""
    scene, cam = scenes.heightfield(xf, 48, 48, seed=2)
    dev, osc = api.Scene(gpu_ctx, scene), oracle.OracleScene(scene)
    rng = np.random.default_rng(3)
    n = (1 << 22) + 12345
    o, d = _random_rays(rng, n, (-0.7, -0.4, -0.7), (0.7, 0.6, 0.7))
    t, ids, cnt = dev.intersect(o, d)
    occ = dev.occluded(o, d)
    for lo, hi in ((0, 3000), ((1 << 22) - 1500, (1 << 22) + 1500), (n - 3000, n)):
        st, sids, scnt = dev.intersect(o[lo:hi], d[lo:hi])
        assert np.array_equal(t[lo:hi].view(np.uint32), st.view(np.uint32)) and np.array_equal(ids[lo:hi], sids) and np.array_equal(cnt[lo:hi], scnt)
        assert np.array_equal(occ[lo:hi], dev.occluded(o[lo:hi], d[lo:hi]))
        ot, oids, ocnt = osc.trace(o[lo:hi], d[lo:hi])
        assert np.array_equal(st.view(np.uint32), ot.view(np.uint32)) and np.array_equal(sids, oids) and np.array_equal(scnt, ocnt)
    film = D.FilmSettings((64, 48), 16)
    r = api.Renderer(gpu_ctx).render(dev, cam, film, D.SamplerType.uniform(1), D.IntegratorType.bvh_intersections())
    o_img, _, _ = osc.render(cam, film, D.SamplerType.uniform(1), D.IntegratorType.bvh_intersections())
    assert np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32))
    dev.close()


@pytest.mark.gpu
def test_concurrent_callers_on_one_context_are_serialised(gpu_ctx, xf):
    """SURVEY.md §8b: several caller threads may use one context; the library serialises the calls that share its pipes.
    (ctypes drops the GIL during a call, so these really overlap.)"""
    import threading
    scene, cam = scenes.heightfield(xf, 48, 48, seed=2)
    dev = api.Scene(gpu_ctx, scene)
    rng = np.random.default_rng(6)
    o, d = _random_rays(rng, 400000, (-0.7, -0.4, -0.7), (0.7, 0.6, 0.7))
    film = D.FilmSettings((256, 192), 16)
    smp, integ = D.SamplerType.stratified(2, 2), D.IntegratorType.path(4)
    want_t, want_ids, want_cnt = dev.intersect(o, d)
    want_occ = dev.occluded(o, d)
    want_film = api.Renderer(gpu_ctx).render(dev, cam, film, smp, integ).film
    errors = []

    def queries():
        try:
            for _ in range(6):
                t, ids, cnt = dev.intersect(o, d)
                assert np.array_equal(t.view(np.uint32), want_t.view(np.uint32)) and np.array_equal(ids, want_ids) and np.array_equal(cnt, want_cnt)
                assert np.array_equal(dev.occluded(o, d), want_occ)
        except Exception as e:  # noqa: BLE001
            errors.append(e)

    def renders():
        try:
            rn = api.Renderer(gpu_ctx)
            for _ in range(6):
                assert np.array_equal(rn.render(dev, cam, film, smp, integ).film.view(np.uint32), want_film.view(np.uint32))
        except Exception as e:  # noqa: BLE001
            errors.append(e)

    threads = [threading.Thread(target=queries), threading.Thread(target=renders), threading.Thread(target=queries)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors
    dev.close()
