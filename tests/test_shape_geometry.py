"""Ray-shape hits and surface interactions against float64 geometry, independently of the oracle.

The other geometry tests pin the CUDA kernels (`sphere_test` / `sphere_surface` / `tri_test` in yk_device.cuh) to the oracle
(`Scene::sphere_intersect` / `triangle_intersect` in oracle/yko_scene.h) bit for bit. Both are transcriptions of the same
reading of shapes/sphere.rs and shapes/triangle.rs, so a misreading they share passes those tests. Here every hit is compared
with the exact ray-quadric / ray-plane geometry of the float32 inputs the kernels receive (the ray, the sphere's
world_to_object matrix and radius, the world-space triangle vertices), evaluated in float64.

Tolerances are not blanket: each is a forward error bound derived per ray (see `sphere_reference` and `triangle_reference`),
and each test also asserts that the bound is tight (most rays within ~1e-5 relative) and reports the largest error / bound
ratio per quantity, so that a vacuous bound cannot pass.

Watertightness: rays through every vertex and shared edge of closed meshes must hit (pbrt's watertight test with the f64
edge-function fallback guarantees it for the shape test alone). The BVH walk has no gamma-widened slab test (bounds.rs:
176-215), so it may cull such a ray that the triangle test would accept; those misses are counted and pinned.
"""
import numpy as np
import pytest

from test_query_surface import _check as _gpu_check, osurf  # noqa: F401 (the oracle's surface query fixture)
from yuki_b200 import api, desc as D, scenes

F32 = np.float32
U = 2.0 ** -24                      # float32 unit roundoff
SPLITS = {"sah": D.SPLIT_SAH, "middle": D.SPLIT_MIDDLE, "equal": D.SPLIT_EQUAL_COUNTS}


def gamma(n):
    """pbrt's gamma(n) = n u / (1 - n u): the relative error bound of n float32 roundings."""
    return n * U / (1.0 - n * U)


def _mat4(a):
    return np.asarray(a, np.float64).reshape(4, 4)


def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def _ratio(err, bound):
    """err / bound, with NaN errors (a NaN output) as inf so that they fail."""
    err = np.where(np.isnan(err), np.inf, err)
    return err / bound


class Worst:
    """The largest error / bound ratio per quantity, asserted <= 1 and reported."""

    def __init__(self, what):
        self.what, self.r = what, {}

    def add(self, name, err, bound, mask=None):
        r = _ratio(np.asarray(err, np.float64), np.asarray(bound, np.float64))
        if mask is not None:
            r = r[mask]
        if r.size == 0:
            return
        i = int(np.argmax(r))
        self.r[name] = max(self.r.get(name, 0.0), float(r.flat[i]))
        assert r.flat[i] <= 1.0, (self.what, name, int((r > 1.0).sum()), float(r.flat[i]))

    def report(self):
        print(self.what, {k: f"{v:.3g}" for k, v in sorted(self.r.items())})


# ---- spheres ------------------------------------------------------------------------------------------------------------
def _neg_zero_frame():
    """The identity, stored with -0 in the y row of world_to_object, so that a ray with o.y = d.y = -0 (and positive x, z)
    reaches object space with p.y = -0 exactly: atan2(-0, x > 0) = -0, the φ seam's other side."""
    m = np.eye(4, dtype=np.float32).reshape(-1)
    mi = m.copy()
    mi[4], mi[6], mi[7] = -0.0, -0.0, -0.0
    return D.Transform(m, mi)


def _sphere_cases(xf):
    """(o2w, radius, diagonal): identity, translated, uniform / non-uniform scale, rotated, mirrored, combinations; radii 1e-2
    ... 1e2, centres up to 1e3 from the origin. `diagonal` transforms keep a ray along the object z axis exactly on it."""
    T, S, R, M = xf.translation, xf.scale, xf.rotation, xf.mul
    return {
        "identity": (xf.translation((0.0, 0.0, 0.0)), 1.0, True),
        "translated": (T((3.5, -2.25, 7.0)), 0.5, True),
        "far-small": (T((1000.0, -400.0, 250.0)), 1e-2, True),
        "uniform-scale": (M(T((-1.0, 2.0, 0.5)), S(3.0, 3.0, 3.0)), 0.75, True),
        "non-uniform-scale": (M(T((0.25, -0.5, 4.0)), S(2.0, 0.5, 1.3)), 1.0, True),
        "rotated": (M(T((1.0, 1.0, -2.0)), R(0.7, (0.3, 1.0, 0.2))), 1.5, False),
        "mirrored": (S(1.0, -1.0, 1.0), 1.0, True),
        "rotated-scaled-mirrored": (M(T((1000.0, 200.0, -600.0)), M(R(2.1, (1.0, 0.4, -0.3)), S(1.5, -0.7, 0.9))), 100.0, False),
        "scaled-mirrored-small": (M(T((-30.0, 12.0, 45.0)), M(S(-0.6, 1.8, 1.1), R(-1.2, (0.0, 0.5, 1.0)))), 0.02, False),
        "neg-zero": (_neg_zero_frame(), 1.0, True),
    }


def sphere_scene(o2w, radius):
    s = D.SceneDesc()
    zero = s.add_texture(D.Texture.constant(0.0))
    s.spheres.append(D.Sphere(o2w, float(radius), s.add_material(D.Material(D.MAT_MATTE, (s.add_texture(D.Texture.constant(0.5)), zero)))))
    return s


def _rand_dirs(rng, n):
    return _unit(rng.normal(size=(n, 3)))


def sphere_rays(o2w, r, diagonal, seed):
    """World-space float32 rays (o, d, t_max) and a kind per ray, made in object space and moved to the world by o2w:
    from outside (hits and misses), from inside (the t1 branch), from just inside the surface, with t_max below t0 / between the roots / beyond t1, grazing
    (impact parameter r (1 +- 1e-3 ... 1e-7)), along the z axis through both poles, across the φ = 0 seam (p.y = +-0 and
    +-1e-6 r), and from far away (|o| = 30 r ... 1e3 r)."""
    rng = np.random.default_rng(seed)
    M = _mat4(o2w.m)
    o_l, d_l, tm_l, kind = [], [], [], []

    def add(o, d, tm, k):
        o_l.append(o); d_l.append(d); tm_l.append(tm); kind.extend([k] * len(o))

    n = 1500
    u = _rand_dirs(rng, n)
    o = u * r * rng.uniform(1.5, 6.0, (n, 1))
    tgt = _rand_dirs(rng, n) * r * rng.uniform(0.0, 1.3, (n, 1))
    d = (tgt - o) * rng.uniform(0.1, 10.0, (n, 1))
    add(o, d, np.full(n, np.inf), "outside")
    o = _rand_dirs(rng, n) * r * rng.uniform(0.0, 0.9, (n, 1)) ** (1 / 3)
    add(o, _rand_dirs(rng, n) * rng.uniform(0.1, 10.0, (n, 1)), np.full(n, np.inf), "inside")
    # t_max around the roots of rays that cross the sphere: the exact roots of the object-space ray, spread by factors
    m = 1500
    u = _rand_dirs(rng, m)
    o = -3.0 * r * u
    w = _unit(np.cross(u, _rand_dirs(rng, m)))
    o = o + w * r * rng.uniform(0.0, 0.9, (m, 1))
    d = u
    b = 2.0 * (o * d).sum(-1)
    c = (o * o).sum(-1) - r * r
    sq = np.sqrt(b * b - 4.0 * c)
    t0, t1 = (-b - sq) / 2.0, (-b + sq) / 2.0
    pick = rng.integers(0, 3, m)
    tm = np.where(pick == 0, t0 * rng.uniform(0.3, 0.99, m), np.where(pick == 1, t0 + (t1 - t0) * rng.uniform(0.05, 0.95, m), t1 * rng.uniform(1.01, 2.0, m)))
    add(o, d, tm, "t_max")
    # the same from inside: t_max below and above t1
    o = _rand_dirs(rng, m) * r * 0.5
    d = _rand_dirs(rng, m)
    b = 2.0 * (o * d).sum(-1)
    c = (o * o).sum(-1) - r * r
    t1 = (-b + np.sqrt(b * b - 4.0 * c)) / 2.0
    add(o, d, t1 * np.where(rng.integers(0, 2, m) == 0, rng.uniform(0.3, 0.99, m), rng.uniform(1.01, 2.0, m)), "t_max-inside")
    # from just inside the surface, heading inwards (b < 0, c ~ 0-): the far root c / q is where the sign choice of
    # q = -0.5 (b -+ sqrt Delta) keeps q free of cancellation
    ns = 600
    u = _rand_dirs(rng, ns)
    o = u * r * (1.0 - rng.choice([1e-3, 1e-4, 3e-5], ns))[:, None]
    add(o, -u + 0.6 * _rand_dirs(rng, ns), np.full(ns, np.inf), "near-surface")
    # grazing
    g = 800
    u = _rand_dirs(rng, g)
    w = _unit(np.cross(u, _rand_dirs(rng, g)))
    eps = rng.choice([1e-3, 1e-4, 1e-5, 1e-6, 1e-7], g) * rng.choice([-1.0, 1.0], g)
    add(-3.0 * r * u + w * r * (1.0 + eps)[:, None], u, np.full(g, np.inf), "grazing")
    # far away
    f = 800
    o = _rand_dirs(rng, f) * r * np.exp(rng.uniform(np.log(30.0), np.log(1e3), (f, 1)))
    add(o, (_rand_dirs(rng, f) * r * rng.uniform(0.0, 0.8, (f, 1)) - o), np.full(f, np.inf), "far")
    # the φ = 0 seam: hit points at y = 0 with x > 0, from origins in the plane y = 0 and just off it
    s = 400
    ang = rng.uniform(-1.2, 1.2, s)
    tgt = np.stack([np.cos(ang), np.zeros(s), np.sin(ang)], -1) * r
    o = tgt + np.stack([np.cos(ang), np.zeros(s), np.sin(ang)], -1) * r * 2.0 + np.stack([np.zeros(s), np.zeros(s), rng.uniform(-0.5, 0.5, s)], -1) * r
    off = rng.choice([0.0, 1e-6, -1e-6], s) * r
    o[:, 1] = off
    tgt[:, 1] = off
    add(o, tgt - o, np.full(s, np.inf), "seam")
    o_obj = np.concatenate(o_l)
    d_obj = np.concatenate(d_l)
    o_w = (o_obj @ M[:3, :3].T + M[:3, 3]).astype(F32)
    d_w = (d_obj @ M[:3, :3].T).astype(F32)
    extra_o, extra_d, extra_kind = [], [], []
    if diagonal:
        # along the object z axis, both directions, from outside and inside: p.x = p.y = 0 exactly (the pole nudge)
        for z0, dz in ((3.0, -1.0), (-3.0, 1.0), (0.0, 1.0), (0.0, -1.0), (0.25, 1.0), (-0.5, -1.0)):
            extra_o.append(M[:3, :3] @ np.array([0.0, 0.0, z0 * r]) + M[:3, 3])
            extra_d.append(M[:3, :3] @ np.array([0.0, 0.0, dz]))
            extra_kind.append("pole")
        if np.array_equal(_mat4(o2w.m), np.eye(4)):
            # p.y = +0 and -0 on the seam (neg-zero's world_to_object keeps -0; the identity's turns it into +0)
            for oy, dy in ((0.0, 0.0), (-0.0, -0.0)):
                extra_o.append(np.array([0.3, oy, 0.2]))
                extra_d.append(np.array([1.0, dy, 0.5]))
                extra_kind.append("seam")
    if extra_o:
        o_w = np.concatenate([o_w, np.array(extra_o, F32)])
        d_w = np.concatenate([d_w, np.array(extra_d, F32)])
        kind += extra_kind
    tm = np.concatenate(tm_l + [np.full(len(extra_o), np.inf)]).astype(F32)
    return o_w, d_w, tm, np.array(kind)


def sphere_reference(o2w, radius, o, d, t_max):
    """Exact hit of the float32 rays with the quadric |W o + t W d|^2 = r^2 (W: the float32 world_to_object the kernel
    applies), in float64, with a forward error bound for every quantity the kernel returns.

    Error analysis (u = 2^-24, gamma(n) = n u / (1 - n u)):
    * object-space ray: o' = W o + w and d' = W d are computed here in float32 as the kernel computes them (transform.rs:
      103-142: ((m0 x + m1 y) + m2 z) + m3, no fused multiply-add), so their rounding is known exactly; one more rounding of
      |o'|, |d'| covers a kernel that sums in another order. (Under a translation o' is often exact: Sterbenz.)
    * a = d'.d' (3 roundings), b = 2 d'.o' (3), c = o'.o' - r^2 (4, plus r^2's), each also moved by the errors of o', d':
      da <= gamma(3) a + 2 |d'| . dd', db <= 2 (gamma(3) |d'| . |o'| + |d'| . do' + |o'| . dd'),
      dc <= gamma(5) (|o'|^2 + r^2) + 2 |o'| . do'. The last term is the cancellation in c = |o|^2 - r^2 for distant origins;
    * the discriminant's own rounding, gamma(2) (b^2 + 4 a |c|), moves the roots as a change of c by that over 4a would
      (dt = dDelta / (4 a sqrt Delta));
    * at an exact root t, F(t) = a t^2 + b t + c moves by dF <= t^2 da + |t| db + dc', and the root by the x that solves
      sqrt(Delta) x + a x^2 = dF, i.e. x = 2 dF / (sqrt Delta + sqrt(Delta + 4 a dF)): dF / sqrt Delta away from grazing,
      sqrt(dF / a) at it;
    * sqrt, q = -0.5 (b -+ sqrt Delta) (no cancellation: the sign follows b), q / a and c / q add gamma(4) |t| and u
      sqrt(Delta) / (2a).
    The hit / miss decision is only determined where |Delta| exceeds its bound dDelta = 2 |b| db + 4 (a dc + |c| da) +
    gamma(3) (b^2 + 4 a |c|), and where each root is further than its bound from 0 and from t_max.

    The point p = o' + t d' errs by E <= |do'| + t |dd'| + |d'| dt + gamma(3) (|o'| + t |d'|); its projection onto the sphere
    (p r / |p|) by at most E r / (r - E) <= E (1 + 2 E / r), plus gamma(8) r for len, the division and the product. World quantities go through the float32 object_to_world M."""
    W, M = _mat4(o2w.m_inv), _mat4(o2w.m)
    o, d, t_max = (np.asarray(a, np.float64) for a in (o, d, t_max))
    r = float(F32(radius))
    Wa, Ma = np.abs(W[:3, :3]), np.abs(M[:3, :3])
    oo = o @ W[:3, :3].T + W[:3, 3]
    dd = d @ W[:3, :3].T
    W32 = np.asarray(o2w.m_inv, F32).reshape(4, 4)
    o32, d32 = np.asarray(o, F32), np.asarray(d, F32)
    xf32 = lambda v, w: np.stack([((W32[k, 0] * v[:, 0] + W32[k, 1] * v[:, 1]) + W32[k, 2] * v[:, 2]) + w[k] for k in range(3)], -1)
    oo32 = xf32(o32, W32[:3, 3]).astype(np.float64)
    dd32 = xf32(d32, np.zeros(3, F32)).astype(np.float64)
    e_o = np.abs(oo32 - oo) + U * np.abs(oo32)
    e_d = np.abs(dd32 - dd) + U * np.abs(dd32)
    a = (dd * dd).sum(-1)
    b = 2.0 * (dd * oo).sum(-1)
    c = (oo * oo).sum(-1) - r * r
    da = gamma(3) * a + 2.0 * (np.abs(dd) * e_d).sum(-1)
    db = 2.0 * (gamma(3) * np.abs(dd * oo).sum(-1) + (np.abs(dd) * e_o + np.abs(oo) * e_d).sum(-1))
    dc = gamma(5) * ((oo * oo).sum(-1) + r * r) + 2.0 * (np.abs(oo) * e_o).sum(-1)
    disc = b * b - 4.0 * a * c
    d_disc = 2.0 * np.abs(b) * db + 4.0 * (a * dc + np.abs(c) * da) + gamma(3) * (b * b + 4.0 * a * np.abs(c))
    dc_eff = dc + gamma(2) * (b * b + 4.0 * a * np.abs(c)) / (4.0 * a)
    sq = np.sqrt(np.maximum(disc, 0.0))
    with np.errstate(divide="ignore", invalid="ignore"):
        q = -0.5 * (b + np.where(b < 0, -sq, sq))
        r0, r1 = q / a, c / q
    t0, t1 = np.minimum(r0, r1), np.maximum(r0, r1)

    def root_err(t):
        dF = t * t * da + np.abs(t) * db + dc_eff
        return 2.0 * dF / (sq + np.sqrt(disc + 4.0 * a * dF)) + gamma(4) * np.abs(t) + U * sq / (2.0 * a)

    with np.errstate(invalid="ignore"):
        e0, e1 = root_err(t0), root_err(t1)
        real = disc >= 0
        hit = real & ~((t0 > t_max) | (t1 <= 0)) & ((t0 > 0) | (t1 <= t_max))
        first = t0 > 0
        t = np.where(first, t0, t1)
        et = np.where(first, e0, e1)
        near = lambda x, y, e: np.abs(x - y) <= e
        ambiguous = (np.abs(disc) <= d_disc) | near(t0, 0, e0) | near(t1, 0, e1) | near(t0, t_max, e0) | near(t1, t_max, e1)
    p_raw = oo + t[:, None] * dd
    p_obj = p_raw * (r / np.linalg.norm(p_raw, axis=-1, keepdims=True))
    E = (np.linalg.norm(e_o, axis=-1) + np.abs(t) * np.linalg.norm(e_d, axis=-1) + np.linalg.norm(dd, axis=-1) * et
         + gamma(3) * (np.linalg.norm(oo, axis=-1) + np.abs(t) * np.linalg.norm(dd, axis=-1)))
    e_p_obj = E * (1.0 + 2.0 * E / r) + gamma(8) * r
    # the pole nudge (sphere.rs:81-84) of an exact pole hit
    pole = (p_obj[:, 0] == 0.0) & (p_obj[:, 1] == 0.0)
    p_n = p_obj.copy()
    p_n[pole, 0] = 1e-5 * r
    p_w = p_n @ M[:3, :3].T + M[:3, 3]         # the nudged point is the one moved to the world
    e_p = (Ma @ np.ones(3)) * e_p_obj[:, None] + gamma(4) * (np.abs(p_n) @ Ma.T + np.abs(M[:3, 3]))
    # the normal: the object-space outward normal, negated when the transform swaps handedness (sphere.rs:104-110,
    # interaction.rs:105-113: n = cross(dpdu, dpdv), flipped), then moved by the inverse transpose (interaction.rs:141-164).
    # A mirrored sphere's world normal therefore points into it.
    swaps = np.linalg.det(M[:3, :3]) < 0
    n_obj = p_obj / r * (-1.0 if swaps else 1.0)
    v = n_obj @ W[:3, :3]                      # W^T n, row-vector form
    vn = np.linalg.norm(v, axis=-1)
    n_w = v / vn[:, None]
    W2 = np.linalg.norm(W[:3, :3], 2)
    e_n = 2.0 * (W2 * (e_p_obj / r + 20.0 * U) + gamma(3) * np.linalg.norm(Wa, "fro")) / vn + 4.0 * U
    # uv (sphere.rs:85-97): u = phi / 2 pi with phi in [0, 2 pi), v = 1 - theta / pi, from the (nudged) object-space point
    phi = np.mod(np.arctan2(p_n[:, 1], p_n[:, 0]), 2.0 * np.pi)
    uu = phi / (2.0 * np.pi)
    zr = np.hypot(p_n[:, 0], p_n[:, 1])
    e_u = (e_p_obj / zr + 8.0 * U) / (2.0 * np.pi) + 4.0 * U
    cz = np.clip(p_n[:, 2] / r, -1.0, 1.0)
    theta = np.arccos(cz)
    dcz = e_p_obj / r + 4.0 * U
    e_theta = np.maximum(np.abs(np.arccos(np.clip(cz + dcz, -1, 1)) - theta), np.abs(np.arccos(np.clip(cz - dcz, -1, 1)) - theta))
    vv = 1.0 - theta / np.pi
    e_v = (e_theta + 4.0 * U * np.pi) / np.pi + 4.0 * U
    # shading_dpdu = M (-2 pi p.y, 2 pi p.x, 0) (sphere.rs:98), with phi_max = 2 pi in float32
    dp_obj = np.stack([-2.0 * np.pi * p_n[:, 1], 2.0 * np.pi * p_n[:, 0], np.zeros(len(p_n))], -1)
    dpdu = dp_obj @ M[:3, :3].T
    e_dpdu = (Ma @ np.ones(3)) * (2.0 * np.pi * e_p_obj)[:, None] + gamma(6) * (np.abs(dp_obj) @ Ma.T)
    return {"hit": hit, "ambiguous": ambiguous, "t": t, "e_t": et, "t0": t0, "t1": t1, "p": p_w, "e_p": e_p, "n": n_w,
            "e_n": e_n, "u": uu, "e_u": e_u, "v": vv, "e_v": e_v, "dpdu": dpdu, "e_dpdu": e_dpdu, "pole": pole, "swaps": swaps,
            "p_obj": p_obj, "centre": M[:3, 3], "cond": np.linalg.cond(W[:3, :3]), "r": r, "scale": float(np.abs(M[:3, :3]).max()) * r}


def check_sphere(got, ref, o, d, kind, t_max, what):
    """The hits `got` (dict or Hits of the surface query) against `sphere_reference`; returns the Worst record."""
    g = {k: np.asarray(got[k] if isinstance(got, dict) else getattr(got, k)) for k in api.HIT_FIELDS}
    w = Worst(what)
    hit_k = g["orig_id"] >= 0
    det = ~ref["ambiguous"]
    bad = det & (hit_k != ref["hit"])
    assert not bad.any(), (what, "hit / miss", int(bad.sum()), np.unique(kind[bad]).tolist())
    assert np.all(np.isinf(g["t"][~hit_k]))
    h = hit_k & ref["hit"] & det
    w.add("t", np.abs(g["t"] - ref["t"]), ref["e_t"], h)
    assert np.all(g["t"][hit_k] <= t_max[hit_k]) and np.all(g["t"][hit_k] > 0), what
    w.add("p", np.abs(g["p"] - ref["p"]).max(-1), ref["e_p"].max(-1), h)
    w.add("n", np.linalg.norm(g["n"] - ref["n"], axis=-1), ref["e_n"], h)
    # shading_n is n itself (sphere.rs builds no separate shading frame)
    assert np.array_equal(g["shading_n"][h].view(np.uint32), g["n"][h].view(np.uint32)), what
    uk = g["uv"][:, 0].astype(np.float64)
    assert np.all((uk[h] >= 0.0) & (uk[h] <= 1.0)), (what, "u outside [0, 1]", float(uk[h].min()))
    du = np.abs(uk - ref["u"])
    w.add("u", np.minimum(du, 1.0 - du), ref["e_u"], h)      # modulo 1 across the seam
    w.add("v", np.abs(g["uv"][:, 1] - ref["v"]), ref["e_v"], h)
    w.add("shading_dpdu", np.abs(g["shading_dpdu"] - ref["dpdu"]).max(-1), ref["e_dpdu"].max(-1), h)
    # the bounds are tight on the bulk: for 90 % of the well-conditioned hits (not grazing, not far) the bound on t |d| is
    # within 1e-5 of the magnitude L of the coordinates the kernel receives (origin, centre, radius), p's within 3e-5 L, and
    # the normal's, which the origin's rounding reaches through p / r and the inverse transpose amplifies by W's condition
    # number, within 3e-5 cond(W) L / r
    bulk = h & np.isin(kind, ["outside", "inside", "t_max", "t_max-inside"])
    L = np.maximum(np.maximum(np.linalg.norm(np.asarray(o, np.float64), axis=-1), np.linalg.norm(ref["centre"])), ref["scale"])
    if bulk.sum() > 100:
        assert np.mean((ref["e_t"] * np.linalg.norm(np.asarray(d, np.float64), axis=-1) / L)[bulk] <= 1e-5) >= 0.9, what
        assert np.mean((ref["e_p"].max(-1) / L)[bulk] <= 3e-5) >= 0.9, what
        assert np.mean((ref["e_n"] * ref["scale"] / (L * ref["cond"]))[bulk] <= 3e-5) >= 0.9, what
    return w, h


SPHERE_NAMES = ["identity", "translated", "far-small", "uniform-scale", "non-uniform-scale", "rotated", "mirrored",
                "rotated-scaled-mirrored", "scaled-mirrored-small", "neg-zero"]


def _sphere_setup(xf, name):
    o2w, r, diagonal = _sphere_cases(xf)[name]
    o, d, tm, kind = sphere_rays(o2w, r, diagonal, seed=SPHERE_NAMES.index(name) + 11)
    return sphere_scene(o2w, r), o2w, r, o, d, tm, kind


def _sphere_claims(got, ref, kind, h, name, diagonal):
    """What the case names must occur, so that a later change cannot make it pass vacuously."""
    hit_k = np.asarray(got["orig_id"]) >= 0
    uv = np.asarray(got["uv"])
    for k in ("outside", "inside", "t_max", "t_max-inside", "far"):
        assert (h & (kind == k)).sum() > 100, (name, k)
    assert ((kind == "outside") & ~hit_k & ~ref["ambiguous"]).sum() > 20, name             # misses too
    assert (h & (kind == "inside") & (ref["t0"] <= 0)).sum() > 500, name                 # the t1 branch
    tm_kinds = np.isin(kind, ["t_max", "t_max-inside"]) & ~ref["ambiguous"]
    assert (tm_kinds & ~hit_k).sum() > 200 and (tm_kinds & hit_k).sum() > 200, name      # t_max cuts and keeps
    seam = h & (kind == "seam")
    assert (h & (kind == "near-surface")).sum() > 300, name
    assert (h & (kind == "grazing")).sum() > 50 and ((kind == "grazing") & ~hit_k).sum() > 50, name
    if np.spacing(F32(np.abs(ref["centre"]).max())) < 1e-7 * ref["r"]:   # float32 holds the seam rays' y = +-1e-6 r there
        assert (seam & (ref["p_obj"][:, 1] < 0) & (uv[:, 0] > 0.99)).sum() > 20, name     # across the seam: u -> 1 ...
        assert (seam & (ref["p_obj"][:, 1] >= 0) & (uv[:, 0] < 0.01)).sum() > 20, name    # ... and u -> 0
    if diagonal:
        pole = h & (kind == "pole")
        assert pole.sum() >= 4 and np.all(ref["pole"][pole]), name
        assert np.all(uv[pole, 0] == 0.0), name
    if name == "neg-zero":
        # p.y = +0 and -0 on the seam: u = atan2(+-0, x > 0) / 2 pi = +-0 (-0 is not < 0, so no 2 pi is added)
        assert np.array_equal(np.signbit(uv[kind == "seam"][-2:, 0]), [False, True]), uv[kind == "seam"][-2:]
    if ref["swaps"]:
        # a handedness swap: the normal points into the sphere (see sphere_reference)
        out = ((np.asarray(got["p"], np.float64) - ref["centre"]) * np.asarray(got["n"], np.float64)).sum(-1)
        assert np.all(out[h] < 0), name


@pytest.mark.parametrize("name", SPHERE_NAMES)
def test_oracle_sphere_hits_match_float64(osurf, xf, name):
    scene, o2w, r, o, d, tm, kind = _sphere_setup(xf, name)
    osc = osurf(scene)
    got = osc.surface(o, d, tm)
    ref = sphere_reference(o2w, r, o, d, tm)
    w, h = check_sphere(got, ref, o, d, kind, tm, name)
    _sphere_claims(got, ref, kind, h, name, _sphere_cases(xf)[name][2])
    # no vacuous bound: in every case the worst t error is a sizeable part of its bound
    assert w.r["t"] >= 1e-2, w.r
    # t_max at one ulp either side of the returned root: accepted at t == t_max, cut one ulp below. Not for far rays, nor on a
    # sphere whose centre's float32 spacing exceeds 1e-4 r: there the float32 root may fall short of where the unwidened slab
    # test enters the sphere's bounds, which then culls the ray.
    h = h & (kind != "far") & (np.spacing(F32(np.abs(ref["centre"]).max())) < 1e-4 * r)
    t = got["t"][h]
    at = osc.surface(o[h], d[h], t)
    below = osc.surface(o[h], d[h], np.nextafter(t, F32(0)))
    above = osc.surface(o[h], d[h], np.nextafter(t, F32(np.inf)))
    assert np.array_equal(at["t"], t) and np.array_equal(above["t"], t), name
    assert not (below["orig_id"] >= 0).any(), name
    w.report()


@pytest.mark.gpu
@pytest.mark.parametrize("name", SPHERE_NAMES)
def test_gpu_sphere_hits_match_float64_and_the_oracle(gpu_ctx, osurf, xf, name):
    scene, o2w, r, o, d, tm, kind = _sphere_setup(xf, name)
    dev, osc = api.Scene(gpu_ctx, scene), osurf(scene)
    try:
        got = _gpu_check(dev, osc, o, d, tm)
        _gpu_check(dev, osc, o, d)
        h = np.asarray(got.orig_id) >= 0
        t = np.asarray(got.t)[h]
        _gpu_check(dev, osc, o[h], d[h], np.nextafter(t, F32(0)))
    finally:
        dev.close()
    w, _ = check_sphere(got, sphere_reference(o2w, r, o, d, tm), o, d, kind, tm, name)
    w.report()


# ---- triangles ----------------------------------------------------------------------------------------------------------
def _tri_cases(xf):
    """(o2w, with_normals, uv mode): scale 1e-3 ... 1e3, offsets up to 1e4, rotations and mirrors."""
    T, S, R, M = xf.translation, xf.scale, xf.rotation, xf.mul
    return {
        "unit": (xf.identity(), True, "random"),
        "small-rotated": (M(T((0.5, -0.2, 1.0)), M(R(0.9, (1.0, 0.2, 0.4)), S(1e-3, 1e-3, 1e-3))), True, "random"),
        "large-far": (M(T((1e4, -5e3, 8e3)), M(R(-0.4, (0.2, 1.0, 0.1)), S(1e3, 1e3, 1e3))), True, "random"),
        "mirrored": (M(T((100.0, 20.0, -50.0)), M(R(2.0, (0.0, 1.0, 0.3)), S(-1.0, 1.0, 1.0))), True, "random"),
        "mirrored-non-uniform": (M(R(0.3, (1.0, 0.0, 0.0)), S(2.0, -0.5, 1.5)), True, "random"),
        "degenerate-uv": (M(T((-3.0, 1.0, 2.0)), R(1.1, (0.3, 0.3, 1.0))), True, "degenerate"),
        "plain": (S(10.0, 10.0, 10.0), False, None),
    }


TRI_NAMES = ["unit", "small-rotated", "large-far", "mirrored", "mirrored-non-uniform", "degenerate-uv", "plain"]


def tri_scene(xf, name):
    o2w, normals, uvm = _tri_cases(xf)[name]
    pts, idx = scenes.grid_mesh(10, 10, seed=TRI_NAMES.index(name) + 3, height=0.45)
    rng = np.random.default_rng(TRI_NAMES.index(name))
    nrm = (np.array([0.0, 1.0, 0.0]) + rng.uniform(-0.7, 0.7, (len(pts), 3))).astype(F32) if normals else None
    uvs = None
    if uvm == "random":
        uvs = rng.uniform(-1.0, 2.0, (len(pts), 2)).astype(F32)
    elif uvm == "degenerate":
        uvs = np.full((len(pts), 2), 0.25, F32)   # uv_det == 0: dpdu from coordinate_system (triangle.rs:160-163)
    s = D.SceneDesc(max_shapes_in_node=4)
    zero = s.add_texture(D.Texture.constant(0.0))
    m = s.add_material(D.Material(D.MAT_MATTE, (s.add_texture(D.Texture.constant(0.5)), zero)))
    s.meshes.append(D.Mesh(o2w, pts, idx, m, normals=nrm, uvs=uvs))
    world = np.array([xf.point(o2w, p) for p in pts], F32)
    wn = None if nrm is None else np.array([xf.normal(o2w, v) for v in nrm], F32)
    return s, o2w, world, idx.reshape(-1, 3), wn, uvs


def tri_rays(world, seed, n=6000):
    """Incoherent rays through the mesh's bounds (from above, below and the sides), half of them aimed at vertices."""
    rng = np.random.default_rng(seed)
    lo, hi = world.min(0).astype(np.float64), world.max(0).astype(np.float64)
    ext = hi - lo
    c = (lo + hi) / 2.0
    o = c + _rand_dirs(rng, n) * np.linalg.norm(ext) * rng.uniform(0.6, 1.5, (n, 1))
    tgt = lo + rng.uniform(0.0, 1.0, (n, 3)) * ext
    tgt[: n // 4] = world[rng.integers(0, len(world), n // 4)]
    return o.astype(F32), (tgt - o).astype(F32)


def triangle_reference(world, tris, o, d):
    """Every (ray, triangle) pair in float64 from the float32 inputs: the watertight test's sheared coordinates and edge
    functions (triangle.rs:58-106), the exact ray-plane distance, and pbrt-v3's bounds (pbrt-v3 3.9.2):
    * sheared x, y: p - o, sx = -dx / dz, sx z and the sum: dx <= gamma(5) (max|x| + max|sx z|), likewise y;
    * edge functions: dE = 2 (gamma(2) max|x| max|y| + dy max|x| + dx max|y|);
    * t: dz = gamma(3) max|z sz|, dt = 3 (gamma(3) maxE max|z sz| + dE max|z sz| + dz maxE) / |det|.
    Returns (t, inside, ambiguous, dt, barycentrics, dE / |det|) of shape (rays, triangles)."""
    o, d = np.asarray(o, np.float64), np.asarray(d, np.float64)
    P = np.asarray(world, np.float64)[tris]                       # (T, 3, 3)
    ad = np.abs(np.asarray(d, F32))
    kz = np.where(ad[:, 0] > ad[:, 1], np.where(ad[:, 0] > ad[:, 2], 0, 2), np.where(ad[:, 1] > ad[:, 2], 1, 2))
    kx = np.where(kz < 2, kz + 1, 0)
    ky = np.where(kx < 2, kx + 1, 0)
    rows = np.arange(len(o))
    dx, dy, dz = d[rows, kx], d[rows, ky], d[rows, kz]
    sx, sy, sz = -dx / dz, -dy / dz, 1.0 / dz
    rel = P[None, :, :, :] - o[:, None, None, :]                  # (R, T, 3 vertices, 3)
    X = np.take_along_axis(rel, kx[:, None, None, None], 3)[..., 0]
    Y = np.take_along_axis(rel, ky[:, None, None, None], 3)[..., 0]
    Z = np.take_along_axis(rel, kz[:, None, None, None], 3)[..., 0]
    xs = X + sx[:, None, None] * Z
    ys = Y + sy[:, None, None] * Z
    e0 = xs[..., 1] * ys[..., 2] - ys[..., 1] * xs[..., 2]
    e1 = xs[..., 2] * ys[..., 0] - ys[..., 2] * xs[..., 0]
    e2 = xs[..., 0] * ys[..., 1] - ys[..., 0] * xs[..., 1]
    E = np.stack([e0, e1, e2], -1)
    det = E.sum(-1)
    zs = Z * sz[:, None, None]
    max_x = np.abs(xs).max(-1)
    max_y = np.abs(ys).max(-1)
    max_zs = np.abs(zs).max(-1)
    sxz = (np.abs(sx)[:, None, None] * np.abs(Z)).max(-1)
    syz = (np.abs(sy)[:, None, None] * np.abs(Z)).max(-1)
    ddx = gamma(5) * (np.abs(X).max(-1) + sxz)
    ddy = gamma(5) * (np.abs(Y).max(-1) + syz)
    dE = 2.0 * (gamma(2) * max_x * max_y + ddy * max_x + ddx * max_y)
    max_e = np.abs(E).max(-1)
    dzz = gamma(3) * max_zs
    with np.errstate(divide="ignore", invalid="ignore"):
        dt = 3.0 * (gamma(3) * max_e * max_zs + dE * max_zs + dzz * max_e) / np.abs(det)
        n = np.cross(P[:, 1] - P[:, 0], P[:, 2] - P[:, 0])
        t = ((P[None, :, 0] - o[:, None]) * n[None]).sum(-1) / (d @ n.T)
        B = E / det[..., None]
    sgn = np.sign(det)[..., None]
    firm_in = np.all(E * sgn > dE[..., None], -1) & (np.abs(det) > 3.0 * dE)
    firm_out = np.any(E * sgn < -dE[..., None], -1) | (np.abs(det) <= 0)
    inside = firm_in & (t > dt)
    ambiguous = ~firm_out & ~inside & ~(t < -dt)
    with np.errstate(divide="ignore", invalid="ignore"):
        db = dE / np.abs(det)
    return {"t": t, "inside": inside, "ambiguous": ambiguous, "dt": dt, "b": B, "db": db}


def _shading_normal_ref(b, eb, nv):
    """set_shading_geometry of the interpolated vertex normals (triangle.rs:197-224, interaction.rs:126-132) in float64:
    ns = normalize(sum b_i n_i); ss = normalize(dpdu), ts = cross(ss, ns) normalised, ss = cross(ts, ns),
    sh_n = normalize(cross(ss, ts)), which is ns itself. Also the bound on the direction of the float32 sum, from the
    barycentrics' bounds eb and three roundings of each weighted term."""
    v = (b[:, :, None] * nv).sum(1)
    vn = np.linalg.norm(v, axis=-1)
    nn = np.linalg.norm(nv, axis=-1)
    e = (eb * nn).sum(-1) + gamma(3) * (np.abs(b) * nn).sum(-1)
    return v / vn[:, None], e / vn


def check_triangles(got, world, tris, o, d, wn, uvs, swaps, what):
    """The query's hits against `triangle_reference`; returns the Worst record and counts."""
    g = {k: np.asarray(got[k] if isinstance(got, dict) else getattr(got, k)) for k in api.HIT_FIELDS}
    ref = triangle_reference(world, tris, o, d)
    t, inside, amb, dt = ref["t"], ref["inside"], ref["ambiguous"], ref["dt"]
    cand = inside | amb
    R = np.arange(len(o))
    w = Worst(what)
    k = g["orig_id"]
    hit = k >= 0
    # misses only where no triangle is firmly hit
    bad = ~hit & inside.any(1)
    assert not bad.any(), (what, "missed a firm hit", int(bad.sum()))
    # a hit is a candidate of float64, its t within that triangle's bound
    kk = np.maximum(k, 0)
    assert np.all(cand[R, kk][hit]), (what, "hit a triangle float64 misses", int((~cand[R, kk] & hit).sum()))
    w.add("t", np.abs(g["t"] - t[R, kk]), dt[R, kk], hit)
    # the closest: where the float64 closest candidate is firm and the next candidate is more than 2 dt behind
    tc = np.where(cand, t, np.inf)
    order = np.argsort(tc, axis=1)
    c0, c1 = order[:, 0], order[:, 1] if tc.shape[1] > 1 else order[:, 0]
    t0, t1 = tc[R, c0], tc[R, c1]
    decided = inside[R, c0] & (t1 - t0 > 2.0 * np.maximum(dt[R, c0], np.where(np.isfinite(t1), dt[R, c1], 0.0)))
    bad = decided & (k != c0)
    assert not bad.any(), (what, "not the closest triangle", int(bad.sum()))
    # p, uv from the barycentrics: db_i <= dE / |det| (+ |b_i| 3 dE / |det| through det), then the weighted sums
    b, db = ref["b"][R, kk], ref["db"][R, kk]
    ebi = db[:, None] * (1.0 + 3.0 * np.abs(b)) + 2.0 * U * np.abs(b)
    P = np.asarray(world, np.float64)[tris[kk]]
    p_ref = (b[:, :, None] * P).sum(1)
    e_p = (ebi[:, :, None] * np.abs(P)).sum(1) + gamma(3) * (np.abs(b)[:, :, None] * np.abs(P)).sum(1)
    w.add("p", np.abs(g["p"] - p_ref).max(-1), e_p.max(-1), hit)
    w.add("p vs o + t d", np.abs(g["p"] - (o + t[R, kk][:, None] * np.asarray(d, np.float64))).max(-1),
          e_p.max(-1) + np.abs(np.asarray(d, np.float64)).max(-1) * dt[R, kk], hit)
    if uvs is not None:
        UV = uvs.astype(np.float64)[tris[kk]]
    else:
        UV = np.broadcast_to(np.array([(0.0, 0.0), (1.0, 0.0), (1.0, 1.0)]), (len(o), 3, 2))
    uv_ref = (b[:, :, None] * UV).sum(1)
    e_uv = (ebi[:, :, None] * np.abs(UV)).sum(1) + gamma(3) * (np.abs(b)[:, :, None] * np.abs(UV)).sum(1)
    w.add("uv", np.abs(g["uv"] - uv_ref).max(-1), e_uv.max(-1) + 1e-30, hit)
    # geometric normal: normalize(cross(p0 - p2, p1 - p2)) (triangle.rs:187-194), negated on a handedness swap; float32
    # differences err by u each, the f64 cross is rounded once, the normalisation adds 3 roundings
    e02, e12 = P[:, 0] - P[:, 2], P[:, 1] - P[:, 2]
    cr = np.cross(e02, e12)
    crn = np.linalg.norm(cr, axis=-1)
    ng = cr / crn[:, None] * (-1.0 if swaps else 1.0)
    e_n = 2.0 * (2.0 * U * np.sqrt(3.0) * np.linalg.norm(e02, axis=-1) * np.linalg.norm(e12, axis=-1) / crn + 4.0 * U)
    if wn is not None:
        ns, e_ns = _shading_normal_ref(b, ebi, wn.astype(np.float64)[tris[kk]])
        # the shading frame's float32 chain: ss = normalize(dpdu) crossed with ns, error growing as 1 / |ss x ns|
        ng = np.where(((ng * ns).sum(-1) < 0)[:, None], -ng, ng)   # n faces the shading normal (interaction.rs:130)
        clear = hit & (np.abs((ng * ns).sum(-1)) > 1e-3)
        sinang = _dpdu_sin(P, UV, ns, swaps)
        w.add("shading_n", np.linalg.norm(g["shading_n"] - ns, axis=-1), 2.0 * e_ns + 40.0 * U / np.maximum(sinang, 1e-3), clear & (sinang > 1e-3))
        w.add("n", np.linalg.norm(g["n"] - ng, axis=-1), e_n, clear)
    else:
        w.add("n", np.linalg.norm(g["n"] - ng, axis=-1), e_n, hit)
        assert np.array_equal(g["shading_n"][hit], g["n"][hit]), what
    counts = {"hits": int(hit.sum()), "decided": int(decided.sum()), "edge-ambiguous": int((amb.any(1)).sum())}
    return w, counts, ref


def _dpdu_sin(P, UV, ns, swaps):
    """|sin| of the angle between dpdu (triangle.rs:143-172, coordinate_system of the face normal when uv_det == 0) and ns."""
    duv02, duv12 = UV[:, 0] - UV[:, 2], UV[:, 1] - UV[:, 2]
    dp02, dp12 = P[:, 0] - P[:, 2], P[:, 1] - P[:, 2]
    det = duv02[:, 0] * duv12[:, 1] - duv02[:, 1] * duv12[:, 0]
    with np.errstate(divide="ignore", invalid="ignore"):
        dpdu = (dp02 * duv12[:, 1:2] - dp12 * duv02[:, 1:2]) / det[:, None]
    n = _unit(np.cross(P[:, 2] - P[:, 0], P[:, 1] - P[:, 0]))
    alt = np.where((np.abs(n[:, 0]) > np.abs(n[:, 1]))[:, None], np.stack([-n[:, 2], 0 * n[:, 0], n[:, 0]], -1),
                   np.stack([0 * n[:, 0], n[:, 2], -n[:, 1]], -1))
    dpdu = np.where((det == 0)[:, None], alt, dpdu)
    return np.linalg.norm(np.cross(_unit(dpdu), ns), axis=-1)


def _tri_setup(xf, name):
    scene, o2w, world, tris, wn, uvs = tri_scene(xf, name)
    o, d = tri_rays(world, TRI_NAMES.index(name) + 40)
    swaps = np.linalg.det(_mat4(o2w.m)[:3, :3]) < 0
    return scene, world, tris, wn, uvs, o, d, swaps


@pytest.mark.parametrize("name", TRI_NAMES)
def test_oracle_triangle_hits_match_float64(osurf, xf, name):
    scene, world, tris, wn, uvs, o, d, swaps = _tri_setup(xf, name)
    got = osurf(scene).surface(o, d)
    w, counts, ref = check_triangles(got, world, tris, o, d, wn, uvs, swaps, name)
    assert counts["hits"] > 2000 and counts["decided"] > 0.7 * counts["hits"], counts   # a quarter aim at vertices
    # the bound is not vacuous: pbrt-v3's dt (its factor 3, and maxE max|z| in place of each term's own size) sits at a median
    # of ~4e-5 relative to t; 90 % of the hits are within 2e-4
    hit = got["orig_id"] >= 0
    kk = np.maximum(got["orig_id"], 0)
    rel = ref["dt"][np.arange(len(o)), kk] / np.abs(ref["t"][np.arange(len(o)), kk])
    assert np.mean(rel[hit] <= 2e-4) >= 0.9, np.median(rel[hit])
    w.report()
    print(name, counts)


@pytest.mark.gpu
@pytest.mark.parametrize("name", TRI_NAMES)
def test_gpu_triangle_hits_match_float64_and_the_oracle(gpu_ctx, osurf, xf, name):
    scene, world, tris, wn, uvs, o, d, swaps = _tri_setup(xf, name)
    dev, osc = api.Scene(gpu_ctx, scene), osurf(scene)
    try:
        got = _gpu_check(dev, osc, o, d)
    finally:
        dev.close()
    w, counts, _ = check_triangles(got, world, tris, o, d, wn, uvs, swaps, name)
    assert counts["hits"] > 2000
    w.report()


# ---- watertightness -----------------------------------------------------------------------------------------------------
def _weld(pts, idx):
    """Merge vertices that differ by rounding only (the uv sphere's seam column and its pole rings), so that the mesh is closed
    bit for bit: triangles that share an edge share its two vertices."""
    key = np.round(pts.astype(np.float64) * 1e5).astype(np.int64)
    _, first, inv = np.unique(key, axis=0, return_index=True, return_inverse=True)
    inv = inv.reshape(-1)
    new_idx = inv[idx]
    tri = new_idx.reshape(-1, 3)
    keep = (tri[:, 0] != tri[:, 1]) & (tri[:, 1] != tri[:, 2]) & (tri[:, 0] != tri[:, 2])
    return pts[first], tri[keep].reshape(-1).astype(np.uint32)


def _octahedron(levels=2):
    """A unit octahedron subdivided `levels` times, midpoints pushed onto the unit sphere; outward winding."""
    v = [(1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)]
    f = [(0, 2, 4), (2, 1, 4), (1, 3, 4), (3, 0, 4), (2, 0, 5), (1, 2, 5), (3, 1, 5), (0, 3, 5)]
    pts = [np.array(p, np.float64) for p in v]
    for _ in range(levels):
        mid, nf = {}, []

        def m(a, b):
            key = (min(a, b), max(a, b))
            if key not in mid:
                mid[key] = len(pts)
                pts.append(_unit(pts[a] + pts[b]))
            return mid[key]

        for a, b, c in f:
            ab, bc, ca = m(a, b), m(b, c), m(c, a)
            nf += [(a, ab, ca), (ab, b, bc), (ca, bc, c), (ab, bc, ca)]
        f = nf
    return np.array(pts, F32), np.array(f, np.uint32).reshape(-1)


def _closed_meshes(xf):
    T, S, R, M = xf.translation, xf.scale, xf.rotation, xf.mul
    box = scenes._box((-0.5, -0.25, -1.0), (1.5, 0.75, 0.25))
    sp, si, _, _ = scenes._uv_sphere(1.0, stacks=12, slices=24, with_normals=False)
    return {
        "box": (box, xf.identity()),
        "uv-sphere": (_weld(sp, si), M(T((0.3, -0.2, 0.1)), M(R(0.8, (0.4, 1.0, -0.2)), S(1.6, 0.7, 1.1)))),
        "octahedron": (_octahedron(2), M(T((-2.0, 1.0, 3.0)), R(0.5, (1.0, -0.3, 0.6)))),
    }


def _edge_rays(world, tris, seed):
    """Rays from an interior point at every vertex and at points on every shared edge (parameters 0.5 and two random ones, and
    one float32 ulp from each end towards the other), and exterior rays crossing the surface through the same points. The edge points are computed in
    float64 and rounded; the ray's direction is the float32 difference, as a caller would form it."""
    rng = np.random.default_rng(seed)
    W = np.asarray(world, np.float64)
    e = np.sort(np.concatenate([tris[:, [0, 1]], tris[:, [1, 2]], tris[:, [2, 0]]]), axis=1)
    edges, cnt = np.unique(e, axis=0, return_counts=True)
    assert np.all(cnt == 2), "not a closed 2-manifold"
    s = np.stack([np.full(len(edges), 0.5), rng.uniform(0, 1, len(edges)), rng.uniform(0, 1, len(edges))], 1)
    a, b = W[edges[:, 0]], W[edges[:, 1]]
    pts = (a[:, None] + s[..., None] * (b - a)[:, None]).reshape(-1, 3)
    # one ulp from each end: every coordinate of the vertex moved by one float32 ulp towards the other vertex
    a32, b32 = world[edges[:, 0]], world[edges[:, 1]]
    ulp = np.concatenate([np.nextafter(a32, b32), np.nextafter(b32, a32)])
    targets = np.concatenate([W.astype(F32), pts.astype(F32), ulp])
    c = W.mean(0)
    inner = [c, c + 0.2 * (W.max(0) - W.min(0)) * np.array([0.3, -0.5, 0.4])]
    o, d = [], []
    for ci in inner:
        ci32 = ci.astype(F32)
        o.append(np.broadcast_to(ci32, targets.shape))
        d.append(targets - ci32)
        out = (targets.astype(np.float64) + (targets.astype(np.float64) - ci)).astype(F32)    # outside a convex mesh
        o.append(out)
        d.append(ci32 - out)
    return np.concatenate(o).astype(F32), np.concatenate(d).astype(F32), len(edges)


# The BVH walk's culls of rays that the triangle test accepts (misses, or hits behind brute force's closest hit), per mesh,
# split method and leaf size:
# the slab test of bounds.rs:176-215 is not widened by gamma(3) as pbrt's is. Pinned; see DESIGN.md §2.
# Rays: box 392, uv sphere 16 904, octahedron 4 104 (see _edge_rays).
SLAB_MISSES = {
    ("box", "sah", 1): 1, ("box", "sah", 4): 1, ("box", "middle", 1): 1, ("box", "middle", 4): 1,
    ("box", "equal", 1): 1, ("box", "equal", 4): 0,
    ("uv-sphere", "sah", 1): 16, ("uv-sphere", "sah", 4): 5, ("uv-sphere", "middle", 1): 16, ("uv-sphere", "middle", 4): 6,
    ("uv-sphere", "equal", 1): 16, ("uv-sphere", "equal", 4): 8,
    ("octahedron", "sah", 1): 2, ("octahedron", "sah", 4): 0, ("octahedron", "middle", 1): 2, ("octahedron", "middle", 4): 0,
    ("octahedron", "equal", 1): 2, ("octahedron", "equal", 4): 1,
}


def _culled(t, t_brute):
    """Rays the walk misses or hits behind the brute-force closest hit."""
    t, tb = t.astype(np.float64), t_brute.astype(np.float64)
    return ~(t <= tb * (1.0 + 8.0 * U))


WATERTIGHT_CASES = [(m, s, leaf) for m in ("box", "uv-sphere", "octahedron") for s in SPLITS for leaf in (1, 4)]


def _watertight_setup(xf, mesh, split, leaf):
    (pts, idx), o2w = _closed_meshes(xf)[mesh]
    s = D.SceneDesc(split_method=SPLITS[split], max_shapes_in_node=leaf)
    zero = s.add_texture(D.Texture.constant(0.0))
    s.meshes.append(D.Mesh(o2w, pts, idx, s.add_material(D.Material(D.MAT_MATTE, (s.add_texture(D.Texture.constant(0.5)), zero)))))
    world = np.array([xf.point(o2w, p) for p in pts], F32)
    o, d, n_edges = _edge_rays(world, idx.reshape(-1, 3), seed=len(pts))
    return s, o, d


@pytest.mark.parametrize("mesh,split,leaf", WATERTIGHT_CASES, ids=[f"{m}-{s}-leaf{l}" for m, s, l in WATERTIGHT_CASES])
def test_oracle_closed_meshes_are_watertight(oracle, xf, mesh, split, leaf):
    scene, o, d = _watertight_setup(xf, mesh, split, leaf)
    osc = oracle.OracleScene(scene)
    # pbrt's guarantee for the shape test alone: every ray through a vertex or a shared edge hits
    tb, ib, _ = osc.trace(o, d, brute_force=True)
    assert np.all(ib >= 0), (mesh, "brute force missed", int((ib < 0).sum()))
    # the walk: its misses, and its hits behind brute force's closest one (an exterior ray whose entry the slab test culled
    # goes on to the far side), are rays the triangle test accepts and the unwidened slab test culls. Elsewhere it meets
    # brute force's distance, to the ulps by which the triangles sharing the point differ (the walk may reach another first)
    t, ids, _ = osc.trace(o, d)
    culled = _culled(t, tb)
    tw, tbf = t[~culled].astype(np.float64), tb[~culled].astype(np.float64)
    assert np.all(np.abs(tw - tbf) <= 8.0 * U * tbf), float((np.abs(tw - tbf) / tbf).max())
    print(mesh, split, leaf, "rays", len(o), "slab-test culls", int(culled.sum()), "of which misses", int((ids < 0).sum()))
    assert int(culled.sum()) == SLAB_MISSES[(mesh, split, leaf)], int(culled.sum())


@pytest.mark.gpu
@pytest.mark.parametrize("mesh,split,leaf", WATERTIGHT_CASES, ids=[f"{m}-{s}-leaf{l}" for m, s, l in WATERTIGHT_CASES])
def test_gpu_closed_meshes_walk_like_the_oracle(gpu_ctx, oracle, xf, mesh, split, leaf):
    scene, o, d = _watertight_setup(xf, mesh, split, leaf)
    osc = oracle.OracleScene(scene)
    dev = api.Scene(gpu_ctx, scene)
    try:
        t, ids, cnt = dev.intersect(o, d)
    finally:
        dev.close()
    ot, oids, ocnt = osc.trace(o, d)
    assert np.array_equal(ids, oids) and np.array_equal(t.view(np.uint32), ot.view(np.uint32)) and np.array_equal(cnt, ocnt)
    tb, ib, _ = osc.trace(o, d, brute_force=True)
    assert int(_culled(t, tb).sum()) == SLAB_MISSES[(mesh, split, leaf)]
