"""Every material kind under every light kind, and Whitted's glass tree, against float64 restatements of the reference.

The other radiance tests pin the CUDA kernels to the oracle bit for bit; a formula both misread the same way passes them.
Here the reference's equations are restated in numpy and evaluated in float64, independently of the oracle's lobe and light
code (only its camera rays and sampler draws are used, both pinned elsewhere):

* lobes in the shading frame (bsdfs/{lambertian,oren_nayar,microfacet,trowbridge_reitz,fresnel}.rs) with the materials'
  parameter mapping (materials/{matte,metal,glossy}.rs), including `roughness_to_alpha` and the 1e-3 alpha floor;
* the four lights' `sample_li` (lights/{point,spot,rectangular,distant}_light.rs) and the direct-lighting fold
  f(wo, wi) * Li * clamp(n_s . wi, 0, 1) / pdf summed over lights (path.rs:102-119, whitted.rs:109-126), which is the whole
  film at Path depth 1 and Whitted depth 1 on a single plane;
* the specular tree whitted.rs:132-170 walks through a glass slab, as a float64 recursion over the analytic planes.

As in test_shadow_modes.py, every case has a CPU part (the oracle against float64, plus asserts that the scene reaches what the
case claims, so that a later change cannot make it pass vacuously) and a GPU part (the GPU film against the same float64
reference, and bit-equal to the oracle).
"""
import functools

import numpy as np
import pytest

from test_oracle_geometry import _quad_scene
from yuki_b200 import api, desc as D, transforms as xf

F32 = np.float32
EPS32 = 2.0 ** -24   # float32 unit roundoff

# ---- 1. float64 restatement of the lobes (shading frame: z = n_s, x = normalize(dpdu)) ------------------------------
def _sin2(w):            # bsdfs/mod.rs:225-300
    return np.maximum(1.0 - w[..., 2] ** 2, 0.0)


def _phi(w):
    """(cos phi, sin phi), each clamped to [-1, 1], and 1 when sin theta = 0 (bsdfs/mod.rs:238-252, the reference's quirk)."""
    st = np.sqrt(_sin2(w))
    safe = np.where(st == 0.0, 1.0, st)
    return (np.where(st == 0.0, 1.0, np.clip(w[..., 0] / safe, -1.0, 1.0)),
            np.where(st == 0.0, 1.0, np.clip(w[..., 1] / safe, -1.0, 1.0)))


def oren_nayar_f(kd, sigma, wo, wi):
    """oren_nayar.rs:18-53; sigma in radians as stored. The impl names its parameters (wi, wo): the trait's wo comes first."""
    s2 = sigma * sigma
    a = 1.0 - s2 / (2.0 * (s2 + 0.33))
    b = 0.45 * s2 / (s2 + 0.09)
    sin_i, sin_o = np.sqrt(_sin2(wo)), np.sqrt(_sin2(wi))
    (ci, si), (co, so) = _phi(wo), _phi(wi)
    max_cos = np.where((sin_i > 1e-4) & (sin_o > 1e-4), np.maximum(ci * co + si * so, 0.0), 0.0)
    first = np.abs(wo[..., 2]) > np.abs(wi[..., 2])
    sin_alpha = np.where(first, sin_o, sin_i)
    tan_beta = np.where(first, sin_i / np.abs(wo[..., 2]), sin_o / np.abs(wi[..., 2]))
    return kd / np.pi * (a + b * max_cos * sin_alpha * tan_beta)[..., None]


def ggx_d(alpha, wh):    # trowbridge_reitz.rs:34-44
    c2 = wh[..., 2] ** 2
    t2 = _sin2(wh) / c2
    cp, sp = _phi(wh)
    a2 = alpha * alpha
    e = (cp * cp / a2 + sp * sp / a2) * t2
    return 1.0 / (np.pi * a2 * c2 * c2 * (1.0 + e) ** 2)


def ggx_lambda(alpha, w):   # trowbridge_reitz.rs:46-58
    tan = np.abs(np.sqrt(_sin2(w)) / w[..., 2])
    cp, sp = _phi(w)
    a = np.sqrt(cp * cp * alpha * alpha + sp * sp * alpha * alpha)
    return (-1.0 + np.sqrt(1.0 + (a * tan) ** 2)) / 2.0


def fr_conductor(eta, k, c):   # fresnel.rs:68-96 with eta_i = 1
    c = np.minimum(np.abs(c), 1.0)[..., None]
    c2, s2 = c * c, 1.0 - c * c
    t0 = eta * eta - k * k - s2
    a2b2 = np.sqrt(t0 * t0 + 4.0 * eta * eta * k * k)
    t1 = a2b2 + c2
    a = np.sqrt((a2b2 + t0) * 0.5)
    t2 = 2.0 * a * c
    rs = (t1 - t2) / (t1 + t2)
    t3 = a2b2 * c2 + s2 * s2
    t4 = t2 * s2
    return (rs * (t3 - t4) / (t3 + t4) + rs) * 0.5


def fr_schlick(rs, c):   # fresnel.rs:108-117
    v = 1.0 - np.clip(c, -1.0, 1.0)[..., None]
    return rs + (1.0 - rs) * v ** 5


def microfacet_f(alpha, fresnel, wo, wi):
    """microfacet.rs:53-74: D(wh) G(wo, wi) Fr(wi . faceforward(wh, +z)) / (4 |cos_i| |cos_o|), G = 1 / (1 + Lo + Li).
    Also returns the relative error float32 adds through D's sin^2 theta_h = 1 - cos^2 theta_h, which cancels near the peak:
    t2 = sin^2 / cos^2 errs by ~2 ulp of 1 over sin^2 theta_h, and |d ln D / d ln t2| = 2e / (1 + e) with e = t2 / alpha^2, so
    D errs by 2e / (1 + e) * 2^-23 / sin^2 = 2^-22 / (cos^2 alpha^2 (1 + e)): 1.5e-4 at the peak of alpha = 0.04."""
    wh = wo + wi
    wh = wh / np.linalg.norm(wh, axis=-1, keepdims=True)
    whf = np.where((wh[..., 2] < 0.0)[..., None], -wh, wh)
    g = 1.0 / (1.0 + ggx_lambda(alpha, wo) + ggx_lambda(alpha, wi))
    fr = fresnel((wi * whf).sum(axis=-1))
    c2 = wh[..., 2] ** 2
    d_err = 4.0 * EPS32 / (c2 * alpha * alpha * (1.0 + _sin2(wh) / c2 / (alpha * alpha)))
    return (ggx_d(alpha, wh) * g / (4.0 * np.abs(wi[..., 2]) * np.abs(wo[..., 2])))[..., None] * fr, d_err


ALPHA_POLY = (1.62142, 0.819955, 0.1734, 0.0171201, 0.000640711)   # trowbridge_reitz.rs:22-30 (pbrt-v3)


def roughness_to_alpha(r):
    x = np.log(np.maximum(r, 1e-3))
    return sum(c * x ** i for i, c in enumerate(ALPHA_POLY))


def alpha_rel_error(r, remap, squared):
    """A bound on the relative float32 error of alpha. Remapped: every term c * x^i carries at most i + 1 roundings (and the
    float32 constants one more), every partial sum one; the terms nearly cancel for small r (at r = 1e-3 they reach 8.3 for a
    sum of 0.047), so the bound is 2^-24 * (sum_i (i + 2) |c x^i| + sum |partial sums|) / |alpha|. Squaring adds one
    rounding and doubles the relative error."""
    if not remap:
        e = np.full(np.shape(r), EPS32)
    else:
        x = np.log(np.maximum(r, 1e-3))
        terms = [c * x ** i for i, c in enumerate(ALPHA_POLY)]
        partial = np.cumsum(terms, axis=0)
        bound = sum((i + 2) * np.abs(t) for i, t in enumerate(terms)) + np.abs(partial).sum(axis=0)
        e = EPS32 * bound / np.abs(partial[-1])
    return 2.0 * e + EPS32 if squared else e


class Mat:
    """A material of the test plane: its scene description and its float64 lobe."""

    def __init__(self, name, kind, params, image=None, remap=False):
        self.name, self.kind, self.params, self.image, self.remap = name, kind, params, image, remap

    def add_to(self, scene):
        def tex(v):
            return scene.add_texture(D.Texture.constant(*np.atleast_1d(v)))
        img = None if self.image is None else scene.add_texture(D.Texture.from_image(np.repeat(self.image[..., None], 3, axis=2)))
        p = self.params
        if self.kind == D.MAT_MATTE:
            return scene.add_material(D.Material(D.MAT_MATTE, (tex(p["kd"]), img if img is not None else tex(p["sigma"]))))
        if self.kind == D.MAT_METAL:
            return scene.add_material(D.Material(D.MAT_METAL, (tex(p["eta"]), tex(p["k"]), img if img is not None else tex(p["rough"])),
                                                 remap_roughness=self.remap))
        return scene.add_material(D.Material(D.MAT_GLOSSY, (tex(p["rs"]), img if img is not None else tex(p["rough"])),
                                             remap_roughness=self.remap))

    def scalar(self, texel):
        """The per-pixel scalar parameter (sigma or roughness): the constant, or the image's texel value."""
        key = "sigma" if self.kind == D.MAT_MATTE else "rough"
        return np.float64(F32(self.params[key])) * np.ones(texel.shape) if self.image is None else self.image.astype(np.float64)[texel]

    def alpha(self, r):
        a = roughness_to_alpha(r) if self.remap else r
        return np.maximum(a * a if self.kind == D.MAT_GLOSSY else a, 1e-3)   # glossy.rs:49, trowbridge_reitz.rs:16-20

    def f(self, wo, wi, texel):
        """(N, 3) f(wo, wi) of the one lobe in the local frame, sigma / roughness per pixel through `texel`; and the relative
        error float32 adds beyond RTOL (microfacet_f, rtol_extra)."""
        p, v = self.params, self.scalar(texel)
        f64 = lambda c: np.asarray(F32(c), np.float64)
        if self.kind == D.MAT_MATTE:
            on = oren_nayar_f(f64(p["kd"]), v, wo, wi)
            return np.where((v == 0.0)[..., None], f64(p["kd"]) / np.pi, on), 0.0   # sigma == 0: Lambert, matte.rs:33
        if self.kind == D.MAT_METAL:
            f, d_err = microfacet_f(self.alpha(v), lambda c: fr_conductor(f64(p["eta"]), f64(p["k"]), c), wo, wi)
        else:
            f, d_err = microfacet_f(self.alpha(v), lambda c: fr_schlick(f64(p["rs"]), c), wo, wi)
        return f, d_err + self.rtol_extra(texel)

    def rtol_extra(self, texel):
        """Relative error of f from alpha's own float32 rounding: |d ln f / d ln alpha| <= 2 for D (D = a^2 / (pi c^4 (a^2 +
        t^2)^2)) and <= 1 for G, so 3 times alpha's relative error."""
        if self.kind == D.MAT_MATTE:
            return 0.0
        return 3.0 * alpha_rel_error(self.scalar(texel), self.remap, self.kind == D.MAT_GLOSSY)


COPPER_ETA, COPPER_K = (0.27105, 0.67693, 1.31640), (3.60920, 2.62480, 2.29210)   # scenes.py copper, scene/mod.rs:214-223
KD, GLOSSY_RS = (0.7, 0.6, 0.3), (0.6, 0.45, 0.3)
ROUGH_TEXELS = np.array([[5e-4, 2e-3, 0.01, 0.05], [0.1, 0.3, 0.6, 1.0]], np.float32)    # 5e-4: below the 1e-3 floor
SIGMA_TEXELS = np.array([[0.0, 0.1, 0.35, 0.6], [0.8, 1.05, 1.3, 1.5]], np.float32)


def _materials():
    rad = lambda deg: float(F32(np.deg2rad(deg)))
    m = [Mat("matte", D.MAT_MATTE, {"kd": KD, "sigma": 0.0}),
         Mat("oren-nayar-20", D.MAT_MATTE, {"kd": KD, "sigma": rad(20.0)}),
         Mat("oren-nayar-60", D.MAT_MATTE, {"kd": KD, "sigma": rad(60.0)})]
    m += [Mat(f"copper-a{a}", D.MAT_METAL, {"eta": COPPER_ETA, "k": COPPER_K, "rough": a}) for a in (0.8, 0.3, 0.05)]
    m.append(Mat("copper-r0.01-remap", D.MAT_METAL, {"eta": COPPER_ETA, "k": COPPER_K, "rough": 0.01}, remap=True))
    m += [Mat(f"glossy-r{r}" + ("-remap" if remap else ""), D.MAT_GLOSSY, {"rs": GLOSSY_RS, "rough": r}, remap=remap)
          for r in (0.5, 0.2) for remap in (False, True)]
    return {x.name: x for x in m}


IMAGE_MATERIALS = {
    "oren-nayar-image": Mat("oren-nayar-image", D.MAT_MATTE, {"kd": KD, "sigma": None}, image=SIGMA_TEXELS),
    "copper-image-remap": Mat("copper-image-remap", D.MAT_METAL, {"eta": COPPER_ETA, "k": COPPER_K, "rough": None}, image=ROUGH_TEXELS, remap=True),
    "glossy-image-remap": Mat("glossy-image-remap", D.MAT_GLOSSY, {"rs": GLOSSY_RS, "rough": None}, image=ROUGH_TEXELS, remap=True),
}
MATERIALS = _materials()


# ---- the planes ---------------------------------------------------------------------------------------------------------
class Plane:
    """_quad_scene's square (uv = (x + 1) / 2, (y + 1) / 2), with a mesh transform or without. Geometry in float64 from the
    float32 world vertices the renderer intersects."""

    def __init__(self, name, to_world=None):
        self.name, self.to_world = name, to_world
        pts = np.array([(-1, -1, 0), (1, -1, 0), (1, 1, 0), (-1, 1, 0)], np.float32)
        self.v = np.array([xf.point(to_world, p) if to_world is not None else p for p in pts], np.float64)
        v0, v1, v2, v3 = self.v
        self.n = np.cross(v0 - v2, v1 - v2)                # triangle.rs:187-194
        self.n /= np.linalg.norm(self.n)
        self.ss = (v1 - v0) / np.linalg.norm(v1 - v0)      # dpdu = p1 - p0 for uv (0,0), (1,0), (1,1): the shading s axis
        self.ts = np.cross(self.n, self.ss)                # bsdfs/mod.rs:87-99
        self.eu, self.ev = v1 - v0, v3 - v0

    def scene(self, mat):
        s, cam = _quad_scene()
        if self.to_world is not None:
            s.meshes[0].object_to_world = self.to_world
        s.meshes[0].material = mat.add_to(s)
        return s, cam

    def hit(self, o, d):
        """float64 hit of rays (o, d) with the plane: p, uv, inside, and distance of p to the outline."""
        o, d = np.asarray(o, np.float64), np.asarray(d, np.float64)
        t = ((self.v[0] - o) @ self.n) / (d @ self.n)
        p = o + t[..., None] * d
        q = p - self.v[0]
        u = (q @ self.eu) / (self.eu @ self.eu)
        v = (q @ self.ev) / (self.ev @ self.ev)
        inside = (t > 0) & (u > 0) & (u < 1) & (v > 0) & (v < 1)
        edge = 2.0 * np.minimum(np.minimum(u, 1 - u), np.minimum(v, 1 - v))   # the square's side is 2
        return p, np.stack([u, v], axis=-1), inside, edge

    def local(self, w):
        return np.stack([w @ self.ss, w @ self.ts, w @ self.n], axis=-1)


PLANES = {"flat": Plane("flat"),
          "tilted": Plane("tilted", xf.mul(xf.rotation(float(F32(0.5)), (0.0, 0.0, 1.0)), xf.rotation(float(F32(0.45)), (1.0, 0.6, 0.0))))}


# ---- lights ------------------------------------------------------------------------------------------------------------
class Light:
    def __init__(self, desc):
        self.desc = desc
        self.m = desc.light_to_world.m.astype(np.float64).reshape(4, 4)
        self.m_inv = desc.light_to_world.m_inv.astype(np.float64).reshape(4, 4)
        self.i = np.asarray(F32(desc.intensity), np.float64)
        self.pos = self.m[:3, 3]

    def sample(self, p, n, u):
        """sample_li at points p (geometric normal n) with draws u: wi, Li, pdf and whether a shadow ray exists."""
        k, N = self.desc.kind, p.shape[0]
        ones = np.ones(N)
        if k == D.LIGHT_POINT:   # point_light.rs:27-49: I / d^2
            to = self.pos - p
            d2 = (to * to).sum(axis=-1)
            return to / np.sqrt(d2)[:, None], self.i / d2[:, None], ones, ones > 0
        if k == D.LIGHT_SPOT:    # spot_light.rs:38-80: I * falloff / d^2, falloff = delta^4 in the blend, no shadow ray at 0
            to = self.pos - p
            d2 = (to * to).sum(axis=-1)
            wi = to / np.sqrt(d2)[:, None]
            fall = self.falloff(p)
            return wi, self.i * (fall / d2)[:, None], ones, fall > 0
        if k == D.LIGHT_DISTANT:   # distant_light.rs:17-43: L along w as given, not normalised
            w = np.asarray(F32(self.desc.direction), np.float64)
            return np.broadcast_to(w, p.shape), np.broadcast_to(self.i, p.shape), ones, ones > 0
        # rectangular_light.rs:27-72: the point (u.x, 0, u.y) of the unit square scaled to `size`, one-sided radiance along the
        # transformed -y normal (not normalised), pdf = d^2 / (|cos_l| * area)
        sx, sz = (float(F32(v)) for v in self.desc.size)
        lp_local = np.stack([sx * (u[:, 0] - 0.5), np.zeros(N), sz * (u[:, 1] - 0.5)], axis=-1)
        lp = lp_local @ self.m[:3, :3].T + self.m[:3, 3]
        nl = self.m_inv[:3, :3].T @ np.array([0.0, -1.0, 0.0])   # normals transform by the inverse transpose
        wi = lp - p
        d2 = (wi * wi).sum(axis=-1)
        wi = wi / np.sqrt(d2)[:, None]
        cos_l = -(wi @ nl)
        li = np.where((cos_l > 0)[:, None], self.i, 0.0)
        area = float(F32(F32(sx) * F32(sz)))
        return wi, li, d2 / (np.abs(cos_l) * area), ones > 0

    def cos_spot(self, p):
        dl = (p - self.pos) @ self.m_inv[:3, :3].T      # world_to_light applied to -wi (the direction from the light)
        return dl[:, 2] / np.linalg.norm(dl, axis=-1)

    def cone(self):
        return np.cos(np.deg2rad(self.desc.total_width_deg)), np.cos(np.deg2rad(self.desc.falloff_start_deg))

    def falloff(self, p):
        ct = self.cos_spot(p)
        c_tot, c_fall = self.cone()
        delta = (ct - c_tot) / (c_fall - c_tot)
        return np.where(ct < c_tot, 0.0, np.where(ct > c_fall, 1.0, delta ** 4))


def _light_descs(place):
    """The light sets, placed in the frame of the plane's mesh transform `place` (None: the world), so that each reaches the
    same situation on either plane."""
    rot = lambda deg, axis: xf.rotation(float(F32(np.deg2rad(deg))), axis)
    at = (lambda t: t) if place is None else (lambda t: xf.mul(place, t))
    along = (lambda v: v) if place is None else (lambda v: tuple(float(c) for c in xf.vec(place, v)))
    w = np.array([0.3, -0.4, 0.85])
    w_unit = along(tuple(float(v) for v in F32(w / np.linalg.norm(w))))
    out = {
        "point-high": [D.Light(D.LIGHT_POINT, at(xf.translation((0.4, 0.3, 2.0))), (3.0, 2.0, 1.0))],
        # low and to the side: grazing incidence, where Lambda is large enough to tell the Smith forms apart
        "point-low": [D.Light(D.LIGHT_POINT, at(xf.translation((3.0, 0.5, 0.4))), (30.0, 25.0, 20.0))],
        # aimed down (local +z maps to about -z) at a slant; its 30 deg cone edge crosses the visible plane
        "spot": [D.Light(D.LIGHT_SPOT, at(xf.mul(xf.translation((0.2, -0.1, 1.5)), rot(170.0, (1.0, 0.3, 0.0)))), (4.0, 3.0, 2.0),
                         total_width_deg=30.0, falloff_start_deg=12.0)],
        "distant-unit": [D.Light(D.LIGHT_DISTANT, xf.identity(), (1.5, 1.2, 0.9), direction=w_unit)],
        "distant-non-unit": [D.Light(D.LIGHT_DISTANT, xf.identity(), (1.5, 1.2, 0.9), direction=tuple(float(F32(0.7 * v)) for v in w_unit))],
        # rotated +90 deg about x, the light's -y normal points down at the plane; -90 deg points it away
        "rect": [D.Light(D.LIGHT_RECT, at(xf.mul(xf.translation((0.2, 0.1, 1.2)), xf.mul(rot(15.0, (0.0, 1.0, 0.0)), rot(90.0, (1.0, 0.0, 0.0))))),
                         (4.0, 3.5, 3.0), size=(0.6, 0.4))],
        "rect-away": [D.Light(D.LIGHT_RECT, at(xf.mul(xf.translation((0.2, 0.1, 1.2)), rot(-90.0, (1.0, 0.0, 0.0)))), (4.0, 3.5, 3.0), size=(0.6, 0.4))],
    }
    out["all-four"] = out["point-high"] + out["spot"] + out["distant-non-unit"] + out["rect"]
    return out


LIGHTS = {name: _light_descs(plane.to_world) for name, plane in PLANES.items()}
LIGHT_NAMES = list(LIGHTS["flat"])


def _has_rect(lights):
    return any(l.kind == D.LIGHT_RECT for l in lights)


# ---- films and tolerances -----------------------------------------------------------------------------------------------
DELTA_FILM, DELTA_SAMPLER = D.FilmSettings((96, 72), 16), D.SamplerType.stratified(1, 1, jitter=False)   # pixel centres
RECT_FILM, RECT_SAMPLER = D.FilmSettings((48, 36), 16), D.SamplerType.stratified(4, 4)
# Relative tolerance of one pixel, for every lobe, light and the fold. The kernel evaluates f * Li * cos / pdf in float32 from
# float32 inputs: about 60 roundings of at most 2^-24 each on the longest chain (the conductor Fresnel and GGX), 4e-6. Its
# shading point is the float32 hit, a few ulp (<= 5e-7 absolute) from the float64 point here; towards a light >= 0.4 away that
# turns wi by <= 1.2e-6 rad, which moves cos_i (>= 0.05 where kept, see COS_CUTOFF) by <= 2.4e-5 relative and GGX's D, whose
# log-derivative in theta_h is at most 2 / alpha, by ~(2 / alpha) * 6e-7, i.e. 2.4e-5 at the smallest constant alpha, 0.05.
# (In practice the point errs by ~1 ulp: the worst errors measured on the oracle are below 1e-5.) A rect-light pixel is the mean
# of 16 such terms summed in float32 (15 more roundings, 1e-6). 5e-5 covers the sum of these bounds.
RTOL = 5e-5
COS_CUTOFF = 0.05      # shading cosines below this (grazing light) are left out: cos is where the relative error is 1 / cos
EDGE = 1e-2            # distance to the square's outline below which a pixel is left out
SPOT_CT_ERR = 1e-6     # spot falloff: the float32 cos_theta of the cone test (a normalised float32 vector) is within ~4 ulp


@functools.lru_cache(maxsize=None)
def _rect_draws(n_lights):
    """The camera's 2-D draw, then one 2-D draw per light in light order (yko_render.h:88, 312), of every (pixel, sample) of
    RECT_FILM: (res_y, res_x, spp, 2 + 2 * n_lights)."""
    from oracle import oracle as O
    spp = RECT_SAMPLER.samples_per_pixel()
    w, h = RECT_FILM.res
    out = np.zeros((h, w, spp, 2 + 2 * n_lights), np.float32)
    for y in range(h):
        for x in range(w):
            for i in range(spp):
                out[y, x, i] = O.sampler_draws(RECT_SAMPLER, x, y, i, [2] * (1 + n_lights))
    return out


def _texel(mat, uv):
    """image_texture.rs:85-110: nearest texel with v flipped; plus whether the choice is away from a texel boundary."""
    if mat.image is None:
        return np.zeros(uv.shape[:-1], int), np.ones(uv.shape[:-1], bool)
    h, w = mat.image.shape
    fx, fy = uv[..., 0] * w - 0.5, (1.0 - uv[..., 1]) * h - 0.5
    ix, iy = np.clip(np.trunc(fx), 0, w - 1).astype(int), np.clip(np.trunc(fy), 0, h - 1).astype(int)
    safe = (np.abs(fx - np.round(fx)) > 1e-3) & (np.abs(fy - np.round(fy)) > 1e-3)
    return (iy, ix), safe


def _shade(plane, mat, lights, o, d, u_lights):
    """float64 radiance of Path / Whitted depth 1 for camera rays (o, d) (N, 3) and light draws (N, 2 * lights), plus masks and
    per-ray relative tolerances. The fold of path.rs:102-119: sum_k f(wo, wi_k) * Li_k * clamp(n_s . wi_k, 0, 1) / pdf_k."""
    p, uv, inside, edge = plane.hit(o, d)
    texel, tex_safe = _texel(mat, uv)
    wo_w = -np.asarray(d, np.float64)
    wo = plane.local(wo_w)
    L = np.zeros(p.shape)
    keep = inside & (edge > EDGE) & tex_safe
    tol = np.full(len(p), RTOL)   # the sum of positive terms errs by at most its worst term's relative error
    abs_tol = np.zeros(p.shape)
    info = {"cos": [], "fall": [], "li_nonzero": np.zeros(len(p), bool), "texel": texel}
    for k, desc in enumerate(lights):
        lt = Light(desc)
        wi_w, li, pdf, vis = lt.sample(p, plane.n, u_lights[:, 2 * k:2 * k + 2].astype(np.float64))
        # Bsdf::f (bsdfs/mod.rs:125-147): only reflection lobes, taken when wi and wo lie on the same side of n_g
        refl = (wi_w @ plane.n) * (wo_w @ plane.n) > 0.0
        f, f_err = mat.f(wo, plane.local(np.asarray(wi_w)), texel)
        f = np.where(refl[:, None], f, 0.0)
        cos = np.clip(np.asarray(wi_w) @ plane.n, 0.0, 1.0)
        term = np.where(vis[:, None], f * li * cos[:, None] / pdf[:, None], 0.0)
        L += term
        info["li_nonzero"] |= (li.max(axis=-1) > 0) & refl
        lit = refl & (li.max(axis=-1) > 0) & vis
        tol = np.maximum(tol, np.where(lit, RTOL + f_err, 0.0))
        keep &= ~(lit & (cos < COS_CUTOFF))
        info["cos"].append(np.where(lit, cos, np.nan))
        if desc.kind == D.LIGHT_SPOT:
            # the falloff's rounding: d(delta^4)/d(cos_theta) = 4 delta^3 / (cos_falloff - cos_total), times SPOT_CT_ERR
            c_tot, c_fall = lt.cone()
            ct = lt.cos_spot(p)
            delta = np.clip((ct - c_tot) / (c_fall - c_tot), 0.0, 1.0)
            blend = (ct > c_tot) & (ct < c_fall)
            slope = np.where(blend, 4.0 * delta ** 3 / (c_fall - c_tot) * SPOT_CT_ERR, 0.0)
            unit = np.where(vis[:, None] | blend[:, None], f * (lt.i / ((lt.pos - p) ** 2).sum(axis=-1)[:, None]) * cos[:, None], 0.0)
            abs_tol += slope[:, None] * unit
            info["fall"].append((ct, c_tot, c_fall))
    return np.where(inside[:, None], L, 0.0), keep, inside, tol, abs_tol, info


def _reference(plane, mat, lights):
    """(want, keep, inside-but-not-kept pixels, per-pixel tolerances, info) at the film's resolution. Delta lights: pixel
    centres; rect lights: every (pixel, sample) from its exact draws, averaged as the film does."""
    from oracle import oracle as O
    _, cam = _quad_scene()
    if not _has_rect(lights):
        w, h = DELTA_FILM.res
        ys, xs = np.mgrid[0:h, 0:w]
        pf = np.stack([xs + 0.5, ys + 0.5], axis=-1).reshape(-1, 2).astype(np.float32)
        o, d = O.camera_rays(cam, DELTA_FILM, pf)
        L, keep, inside, tol, abs_tol, info = _shade(plane, mat, lights, o, d, np.zeros((len(o), 2 * len(lights)), np.float32))
        sh = (h, w)
        info = {"cos": [c.reshape(sh) for c in info["cos"]], "fall": [tuple(np.reshape(a, sh) if np.ndim(a) else a for a in f) for f in info["fall"]],
                "li_nonzero": info["li_nonzero"].reshape(sh),
                "texel": None if mat.image is None else tuple(t.reshape(sh) for t in info["texel"])}
        return L.reshape(sh + (3,)), keep.reshape(sh), inside.reshape(sh), tol.reshape(sh), abs_tol.reshape(sh + (3,)), info
    w, h = RECT_FILM.res
    spp = RECT_SAMPLER.samples_per_pixel()
    draws = _rect_draws(len(lights))
    ys, xs = np.mgrid[0:h, 0:w]
    pf = np.stack([xs[..., None].astype(np.float32) + draws[..., 0], ys[..., None].astype(np.float32) + draws[..., 1]], axis=-1)
    o, d = O.camera_rays(cam, RECT_FILM, pf.reshape(-1, 2))
    L, keep, inside, tol, abs_tol, info = _shade(plane, mat, lights, o, d, draws[..., 2:].reshape(-1, 2 * len(lights)))
    sh = (h, w, spp)
    # a pixel is kept when all its samples are: the mean of the samples, within the largest of their tolerances
    keep_px = keep.reshape(sh).all(axis=-1) | ~inside.reshape(sh).any(axis=-1)
    keep_px &= inside.reshape(sh).all(axis=-1) | ~inside.reshape(sh).any(axis=-1)
    info = {"cos": [c.reshape(sh) for c in info["cos"]], "fall": [(f[0].reshape(sh),) + f[1:] for f in info["fall"]],
            "li_nonzero": info["li_nonzero"].reshape(sh).any(axis=-1)}
    return (L.reshape(sh + (3,)).mean(axis=2), keep_px, inside.reshape(sh).any(axis=-1), tol.reshape(sh).max(axis=-1),
            abs_tol.reshape(sh + (3,)).max(axis=2), info)


def _check(img, ref, what=""):
    want, keep, inside, tol, abs_tol, _ = ref
    got = np.asarray(img, np.float64)
    err = np.abs(got - want)
    bound = tol[..., None] * want + abs_tol
    bad = keep[..., None] & (err > bound)
    assert not bad.any(), (what, int(bad.any(axis=-1).sum()), float((err / np.maximum(want, 1e-30))[bad].max()))
    zero = keep & (want.max(axis=-1) == 0.0)
    assert np.all(got[zero] == 0.0), what   # a light facing away, a spot's outside, a light below the plane: exactly 0
    assert np.all(got[~inside] == 0.0), what   # black background


def _film_sampler(lights):
    return (RECT_FILM, RECT_SAMPLER) if _has_rect(lights) else (DELTA_FILM, DELTA_SAMPLER)


def _claims(plane, mat, light_name, lights, ref, img, st):
    """What the case names must occur in it, in enough pixels."""
    want, keep, inside, _, _, info = ref
    lit = keep & (want.max(axis=-1) > 0)
    min_px = 300 if _has_rect(lights) else 1500
    if light_name == "rect-away":
        assert np.all(img == 0.0) and st.shadow_rays == 0 and inside.sum() > 500   # one-sided: no radiance, no shadow ray
        return
    assert lit.sum() > min_px
    assert (keep & inside).sum() > 0.8 * inside.sum(), "the masks leave out too much"
    if light_name == "point-low":
        cos = info["cos"][0]
        assert (keep & (cos < 0.3)).sum() > 800   # grazing incidence
    if light_name in ("spot", "all-four"):
        ct, c_tot, c_fall = info["fall"][0]
        if ct.ndim == 3:   # rect film: count (pixel, sample) pairs of kept pixels
            keep, inside = np.repeat(keep[..., None], ct.shape[2], axis=2), np.repeat(inside[..., None], ct.shape[2], axis=2)
        margin = np.cos(np.deg2rad(30.0 - 0.05)) - c_tot   # a twentieth of a degree inside the cone edge
        assert (keep & (ct > c_fall + 1e-4)).sum() > 300      # inside the inner cone
        assert (keep & (ct < c_fall - 1e-4) & (ct > c_tot + margin)).sum() > 300   # in the blend
        outside = inside & (ct < c_tot - margin)
        assert outside.sum() > 300
        if light_name == "spot":
            assert np.all(img[outside] == 0.0)   # no radiance and no shadow ray outside the cone
    if light_name == "distant-non-unit":
        assert abs(np.linalg.norm(np.float32(lights[0].direction)) - 0.7) < 1e-6
    if mat.image is not None:
        iy, ix = info["texel"]
        for ty in range(mat.image.shape[0]):
            for tx in range(mat.image.shape[1]):
                assert (lit & (iy == ty) & (ix == tx)).sum() > 60, (ty, tx)   # every texel, 5e-4 (below the floor) included


def _cases():
    out = []
    for plane in PLANES:
        for light in LIGHT_NAMES:
            for mat in MATERIALS:
                out.append(f"{plane}-{mat}-{light}")
        for mat in IMAGE_MATERIALS:
            for light in ("point-high", "point-low"):
                out.append(f"{plane}-{mat}-{light}")
    return out


CASES = _cases()


def _case(case):
    plane_name = next(p for p in PLANES if case.startswith(p + "-"))
    rest = case[len(plane_name) + 1:]
    light_name = next(l for l in sorted(LIGHT_NAMES, key=len, reverse=True) if rest.endswith("-" + l))
    mat_name = rest[:-(len(light_name) + 1)]
    mat = MATERIALS.get(mat_name) or IMAGE_MATERIALS[mat_name]
    return PLANES[plane_name], mat, light_name, LIGHTS[plane_name][light_name]


def _scene(plane, mat, lights):
    scene, cam = plane.scene(mat)
    scene.lights = list(lights)
    return scene, cam


@pytest.mark.parametrize("case", CASES)
def test_oracle_direct_lighting_matches_float64(oracle, case):
    plane, mat, light_name, lights = _case(case)
    scene, cam = _scene(plane, mat, lights)
    film, smp = _film_sampler(lights)
    osc = oracle.OracleScene(scene)
    img, ids, st = osc.render(cam, film, smp, D.IntegratorType.path(1), want_hit_ids=True)
    img_w, _, _ = osc.render(cam, film, smp, D.IntegratorType.whitted(1))
    assert np.array_equal(img.view(np.uint32), img_w.view(np.uint32))   # the fold is the whole film at depth 1 of both
    ref = _reference(plane, mat, lights)
    _check(img, ref, case)
    _claims(plane, mat, light_name, lights, ref, img, st)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_gpu_direct_lighting_matches_float64_and_the_oracle(gpu_ctx, oracle, case):
    plane, mat, _, lights = _case(case)
    scene, cam = _scene(plane, mat, lights)
    film, smp = _film_sampler(lights)
    o_img, o_ids, o_st = oracle.OracleScene(scene).render(cam, film, smp, D.IntegratorType.path(1), want_hit_ids=True)
    dev = api.Scene(gpu_ctx, scene)
    try:
        rn = api.Renderer(gpu_ctx)
        r = rn.render(dev, cam, film, smp, D.IntegratorType.path(1), want_hit_ids=True)
        rw = rn.render(dev, cam, film, smp, D.IntegratorType.whitted(1))
    finally:
        dev.close()
    assert np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32)) and np.array_equal(r.hit_ids, o_ids), case
    assert r.stats.shadow_rays == o_st.shadow_rays, case
    assert np.array_equal(rw.film.view(np.uint32), r.film.view(np.uint32)), case
    _check(r.film, _reference(plane, mat, lights), case)


# ---- image-textured roughness: the device's roughness_to_alpha against the host's --------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", [D.MAT_METAL, D.MAT_GLOSSY], ids=["metal", "glossy"])
@pytest.mark.parametrize("remap", [False, True], ids=["raw", "remap"])
def test_gpu_constant_roughness_equals_a_1x1_image_of_it(gpu_ctx, kind, remap):
    """A constant roughness becomes alpha on the host at scene creation (glibc's logf, render.cu); an image texel goes through
    the device's roughness_to_alpha and restated logf per hit. A 1x1 image of the same value must give the same film bits."""
    rn = api.Renderer(gpu_ctx)
    for r in (5e-4, 1e-3, 0.01, 0.05, 0.2, 0.7, 1.0):
        films = []
        for image in (False, True):
            scene, cam = _quad_scene()
            rough = scene.add_texture(D.Texture.from_image(np.full((1, 1, 3), r, np.float32)) if image else D.Texture.constant(r))
            if kind == D.MAT_METAL:
                tex = (scene.add_texture(D.Texture.constant(*COPPER_ETA)), scene.add_texture(D.Texture.constant(*COPPER_K)), rough)
            else:
                tex = (scene.add_texture(D.Texture.constant(*GLOSSY_RS)), rough)
            scene.meshes[0].material = scene.add_material(D.Material(kind, tex, remap_roughness=remap))
            scene.lights = LIGHTS["flat"]["point-high"] + LIGHTS["flat"]["point-low"]
            dev = api.Scene(gpu_ctx, scene)
            try:
                films.append(rn.render(dev, cam, DELTA_FILM, DELTA_SAMPLER, D.IntegratorType.path(1)).film)
            finally:
                dev.close()
        assert films[0].max() > 0 and np.array_equal(films[0].view(np.uint32), films[1].view(np.uint32)), r


# ---- 3. Whitted through a glass slab, against a float64 recursion -------------------------------------------------------
GLASS_R, GLASS_T, GLASS_ETA = (0.8, 0.75, 0.7), (0.6, 0.65, 0.7), 1.5   # R != T: the test sees which weight goes where
FLOOR_KD, SKY = (0.6, 0.5, 0.4), (0.2, 0.3, 0.4)                      # a sky, so that escaping reflections count too
SLAB_HALF, SLAB_TOP, SLAB_BOTTOM = 0.5, 0.6, 0.4
SLAB_LIGHT, SLAB_LIGHT_I = (2.5, 0.3, 1.2), (6.0, 5.0, 4.0)
SLAB_CAM = D.CameraParameters((0.15, -0.35, 2.6), (0.0, 0.0, 0.0), fov_axis=D.FOV_X, fov_deg=40.0)
SLAB_FILM, SLAB_SAMPLER = D.FilmSettings((64, 48), 16), D.SamplerType.stratified(1, 1, jitter=False)
WHITTED_DEPTHS = (2, 3, 5, 8)
WEDGE_DEG = 16.0        # the wedge's bottom face tilts by this about y: internal rays gain 2 * 16 deg per reflection, and
                        # pass the critical angle (41.8 deg) at their second reflection off the bottom
SPAWN_OFFSET = 1e-3     # interaction.rs:27-59
EDGE_W = 2e-3           # rays (and shadow segments) that pass within this of a quad's outline are left out
COS_T_CUTOFF = 0.05     # nodes whose transmitted |cos theta_t| is below this (within ~3 deg of the critical angle) are left out
# Relative tolerance of a Whitted pixel. One node's weight R * Fr or T * (1 - Fr), computed in float32 as f = R * Fr / |cos|
# times |cos|, carries ~30 roundings of 2^-24 (1.8e-6); a floor leaf adds the fold's ~10, and the sum up the tree one per
# level. Directions: each reflection or refraction turns the float32 ray by ~1 ulp of a unit vector (1e-7 rad), which changes
# the next Fresnel term by |d ln Fr / d theta| * 1e-7 <= 5e-7 away from the critical angle (COS_T_CUTOFF) and moves the next
# hit by ~3e-7, negligible for the floor's I / d^2 at d >= 1. Seven nodes deep (depth 8): 7 * (1.8e-6 + 5e-7) = 1.6e-5.
# (The oracle's worst pixel is 5e-7 off at every depth.)
WHITTED_RTOL = 3e-5


def _quad(corners):
    return np.array(corners, np.float32), np.array([0, 1, 2, 0, 2, 3], np.uint32)


def slab_scene(wedge=False):
    """A Lambertian floor z = 0 under a glass slab (two quads with outward normals, +z on top, -z below), lit by one point
    light to the side. With `wedge`, the bottom quad tilts by WEDGE_DEG about y, so that internal rays reach total internal
    reflection. Returns the scene and the quads' float32 corners (floor, top, bottom)."""
    s = D.SceneDesc(background=SKY)
    zero = s.add_texture(D.Texture.constant(0.0))
    floor = s.add_material(D.Material(D.MAT_MATTE, (s.add_texture(D.Texture.constant(*FLOOR_KD)), zero)))
    glass = s.add_material(D.Material(D.MAT_GLASS, (s.add_texture(D.Texture.constant(*GLASS_R)), s.add_texture(D.Texture.constant(*GLASS_T))),
                                      eta=GLASS_ETA))
    h, slope = SLAB_HALF, np.tan(np.deg2rad(WEDGE_DEG)) if wedge else 0.0
    zb = lambda x: SLAB_BOTTOM + slope * x
    quads = [
        ([(-2, -2, 0), (2, -2, 0), (2, 2, 0), (-2, 2, 0)], floor),
        ([(-h, -h, SLAB_TOP), (h, -h, SLAB_TOP), (h, h, SLAB_TOP), (-h, h, SLAB_TOP)], glass),
        ([(-h, -h, zb(-h)), (-h, h, zb(-h)), (h, h, zb(h)), (h, -h, zb(h))], glass),   # reversed: normal -z (outward)
    ]
    corners = []
    for c, m in quads:
        p, idx = _quad(c)
        s.meshes.append(D.Mesh(xf.identity(), p, idx, m))
        corners.append(p.astype(np.float64))
    s.lights.append(D.Light(D.LIGHT_POINT, xf.translation(SLAB_LIGHT), SLAB_LIGHT_I))
    return s, corners


def _quad_hits(corners, o, d):
    """float64 ray / quad: t (inf when missed or behind), and the signed distance of the plane point to the outline."""
    v0, v1, v2, v3 = corners
    n = np.cross(v0 - v2, v1 - v2)
    n /= np.linalg.norm(n)
    e1, e2 = v1 - v0, v3 - v0   # orthogonal edges
    with np.errstate(divide="ignore", invalid="ignore"):   # rays parallel to the plane: t = +-inf, then NaN, both a miss
        t = ((v0 - o) @ n) / (d @ n)
        q = o + t[:, None] * d - v0
        a, b = (q @ e1) / (e1 @ e1), (q @ e2) / (e2 @ e2)
        edge = np.minimum(np.minimum(a, 1 - a) * np.linalg.norm(e1), np.minimum(b, 1 - b) * np.linalg.norm(e2))
    ok = (t > 0) & (edge > 0)
    return np.where(ok, t, np.inf), np.where(t > 0, edge, np.inf), n


def fr_dielectric(c, eta_t):
    """fresnel.rs:21-51 with eta_i = 1: the side is the sign of cos, and sin_t >= 1 reflects totally."""
    c = np.clip(c, -1.0, 1.0)
    entering = c > 0
    ei, et = np.where(entering, 1.0, eta_t), np.where(entering, eta_t, 1.0)
    c = np.abs(c)
    st = ei / et * np.sqrt(np.maximum(1.0 - c * c, 0.0))
    ct = np.sqrt(np.maximum(1.0 - st * st, 0.0))
    r_par = (et * c - ei * ct) / (et * c + ei * ct)
    r_perp = (ei * c - et * ct) / (ei * c + et * ct)
    return np.where(st >= 1.0, 1.0, (r_par ** 2 + r_perp ** 2) / 2.0)


def whitted_reference(oracle, corners, max_depth):
    """float64 Whitted radiance of every pixel centre: the tree of whitted.rs:74-182, enumerated level by level. A node adds
    its light fold (floor: kd/pi * I/d^2 * cos if the segment to the light misses the slab; glass: f = 0) and, while
    depth + 1 < max_depth, f * li(child) * |cos| for its reflection child, weight R * Fr(cos), and its transmission child,
    weight T * (1 - Fr) at the transmitted cosine without an eta^2 factor (specular.rs:26-37, 69-92), each spawned 1e-3
    along +-n (interaction.rs:27-59). Returns the film, the pixels kept, and counts of what the tree met."""
    w_res, h_res = SLAB_FILM.res
    ys, xs = np.mgrid[0:h_res, 0:w_res]
    pf = np.stack([xs + 0.5, ys + 0.5], axis=-1).reshape(-1, 2).astype(np.float32)
    o, d = (a.astype(np.float64) for a in oracle.camera_rays(SLAB_CAM, SLAB_FILM, pf))
    n_px = len(o)
    pix, wgt = np.arange(n_px), np.ones((n_px, 3))
    L, flag = np.zeros((n_px, 3)), np.zeros(n_px, bool)
    R, T, kd, sky, li = (np.asarray(F32(v), np.float64) for v in (GLASS_R, GLASS_T, FLOOR_KD, SKY, SLAB_LIGHT_I))
    light = np.asarray(F32(SLAB_LIGHT), np.float64)
    counts = {"floor": np.zeros(n_px, int), "sky": 0, "tir": 0, "shadowed": np.zeros(n_px, bool), "glass_nodes": 0, "deepest": 0}
    for depth in range(max_depth):
        if len(o) == 0:
            break
        hits = [_quad_hits(c, o, d) for c in corners]
        t = np.stack([h[0] for h in hits], axis=1)
        near = np.stack([np.abs(h[1]) < EDGE_W for h in hits], axis=1).any(axis=1)
        flag[pix[near]] = True
        which = np.where(np.isfinite(t).any(axis=1), t.argmin(axis=1), -1)
        tb = t[np.arange(len(o)), np.maximum(which, 0)]
        p = o + np.where(which >= 0, tb, 0.0)[:, None] * d
        counts["deepest"] = max(counts["deepest"], depth if (which > 0).any() else 0)
        # misses: the sky
        miss = which < 0
        np.add.at(L, pix[miss], wgt[miss] * sky)
        counts["sky"] += int(miss.sum())
        # floor: point light, Lambert (no specular children)
        fl = which == 0
        if fl.any():
            pf_, pixf = p[fl], pix[fl]
            to = light - pf_
            d2 = (to * to).sum(axis=1)
            wi = to / np.sqrt(d2)[:, None]
            so = pf_ + np.array([0.0, 0.0, SPAWN_OFFSET])   # spawn_ray_to: light above the floor, offset along +n
            seg = light - so
            blocked = np.zeros(len(pf_), bool)
            for c in corners[1:]:   # the shadow segment, t_max = 0.9999 of (light - origin), against the slab's quads
                ts, es, _ = _quad_hits(c, so, seg)
                blocked |= ts < 0.9999
                flag[pixf[np.abs(es) < EDGE_W]] = True
            term = kd / np.pi * li / d2[:, None] * np.clip(wi[:, 2], 0.0, 1.0)[:, None]
            np.add.at(L, pixf, np.where(blocked[:, None], 0.0, wgt[fl] * term))
            np.add.at(counts["floor"], pixf, 1)
            counts["shadowed"][pixf[blocked]] = True
        # glass: no light (specular f = 0); the children
        gl = which > 0
        counts["glass_nodes"] += int(gl.sum())
        if depth + 1 >= max_depth or not gl.any():
            break
        n = np.stack([hits[k][2] for k in range(len(corners))])[which[gl]]
        pg, wo, wg, pixg = p[gl], -d[gl], wgt[gl], pix[gl]
        cos_o = (wo * n).sum(axis=1)
        refl = -wo + 2.0 * cos_o[:, None] * n
        w_refl = wg * R * fr_dielectric(cos_o, GLASS_ETA)[:, None]
        entering = cos_o > 0
        eta = np.where(entering, 1.0 / GLASS_ETA, GLASS_ETA)
        nf = np.where(entering[:, None], n, -n)
        ci = np.abs(cos_o)
        s2t = eta * eta * np.maximum(1.0 - ci * ci, 0.0)
        tir = s2t >= 1.0
        counts["tir"] += int(tir.sum())
        flag[pixg[np.abs(1.0 - s2t) < COS_T_CUTOFF ** 2]] = True
        ct = np.sqrt(np.maximum(1.0 - s2t, 0.0))
        trans = (-wo * eta[:, None] + nf * (eta * ci - ct)[:, None])[~tir]
        w_trans = wg[~tir] * T * (1.0 - fr_dielectric((trans * n[~tir]).sum(axis=1), GLASS_ETA))[:, None]
        new_d = np.concatenate([refl, trans])
        new_p = np.concatenate([pg, pg[~tir]])
        new_n = np.concatenate([n, n[~tir]])
        side = np.where(((new_d * new_n).sum(axis=1) > 0)[:, None], 1.0, -1.0)
        o, d = new_p + side * SPAWN_OFFSET * new_n, new_d
        wgt = np.concatenate([w_refl, w_trans])
        pix = np.concatenate([pixg, pixg[~tir]])
    sh = (h_res, w_res)
    counts["floor"], counts["shadowed"] = counts["floor"].reshape(sh), counts["shadowed"].reshape(sh)
    return L.reshape(sh + (3,)), ~flag.reshape(sh), counts


def _check_whitted(img, want, keep, what):
    got = np.asarray(img, np.float64)
    err = np.abs(got - want)
    bad = keep[..., None] & (err > WHITTED_RTOL * want)
    assert not bad.any(), (what, int(bad.any(axis=-1).sum()), float((err / np.maximum(want, 1e-30))[bad].max()))


WHITTED_CASES = [(wedge, depth) for wedge in (False, True) for depth in WHITTED_DEPTHS]
WHITTED_IDS = [("wedge" if w else "slab") + f"-depth-{d}" for w, d in WHITTED_CASES]


@pytest.mark.parametrize("wedge,depth", WHITTED_CASES, ids=WHITTED_IDS)
def test_oracle_whitted_glass_matches_float64(oracle, wedge, depth):
    scene, corners = slab_scene(wedge)
    img, ids, st = oracle.OracleScene(scene).render(SLAB_CAM, SLAB_FILM, SLAB_SAMPLER, D.IntegratorType.whitted(depth), want_hit_ids=True)
    want, keep, counts = whitted_reference(oracle, corners, depth)
    _check_whitted(img, want, keep, (wedge, depth))
    through = keep & (ids >= 2)   # camera ray hits the slab's top (triangles 2, 3)
    assert through.sum() > 400 and keep.sum() > 0.85 * keep.size
    assert (keep & (ids < 2) & ~counts["shadowed"]).sum() > 500
    if not wedge:   # the slab shadows part of the floor seen beside it (glass occludes)
        assert (keep & (ids < 2) & counts["shadowed"]).sum() > 100
    if depth >= 3:   # the floor is reached through the slab: top, bottom, floor
        assert (through & (counts["floor"] > 0)).sum() > 300
    if depth >= 5:
        assert (through & (counts["floor"] > 1)).sum() > 200   # and again after internal reflections
    if wedge and depth >= 5:
        assert counts["tir"] > 200
    if not wedge:
        assert counts["tir"] == 0   # parallel faces: a ray that entered can always leave


def test_path_depth_1_sees_no_light_through_the_slab(oracle):
    """Glass has f = 0 and no emission: at Path depth 1 a pixel through the slab is exactly black, the floor beside it lit."""
    scene, corners = slab_scene()
    img, ids, _ = oracle.OracleScene(scene).render(SLAB_CAM, SLAB_FILM, SLAB_SAMPLER, D.IntegratorType.path(1), want_hit_ids=True)
    assert (ids >= 2).sum() > 400 and np.all(img[ids >= 2] == 0.0)
    assert (img[(ids >= 0) & (ids < 2)].max(axis=-1) > 0).sum() > 500 and np.all(img[ids < 0] == np.float32(SKY))


@pytest.mark.gpu
@pytest.mark.parametrize("wedge,depth", WHITTED_CASES, ids=WHITTED_IDS)
def test_gpu_whitted_glass_matches_float64_and_the_oracle(gpu_ctx, oracle, wedge, depth):
    scene, corners = slab_scene(wedge)
    integ = D.IntegratorType.whitted(depth)
    o_img, o_ids, o_st = oracle.OracleScene(scene).render(SLAB_CAM, SLAB_FILM, SLAB_SAMPLER, integ, want_hit_ids=True)
    dev = api.Scene(gpu_ctx, scene)
    try:
        r = api.Renderer(gpu_ctx).render(dev, SLAB_CAM, SLAB_FILM, SLAB_SAMPLER, integ, want_hit_ids=True)
    finally:
        dev.close()
    assert np.array_equal(r.film.view(np.uint32), o_img.view(np.uint32)) and np.array_equal(r.hit_ids, o_ids)
    assert r.stats.ray_count == o_st.ray_count and r.stats.shadow_rays == o_st.shadow_rays
    want, keep, _ = whitted_reference(oracle, corners, depth)
    _check_whitted(r.film, want, keep, (wedge, depth))
