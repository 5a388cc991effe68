"""Path's second and later vertices, sample by sample, against float64 restatements of the reference.

test_direct_lighting.py pins the first vertex (every lobe's f, every light's sample_li, the light fold); this file pins what
makes Path a path (path.rs:49-178): the lobes' sample_f, the throughput update beta *= f |n_s . wi| / pdf with the glass
pick's pdf / 2, emission after a specular bounce (beta applied twice, a reference quirk), the indirect clamp at bounces > 0,
and Russian roulette q = max(1 - beta.g, 0.05) with beta /= 1 - q. The sampler's draws are fixed by (pixel, sample,
dimension), so each sample's radiance is a deterministic function of them: a float64 walk over the analytic planes and
spheres evaluates it, from the float32 draws and camera rays the renderer receives (both pinned elsewhere), and every
per-sample film (an accumulating film rendered onto zeros one sample index at a time) is compared with it.

1. Each lobe's sample_f in float64 against `oracle.lobe_sample`, over a grid of wo and the edge draws.
2. Paths sample by sample: two planes, a glass slab under an area light, a corridor for Russian roulette, the indirect
   clamp, and rotated and scaled spheres. Each sample carries its own error bound, summed along its path (see _walk).
3. The reflection and refraction rays `debug_ray` logs against the float64 sampled directions.

Every case has a CPU part (the oracle against float64, plus asserts that the case reaches what it claims) and a GPU part
(the GPU's per-sample films bit-equal to the oracle's and within the same float64 bound).
"""
import functools

import numpy as np
import pytest

from test_direct_lighting import (COPPER_ETA, COPPER_K, COS_CUTOFF, COS_T_CUTOFF, EDGE_W, EPS32, GLASS_ETA, GLASS_R,
                                  GLASS_T, IMAGE_MATERIALS, RTOL, SLAB_CAM, SPAWN_OFFSET, SPHERES, Light, Mat, _materials,
                                  _texel, fr_conductor, fr_dielectric, fr_schlick, ggx_d, microfacet_f, slab_scene)
from yuki_b200 import api, desc as D, transforms as xf

F32 = np.float32
MATERIALS = {**_materials(), **IMAGE_MATERIALS}
LOBE_DIFFUSE, LOBE_GLOSSY, LOBE_SPEC_R, LOBE_SPEC_T = 5, 9, 17, 18   # BxdfType flags (bsdfs/mod.rs:25-35)


# ---- 1. sample_f in float64 (local frame, z = n_s) ----------------------------------------------------------------------
def concentric_disk(u):
    """sampling/mod.rs:68-87."""
    off = 2.0 * u - 1.0
    ox, oy = off[:, 0], off[:, 1]
    big_x = np.abs(ox) > np.abs(oy)
    with np.errstate(divide="ignore", invalid="ignore"):
        theta = np.where(big_x, np.pi / 4 * (oy / ox), np.pi / 2 - np.pi / 4 * (ox / oy))
    r = np.where(big_x, ox, oy)
    d = r[:, None] * np.stack([np.cos(theta), np.sin(theta)], -1)
    return np.where(((ox == 0) & (oy == 0))[:, None], 0.0, d)


def diffuse_sample(wo, u):
    """lambertian.rs:25-40 / oren_nayar.rs:55-70: cosine_sample_hemisphere (sampling/mod.rs:62-66), z flipped when
    wo.z < 0; pdf = |cos| / pi on the same side, else 0 (no sample). Also the float32 direction error (rad) and whether the
    no-sample decision lies within rounding (|z| within rounding of 0)."""
    d = concentric_disk(u)
    z = np.sqrt(np.maximum(1.0 - (d * d).sum(-1), 0.0))
    z = np.where(wo[:, 2] < 0, -z, z)
    wi = np.concatenate([d, z[:, None]], -1)
    ok = wo[:, 2] * z > 0
    # 1 - x^2 - y^2 carries ~6 roundings of 2^-24 and its sqrt turns them into ~3 ulp / |z|; the disk map adds ~8
    with np.errstate(divide="ignore"):
        err = EPS32 * (12.0 + 4.0 / np.abs(z))
    band = np.abs(z) < 8.0 * np.sqrt(EPS32)
    return wi, np.where(ok, np.abs(z) / np.pi, 0.0), ok, err, band


def ggx_sample(alpha, wo, u):
    """microfacet.rs:76-99 with tr_sample_wh (trowbridge_reitz.rs:60-74, the full distribution): wh from (u.x, u.y),
    flipped into wo's hemisphere, wi = reflect(wo, wh), pdf = D(wh) cos_h / (4 wo . wh) (no abs: negative below the
    surface, as written). No sample when wo.z = 0, wo . wh < 0 or wi leaves wo's hemisphere. Also wh, the float32 error of
    wh and of wi (rad), and the decisions within rounding."""
    ux, uy = u[:, 0], u[:, 1]
    with np.errstate(divide="ignore", invalid="ignore"):
        tan2 = alpha * alpha * ux / (1.0 - ux)     # u.x = 1: infinite, cos_t = 0
        cos_t = 1.0 / np.sqrt(1.0 + tan2)
    phi = 2.0 * np.pi * uy
    sin_t = np.sqrt(np.maximum(1.0 - cos_t * cos_t, 0.0))
    wh = np.stack([sin_t * np.cos(phi), sin_t * np.sin(phi), cos_t], -1)
    wh = np.where((wo[:, 2] * wh[:, 2] > 0)[:, None], wh, -wh)
    dot_ow = (wo * wh).sum(-1)
    wi = -wo + 2.0 * dot_ow[:, None] * wh
    ok = (wo[:, 2] != 0) & (dot_ow >= 0) & (wo[:, 2] * wi[:, 2] > 0)
    with np.errstate(divide="ignore", invalid="ignore"):
        pdf = np.where(ok, ggx_d(alpha, wh) * wh[:, 2] / (4.0 * dot_ow), 0.0)
        # float32: tan2 and cos_t carry ~4 roundings, phi 2, the trig 1 each; sin_t = sqrt(1 - cos^2) cancels for small
        # theta_h, where 1 - cos^2 errs by ~5 ulp of cos^2: theta_h errs by 2.5 ulp / (sin cos), at most sqrt(5 ulp) / cos
        e_wh = np.where(tan2 == 0, 0.0, np.minimum(3.0 * EPS32 / (sin_t * cos_t), 3.0 * np.sqrt(EPS32) / cos_t)) + 16.0 * EPS32
    e_wh = np.where(np.isfinite(e_wh), e_wh, np.inf)
    band = (np.abs(dot_ow) <= 2.0 * e_wh + 8.0 * EPS32) | (np.abs(wi[:, 2]) <= 4.0 * e_wh + 16.0 * EPS32)
    return wi, wh, np.where(ok, pdf, 0.0), ok, e_wh, 2.0 * e_wh + 8.0 * EPS32, band


def _fresnel(mat):
    f64 = lambda c: np.asarray(F32(c), np.float64)
    if mat.kind == D.MAT_METAL:
        return lambda c: fr_conductor(f64(mat.params["eta"]), f64(mat.params["k"]), c)
    return lambda c: fr_schlick(f64(mat.params["rs"]), c)


def d_slope(alpha, wh):
    """|d ln D / d theta_h| of the isotropic GGX D = a^2 / (pi cos^4 (a^2 + t^2)^2), t = tan theta_h: 4t + 4t (1 + t^2) /
    (a^2 + t^2); at most 2 / alpha near the peak."""
    t = np.sqrt(np.maximum(1.0 - wh[:, 2] ** 2, 0.0)) / np.abs(wh[:, 2])
    return 4.0 * t + 4.0 * t * (1.0 + t * t) / (alpha * alpha + t * t)


def glass_sample(wo, u, R, T, eta):
    """Bsdf::sample_f over glass's two specular lobes (bsdfs/mod.rs:150-222): comp = floor(2 u.x) clamped to 1 (exact in
    float32: no rounding band), the lobe's sample (specular.rs:26-37 reflection, :69-92 transmission without an eta^2 factor,
    total internal reflection: no sample), then pdf = 1 / 2. Returns wi, f, pdf, ok, which lobe (1: transmission), cos_t, and
    whether the transmitted cosine is within COS_T_CUTOFF of 0 (the refraction or its Fresnel term near the critical angle)."""
    comp = np.minimum(np.floor(u[:, 0] * 2.0), 1.0).astype(int)
    c = wo[:, 2]
    refl = np.stack([-wo[:, 0], -wo[:, 1], c], -1)
    entering = c > 0
    e = np.where(entering, 1.0 / eta, eta)
    nf = np.where(entering | (c == 0), 1.0, -1.0)   # faceforward((0, 0, 1), wo)
    ci = np.abs(c)
    s2t = e * e * np.maximum(1.0 - ci * ci, 0.0)
    tir = s2t >= 1.0
    ct = np.sqrt(np.maximum(1.0 - s2t, 0.0))
    trans = -wo * e[:, None] + np.stack([np.zeros_like(c), np.zeros_like(c), nf], -1) * (e * ci - ct)[:, None]
    wi = np.where((comp == 1)[:, None], trans, refl)
    with np.errstate(divide="ignore", invalid="ignore"):
        f_r = np.asarray(R)[None, :] * fr_dielectric(c, eta)[:, None] / np.abs(c)[:, None]
        f_t = np.asarray(T)[None, :] * (1.0 - fr_dielectric(trans[:, 2], eta))[:, None] / np.abs(trans[:, 2])[:, None]
    f = np.where((comp == 1)[:, None], f_t, f_r)
    ok = (comp == 0) | ~tir
    near_critical = (comp == 1) & (np.abs(1.0 - s2t) < COS_T_CUTOFF ** 2)
    return wi, np.where(ok[:, None], f, 0.0), np.where(ok, 0.5, 0.0), ok, comp, np.where(comp == 1, ct, 1.0), near_critical


def _lobe_cases():
    """(name, oracle lobe kind, oracle params, material, alpha): one per material of _materials() (alpha as the float32
    the lobe receives; None for the diffuse lobes) plus copper at the 1e-3 alpha floor."""
    from oracle import oracle as O
    out = []
    for m in _materials().values():
        p = m.params
        if m.kind == D.MAT_MATTE:
            sigma = float(F32(p["sigma"]))
            out.append((m.name, O.LOBE_LAMBERT if sigma == 0 else O.LOBE_OREN_NAYAR, list(p["kd"]) + [sigma], m, None))
            continue
        alpha = float(F32(m.alpha(np.float64(F32(p["rough"])))))
        if m.kind == D.MAT_METAL:
            out.append((m.name, O.LOBE_GGX_CONDUCTOR, [1, 1, 1] + list(COPPER_ETA) + list(COPPER_K) + [alpha], m, alpha))
        else:
            out.append((m.name, O.LOBE_GGX_SCHLICK, [1, 1, 1] + list(p["rs"]) + [alpha], m, alpha))
    out.append(("copper-a1e-3-floor", O.LOBE_GGX_CONDUCTOR, [1, 1, 1] + list(COPPER_ETA) + list(COPPER_K) + [1e-3],
                Mat("copper-floor", D.MAT_METAL, {"eta": COPPER_ETA, "k": COPPER_K, "rough": 1e-3}), float(F32(1e-3))))
    return out


def _wo_grid():
    """Unit wo over theta in [0, 180] deg (z < 0 included), grazing within 1e-4 of the horizon, and z = 0 exactly."""
    th = np.concatenate([np.linspace(0.0, np.pi, 31), [1e-4, np.pi / 2 - 1e-4, np.pi / 2 - 0.02, np.pi / 2 + 1e-4, np.pi - 1e-4]])
    ph = np.linspace(0.1, 2 * np.pi, 7, endpoint=False)
    t, p = np.meshgrid(th, ph)
    w = np.stack([np.sin(t) * np.cos(p), np.sin(t) * np.sin(p), np.cos(t)], -1).reshape(-1, 3).astype(F32)
    w[np.abs(np.cos(t.ravel()) ) < 1e-12, 2] = 0.0   # theta = 90 deg: z = 0 exactly
    return w


def _edge_draws():
    """u = 0, 0.5 (the glass pick and the disk's centre), 1 - 2^-24, 1.0f exactly, and a jittered grid."""
    edge = np.array([0.0, 0.5, 1.0 - 2.0 ** -24, 1.0, 0.25, 0.75, 2.0 ** -24], F32)
    ex, ey = np.meshgrid(edge, edge)
    rng = np.random.default_rng(7)
    return np.concatenate([np.stack([ex.ravel(), ey.ravel()], -1), rng.random((60, 2)).astype(F32)]).astype(F32)


def _lobe_compare(name, kind, params, mat, alpha):
    from oracle import oracle as O
    wo_g, u_g = _wo_grid(), _edge_draws()
    wo32 = np.repeat(wo_g, len(u_g), axis=0)
    u32 = np.tile(u_g, (len(wo_g), 1))
    g_wi, g_f, g_pdf, g_type = O.lobe_sample(kind, params, wo32, u32)
    wo, u = wo32.astype(np.float64), u32.astype(np.float64)
    tex = np.zeros(len(wo), int)
    if alpha is None:   # diffuse
        wi, pdf, ok, e_wi, band = diffuse_sample(wo, u)
        f, _ = mat.f(wo, wi, tex)
        f = np.where(ok[:, None], f, 0.0)
        f_rtol = np.full(len(wo), RTOL)
        with np.errstate(divide="ignore"):
            pdf_rtol = 2.0 * EPS32 + e_wi / np.abs(wi[:, 2])
        want_type = LOBE_DIFFUSE
        slope = 0.0 if kind == O.LOBE_LAMBERT else 8.0 / np.maximum(np.minimum(np.abs(wo[:, 2]), np.abs(wi[:, 2])), COS_CUTOFF)
        f_rtol = f_rtol + slope * e_wi
    else:
        wi, wh, pdf, ok, e_wh, e_wi, band = ggx_sample(alpha, wo, u)
        fr = _fresnel(mat)
        with np.errstate(divide="ignore", invalid="ignore"):
            f, d_err = microfacet_f(alpha, fr, wo, wi)
            sd = d_slope(alpha, wh)
            wsum = np.linalg.norm(wo + wi, axis=-1)
            cosmin = np.maximum(np.minimum(np.abs(wo[:, 2]), np.abs(wi[:, 2])), 1e-6)
            f_rtol = RTOL + d_err + sd * (e_wh + 24.0 * EPS32 / wsum) + 8.0 * e_wi / cosmin
            pdf_rtol = RTOL + d_err + sd * e_wh + 8.0 * e_wh / np.maximum((wo * wh).sum(-1), 1e-12)
        f = np.where(ok[:, None], f, 0.0)
        want_type = LOBE_GLOSSY
    return _lobe_assert(name, ok, band, want_type, wi, f, pdf, e_wi, f_rtol, pdf_rtol, g_wi, g_f, g_pdf, g_type)


def _lobe_assert(name, ok, band, want_type, wi, f, pdf, e_wi, f_rtol, pdf_rtol, g_wi, g_f, g_pdf, g_type):
    g_ok = (g_type != 0) & (g_pdf != 0)   # a lobe's pdf of 0 is no sample to Bsdf::sample_f (bsdfs/mod.rs:177-180)
    sure = ~band
    assert np.array_equal(g_ok[sure], ok[sure]), (name, int((g_ok != ok)[sure].sum()))
    assert np.all(g_type[g_ok] == want_type), name
    both = ok & g_ok & sure
    d_err = np.linalg.norm(g_wi[both] - wi[both], axis=-1)
    assert np.all(d_err <= e_wi[both]), (name, float((d_err / e_wi[both]).max()))
    with np.errstate(divide="ignore", invalid="ignore"):
        fr = np.abs(g_f[both] - f[both]) / np.abs(f[both])
        pr = np.abs(g_pdf[both] - pdf[both]) / np.abs(pdf[both])
    fb = np.broadcast_to(f_rtol, ok.shape)[both]
    pb = np.broadcast_to(pdf_rtol, ok.shape)[both]
    fz = f[both] == 0
    assert np.all(np.where(fz, g_f[both] == 0, fr <= fb[:, None])), (name, float(np.nanmax(np.where(fz, 0, fr / fb[:, None]))))
    assert np.all(pr <= pb), (name, float(np.nanmax(pr / pb)))
    return {"n": int(ok.size), "sampled": int(both.sum()), "band": int(band.sum()), "none": int((~ok & sure).sum()),
            "ratio": float(max((d_err / e_wi[both]).max(), np.nanmax(np.where(fz, 0, fr / fb[:, None])), np.nanmax(pr / pb)))}


LOBE_CASES = {c[0]: c for c in _lobe_cases()}


@pytest.mark.parametrize("name", list(LOBE_CASES))
def test_oracle_lobe_sample_f_matches_float64(oracle, name):
    st = _lobe_compare(*LOBE_CASES[name])
    # the no-sample exits are exercised (wo.z = 0 at least); decisions within rounding come from the edge draws: the disk's
    # rim (u = 0, 1 - 2^-24, 1), for GGX u.x = 1 (theta_h = 90 deg) and tiny theta_h at grazing wo
    assert st["sampled"] > 0.3 * st["n"] and st["none"] > 0, st
    assert st["band"] < (0.4 if LOBE_CASES[name][4] is None else 0.12) * st["n"], st
    print(name, st)


def test_oracle_glass_lobes_sample_f_match_float64(oracle):
    """The two specular lobes one at a time (oracle.lobe_sample evaluates one lobe: the pick is checked in the slab renders)."""
    wo32 = _wo_grid()
    u32 = np.zeros((len(wo32), 2), F32)
    wo = wo32.astype(np.float64)
    R, T = np.asarray(F32(GLASS_R), np.float64), np.asarray(F32(GLASS_T), np.float64)
    for comp, kind, params in ((0, oracle.LOBE_SPEC_REFL, list(GLASS_R) + [GLASS_ETA]), (1, oracle.LOBE_SPEC_TRANS, list(GLASS_T) + [GLASS_ETA])):
        g_wi, g_f, g_pdf, g_type = oracle.lobe_sample(kind, params, wo32, u32)
        u = np.full((len(wo), 2), 0.75 if comp else 0.25)
        wi, f, pdf, ok, _, ct, near = glass_sample(wo, u, R, T, GLASS_ETA)
        sure = ~near & (wo[:, 2] != 0)
        assert np.array_equal((g_type != 0)[sure], ok[sure]) and np.all(g_type[g_type != 0] == (LOBE_SPEC_T if comp else LOBE_SPEC_R))
        both = sure & ok & (np.abs(wo[:, 2]) > COS_CUTOFF)   # at grazing 1 - Fr cancels
        assert np.all(np.linalg.norm(g_wi[both] - wi[both], axis=-1) <= 16.0 * EPS32 / np.abs(ct[both]))
        assert np.allclose(g_f[both], f[both], rtol=40.0 * EPS32 / np.abs(ct[both])[:, None] ** 2, atol=0) and np.all(g_pdf[both] == 1.0)
        if comp:
            assert (~ok & sure & (wo[:, 2] < 0)).sum() > 20   # total internal reflection leaving the glass: no sample


# ---- 2. paths sample by sample ------------------------------------------------------------------------------------------
QUAD_UV = np.array([(0, 0), (1, 0), (1, 1), (0, 1)], np.float32)   # dpdu = p1 - p0 on both triangles: the shading s axis
SPHERE_EDGE = 2e-3      # relative silhouette margin below which a ray that meets or passes a sphere is left out
GLASS_MAT = "glass"
# RTOL covers the conductor Fresnel and GGX chains (~60 roundings); a Matte fold term or beta factor takes ~15 (Oren-Nayar's
# a + b max_cos sin tan, the 1 / pi, Li / d^2, the cosine, the pdf), 1e-6, and 1e-5 leaves room for the light's own terms
MATTE_RTOL = 1e-5


class Quad:
    """A parallelogram mesh (two triangles, uv QUAD_UV) in float64 from its float32 world corners: normal cross(v0 - v2,
    v1 - v2) (triangle.rs:187-194), shading frame ss = normalize(v1 - v0), ts = cross(n, ss) (bsdfs/mod.rs:87-99)."""

    def __init__(self, corners, mat, emit=-1):
        self.v = np.asarray(corners, np.float64)
        self.mat, self.emit = mat, emit
        v0, v1, v2, v3 = self.v
        self.n = np.cross(v0 - v2, v1 - v2)
        self.n /= np.linalg.norm(self.n)
        self.ss = (v1 - v0) / np.linalg.norm(v1 - v0)
        self.ts = np.cross(self.n, self.ss)
        self.e1, self.e2 = v1 - v0, v3 - v0

    def crossing(self, o, d):
        """Ray parameter of the plane crossing (inf when parallel), plane coordinates and the signed distance to the outline."""
        with np.errstate(divide="ignore", invalid="ignore"):
            t = ((self.v[0] - o) @ self.n) / (d @ self.n)
            q = o + t[:, None] * d - self.v[0]
            a, b = (q @ self.e1) / (self.e1 @ self.e1), (q @ self.e2) / (self.e2 @ self.e2)
            edge = np.minimum(np.minimum(a, 1 - a) * np.linalg.norm(self.e1), np.minimum(b, 1 - b) * np.linalg.norm(self.e2))
        return np.where(np.isfinite(t), t, np.inf), np.stack([a, b], -1), np.nan_to_num(edge, nan=np.inf)

    def hit(self, o, d):
        t, uv, edge = self.crossing(o, d)
        ok = (t > 0) & (edge > 0)
        return np.where(ok, t, np.inf), (t > 0) & (np.abs(edge) < EDGE_W)

    def surface(self, o, d, t):
        _, uv, _ = self.crossing(o, d)
        each = lambda v: np.broadcast_to(v, o.shape)
        return {"p": o + t[:, None] * d, "n": each(self.n), "ns": each(self.n), "ss": each(self.ss), "ts": each(self.ts),
                "wo": -d, "uv": uv, "frame_err": np.zeros(len(o)), "r": np.inf}

    def shadow(self, o_s, seg):
        """The segment o_s + t seg, t in (0, 0.9999): whether it crosses the quad, and whether it passes within EDGE_W."""
        t, _, edge = self.crossing(o_s, seg)
        inr = (t > 0) & (t < 0.9999)
        return inr & (edge > 0), inr & (np.abs(edge) < EDGE_W)


class Ball:
    """A SphereShape of test_direct_lighting as a path surface: hits from outside (the near root), its per-point frame, the
    wo Bsdf::f receives (normalize(o2w (-d))), and its shadow test."""

    def __init__(self, shape, mat):
        self.shape, self.mat, self.emit = shape, mat, -1
        self.cond = np.linalg.cond(shape.W[:3, :3])

    def hit(self, o, d):
        h = self.shape.hit(o, d)
        oo, dd, a, _, _, _ = self.shape._quadric(o, d)
        ahead = (oo * dd).sum(-1) < 0
        t = ((h["p"] - o) * d).sum(-1) / (d * d).sum(-1)
        return np.where(h["inside"], t, np.inf), ahead & (np.abs(h["edge"]) < SPHERE_EDGE)

    def surface(self, o, d, t):
        h = self.shape.hit(o, d)
        h["uv"] = np.zeros((len(o), 2))
        h["r"] = self.shape.r / self.cond
        return h

    def shadow(self, o_s, seg, p=None, n=None):
        return self.shape.self_shadow(p, n, o_s + seg)


class Scene:
    """Surfaces, lights (test_direct_lighting.Light), background, and the scene description the renderers take."""

    def __init__(self, desc, cam, surfaces, film, sampler, depth, clamp=None):
        self.desc, self.cam, self.surfaces, self.film, self.sampler = desc, cam, surfaces, film, sampler
        self.lights = [Light(l) for l in desc.lights]
        self.bg = np.asarray(F32(desc.background), np.float64)
        self.integ = D.IntegratorType.path(depth, clamp)
        self.depth, self.clamp = depth, clamp


def _draws(sc):
    """Every (pixel, sample)'s draws in the Path pattern: [2] camera, then per vertex one [2] per light in light order and
    [2] for the BSDF, then [1] for roulette after vertices with bounces > 3 (path.rs:102-169)."""
    from oracle import oracle as O
    nl = len(sc.lights)
    pattern = [2]
    for b in range(sc.depth):
        pattern += [2] * nl + [2] + ([1] if b > 3 else [])
    w, h = sc.film.res
    spp = sc.sampler.samples_per_pixel()
    out = np.array([O.sampler_draws(sc.sampler, x, y, i, pattern) for y in range(h) for x in range(w) for i in range(spp)], F32)
    offs, k = [], 2
    for b in range(sc.depth):
        offs.append(k)
        k += 2 * nl + 2 + (1 if b > 3 else 0)
    return out, offs


def _cos_slope(mat, alpha, wo, wi):
    """A bound on |d ln f / d angle| for the lobe at (wo, wi), for the shift of either direction: GGX's D (d_slope at the
    half vector, which turns by half the angle) plus G, F and the cosines; Oren-Nayar's max_cos, sin and tan terms; 0 for
    Lambert."""
    c = np.maximum(np.minimum(np.abs(wo[:, 2]), np.abs(wi[:, 2])), COS_CUTOFF)
    if mat.kind == D.MAT_MATTE:
        return np.where(mat.scalar(np.zeros(len(wo), int)) == 0, 0.0, 8.0 / c) if mat.image is None else 8.0 / c
    wh = wo + wi
    wh /= np.maximum(np.linalg.norm(wh, axis=-1, keepdims=True), 1e-300)
    return 0.5 * d_slope(alpha, wh) + 8.0 / c


def _local(h, w):
    return np.stack([(w * h["ss"]).sum(-1), (w * h["ts"]).sum(-1), (w * h["ns"]).sum(-1)], -1)


def _world(h, w):
    return h["ss"] * w[:, 0:1] + h["ts"] * w[:, 1:2] + h["ns"] * w[:, 2:3]


def _occluded(sc, p, n, target, skip_emit):
    """spawn_ray_to (interaction.rs:41-59) against every surface; a hit on the target area light's own quad does not occlude
    (bvh.rs:269-280). Returns occluded and whether any crossing is within rounding of a decision."""
    side = np.where((((target - p) * n).sum(-1) > 0), 1.0, -1.0)
    o_s = p + side[:, None] * SPAWN_OFFSET * n
    seg = target - o_s
    occ, near = np.zeros(len(p), bool), np.zeros(len(p), bool)
    for s in sc.surfaces:
        if isinstance(s, Ball):
            a, b = s.shadow(o_s, seg, p, n)
        else:
            if s.emit >= 0 and s.emit == skip_emit:
                continue
            a, b = s.shadow(o_s, seg)
        occ |= a
        near |= b
    return occ, near


def _walk(sc, o, d, draws, offs, variant=None):
    """float64 Path radiance of every sample (path.rs:49-178 in its order: hit, per-point frame, light fold, emitted term
    after a specular bounce or at the camera, clamp at bounces > 0, L += beta radiance, sample_f with wo = -ray.d, beta
    update, spawn 1e-3 along +-n, roulette), with a per-sample absolute error bound per channel and the samples left out.

    The bound sums |term| times the term's relative error over the path's terms. A term's relative error is beta's
    (accumulated per vertex: the lobe's f and pdf errors, the cosine, roulette's 1 / (1 - q)) plus the fold's: RTOL,
    microfacet_f's d_err and rtol_extra, and the float32 path's drift: each sampled direction errs by the lobe's e_wi
    (rad); that moves the next hit by t e_wi / |cos_in|, which turns the light directions by dp / d and the frame on a
    sphere by dp / r, and changes the lobes by their angular slope (_cos_slope) and I / d^2 by 2 dp / d.

    `variant` restates a planted misreading in float64 (for the claims that each case can tell it apart): "beta-once",
    "no-roulette-division", "wo-si" (sample_f given si.wo)."""
    N = len(o)
    L, bound = np.zeros((N, 3)), np.zeros((N, 3))
    beta, tol_b = np.ones((N, 3)), np.zeros(N)
    d_dir, d_pos = np.full(N, 4.0 * EPS32), np.zeros(N)   # the camera ray's direction: a normalised float32 vector
    spec = np.zeros(N, bool)
    alive = np.ones(N, bool)
    excl = {k: np.zeros(N, bool) for k in ("edge", "cos", "roulette", "critical", "band", "self_shadow")}
    info = {k: np.zeros(N, int) for k in ("vertices", "bg", "lit2", "spec_emit", "glass_t", "glass_r", "tir", "rr_kill",
                                           "rr_cont", "clamped", "clamp0_over", "wo_matters", "far_mirror")}
    info["vertex_mat"] = []
    o, d = o.copy(), d.copy()
    for b in range(sc.depth):
        idx = np.flatnonzero(alive)
        if len(idx) == 0:
            break
        oo, dd = o[idx], d[idx]
        ts, near = zip(*[s.hit(oo, dd) for s in sc.surfaces])
        ts = np.stack(ts, 1)
        excl["edge"][idx[np.any(near, axis=0)]] = True
        which = np.where(np.isfinite(ts).any(1), ts.argmin(1), -1)
        miss = which < 0
        m = idx[miss]
        L[m] += beta[m] * sc.bg
        bound[m] += beta[m] * sc.bg * tol_b[m, None]
        info["bg"][m] += b > 0
        alive[m] = False
        for si, surf in enumerate(sc.surfaces):
            sel = which == si
            if not sel.any():
                continue
            j = idx[sel]
            oj, dj, tj = oo[sel], dd[sel], ts[sel, si]
            h = surf.surface(oj, dj, tj)
            p, n = h["p"], h["n"]
            info["vertices"][j] += 1
            dn = dj / np.linalg.norm(dj, axis=-1, keepdims=True)
            c_in = np.abs((dn * n).sum(-1))
            excl["cos"][j[c_in < COS_CUTOFF]] = True
            dp = (d_pos[j] + tj * np.linalg.norm(dj, axis=-1) * d_dir[j]) / np.maximum(c_in, COS_CUTOFF) + 8.0 * EPS32 * np.abs(p).max(-1)
            turn = h["frame_err"] + dp / h["r"]        # the per-point frame's turn (spheres)
            a_wo = d_dir[j] + turn                      # wo's angular error in the frame
            mat = surf.mat
            texel, tex_safe = (np.zeros(len(j), int), np.ones(len(j), bool)) if not isinstance(mat, Mat) else _texel(mat, h["uv"])
            excl["edge"][j[~tex_safe]] = True
            alpha = mat.alpha(mat.scalar(texel)) if isinstance(mat, Mat) and mat.kind != D.MAT_MATTE else None
            rad, rad_b = np.zeros((len(j), 3)), np.zeros((len(j), 3))
            wo_f = _local(h, h["wo"])
            # the light fold (path.rs:102-119)
            for k, lt in enumerate(sc.lights):
                u = draws[j, offs[b] + 2 * k: offs[b] + 2 * k + 2].astype(np.float64)
                wi_w, li, pdf, vis, target = lt.sample(p, n, u)
                wi_w, target = np.asarray(wi_w), np.asarray(target, np.float64)
                li = np.broadcast_to(li, (len(j), 3))
                reaches = li.max(-1) > 0
                if not isinstance(mat, Mat):
                    continue       # glass and the emitters' black matte: f = 0, no shadow ray counts
                if lt.desc.kind == D.LIGHT_RECT:   # the one-sided test and pdf's 1 / |cos_l| at grazing: left out
                    nl = lt.m_inv[:3, :3].T @ np.array([0.0, -1.0, 0.0])
                    cos_l = -(wi_w @ nl) / np.linalg.norm(nl)
                    excl["cos"][j[np.abs(cos_l) < COS_CUTOFF]] = True
                occ, near_s = _occluded(sc, p, n, target, k if lt.desc.kind == D.LIGHT_RECT else -2)
                excl["edge"][j[reaches & near_s]] = True
                cos_g = (wi_w * n).sum(-1)
                refl = cos_g * (h["wo"] * n).sum(-1) > 0.0
                wi_l = _local(h, wi_w)
                f, f_err = mat.f(wo_f, wi_l, texel)
                f = np.where(refl[:, None], f, 0.0)
                cos_s = (wi_w * h["ns"]).sum(-1)
                lit = refl & reaches & vis & ~occ
                term = np.where(lit[:, None], f * li * np.clip(cos_s, 0.0, 1.0)[:, None] / pdf[:, None], 0.0)
                dist = np.linalg.norm(target - p, axis=-1)
                a_li = dp / dist + turn
                slope = _cos_slope(mat, alpha, wo_f, wi_l) if alpha is not None or mat.kind == D.MAT_MATTE else 0.0
                tol = (RTOL if alpha is not None else MATTE_RTOL) + f_err + slope * (a_wo + a_li) + a_li / np.maximum(np.abs(cos_s), COS_CUTOFF) + 2.0 * dp / dist
                rad += term
                rad_b += term * tol[:, None]
                excl["cos"][j[lit & (np.abs(cos_s) < COS_CUTOFF)]] = True
                excl["cos"][j[reaches & vis & (np.abs(cos_g) < COS_CUTOFF)]] = True
                if b > 0:
                    info["lit2"][j] |= (lit & (term.max(-1) > 0)).astype(int) << k
            # emitted radiance at the camera or after a specular bounce, beta applied here and again below (path.rs:121-123)
            if surf.emit >= 0:
                le = np.where(((-dj * n).sum(-1) > 0)[:, None], np.asarray(F32(sc.desc.lights[surf.emit].intensity), np.float64), 0.0)
                em = (b == 0) | spec[j]
                e_term = np.where(em[:, None], (beta[j] if variant != "beta-once" else 1.0) * le, 0.0)
                rad += e_term
                rad_b += e_term * tol_b[j, None]
                info["spec_emit"][j] += (spec[j] & (b > 0) & (le.max(-1) > 0)).astype(int)
            if b == 0 and sc.clamp is not None:
                info["clamp0_over"][j] |= rad.max(-1) > sc.clamp
            if b > 0 and sc.clamp is not None:
                c = np.float64(F32(sc.clamp))
                info["clamped"][j] |= rad.max(-1) > c
                rad = np.minimum(rad, c)                 # min is 1-Lipschitz: the bound carries over
                rad_b = np.minimum(rad_b, np.abs(rad) + rad_b)
            L[j] += beta[j] * rad
            bound[j] += beta[j] * rad_b + beta[j] * rad * tol_b[j, None]
            # sample_f with wo = -ray.d (path.rs:127-131), not si.wo
            wo_s = _local(h, h["wo"] if variant == "wo-si" else -dj)
            u = draws[j, offs[b] + 2 * len(sc.lights): offs[b] + 2 * len(sc.lights) + 2].astype(np.float64)
            if mat == GLASS_MAT:
                wi_l, f, pdf, ok, comp, ct, near_c = glass_sample(wo_s, u, np.asarray(F32(GLASS_R), np.float64), np.asarray(F32(GLASS_T), np.float64), GLASS_ETA)
                excl["critical"][j[near_c]] = True
                info["glass_t"][j] += (ok & (comp == 1)).astype(int)
                info["glass_r"][j] += (comp == 0).astype(int)
                info["tir"][j] += (~ok).astype(int)
                e_wi = 8.0 * EPS32 + np.where(comp == 1, a_wo * GLASS_ETA / np.maximum(np.abs(ct), COS_T_CUTOFF), a_wo)
                r_beta = 48.0 * EPS32 + 4.0 * a_wo / np.maximum(np.abs(ct), COS_T_CUTOFF)
                new_spec = np.ones(len(j), bool)
            elif isinstance(mat, Mat) and mat.kind == D.MAT_MATTE:
                wi_l, pdf, ok, e0, band = diffuse_sample(wo_s, u)
                excl["band"][j[band]] = True
                f, _ = mat.f(wo_s, wi_l, texel)      # Lobe::sample_f evaluates f at its own wo
                e_wi = e0 + turn
                slope = _cos_slope(mat, None, wo_f, wi_l)
                with np.errstate(divide="ignore"):
                    r_beta = MATTE_RTOL + slope * (a_wo + e_wi) + 8.0 * e0 / np.abs(wi_l[:, 2])
                new_spec = np.zeros(len(j), bool)
            elif isinstance(mat, Mat):
                wi_l, wh, pdf, ok, e_wh, e0, band = ggx_sample(alpha, wo_s, u)
                excl["band"][j[band & np.isfinite(e_wh)]] = True
                with np.errstate(divide="ignore", invalid="ignore"):
                    f, d_err = microfacet_f(alpha, _fresnel(mat), wo_s, wi_l)
                    sd = d_slope(alpha, wh)
                    wsum = np.linalg.norm(wo_s + wi_l, axis=-1)
                    cmin = np.maximum(np.minimum(np.abs(wo_s[:, 2]), np.abs(wi_l[:, 2])), COS_CUTOFF)
                    e_wi = e0 + 2.0 * a_wo
                    r_beta = (2.0 * RTOL + 2.0 * d_err + mat.rtol_extra(texel) + sd * (2.0 * e_wh + 24.0 * EPS32 / wsum + a_wo)
                              + 16.0 * (e_wi + a_wo) / cmin + 8.0 * e_wh / np.maximum((wo_s * wh).sum(-1), 1e-12))
                mirror = np.stack([-wo_s[:, 0], -wo_s[:, 1], wo_s[:, 2]], -1)
                info["far_mirror"][j] |= ok & (np.arccos(np.clip((mirror * wi_l).sum(-1) / np.linalg.norm(wo_s, axis=-1), -1, 1)) > 0.3)
                new_spec = np.zeros(len(j), bool)
            else:                                   # the emitters' black matte: no lobe, no sample
                ok = np.zeros(len(j), bool)
                wi_l, f, pdf, e_wi, r_beta, new_spec = np.zeros((len(j), 3)), np.zeros((len(j), 3)), np.zeros(len(j)), 0.0, 0.0, np.zeros(len(j), bool)
            wi_w = _world(h, wi_l)
            if variant is None and isinstance(surf, Ball) and isinstance(mat, Mat):
                # the claim that sample_f's wo matters: si.wo instead of -ray.d moves wi or beta by more than 10 tolerances
                alt_wi, alt_fac = _walk_alt(mat, alpha, h, texel, u)
                with np.errstate(divide="ignore", invalid="ignore"):
                    fac0 = f * np.abs(wi_l[:, 2:3]) / pdf[:, None]
                    moved = (np.linalg.norm(alt_wi - wi_l, axis=-1) > 10.0 * e_wi) | \
                            (np.abs(alt_fac - fac0) > 10.0 * r_beta[:, None] * np.abs(fac0)).any(-1)
                info["wo_matters"][j] |= ok & moved
            f = np.where(ok[:, None], f, 0.0)
            ok &= (f.max(-1) > 0) & (pdf != 0)
            cos_o = np.abs((wi_w * h["ns"]).sum(-1))
            excl["cos"][j[ok & ~new_spec & (cos_o < COS_CUTOFF)]] = True
            alive[j[~ok]] = False
            with np.errstate(divide="ignore", invalid="ignore"):
                fac = np.where(ok[:, None], f * cos_o[:, None] / np.where(ok, pdf, 1.0)[:, None], 0.0)
            beta[j] *= fac
            tol_b[j] += np.where(ok, r_beta + e_wi / np.maximum(cos_o, COS_CUTOFF) + 4.0 * EPS32, 0.0)
            spec[j] = new_spec
            side = np.where(((wi_w * n).sum(-1) > 0), 1.0, -1.0)
            o[j] = p + side[:, None] * SPAWN_OFFSET * n
            d[j] = wi_w
            d_dir[j] = e_wi
            d_pos[j] = dp
            info["vertex_mat"].append((b, j[ok], surf))
        if b > 3:   # Russian roulette (path.rs:163-169); q >= 1 ends the path whatever the draw (yko_render.h:189-195)
            r_idx = np.flatnonzero(alive)
            r_idx = r_idx[np.isin(r_idx, idx)]
            q = np.maximum(1.0 - beta[r_idx, 1], 0.05)
            dq = beta[r_idx, 1] * tol_b[r_idx] + 2.0 * EPS32
            draw = draws[r_idx, offs[b] + 2 * len(sc.lights) + 2].astype(np.float64)
            excl["roulette"][r_idx[np.abs(draw - q) <= 2.0 * dq]] = True
            kill = (draw < q) | (q >= 1.0)
            info["rr_kill"][r_idx[kill]] += 1
            info["rr_cont"][r_idx[~kill]] += 1
            alive[r_idx[kill]] = False
            cont = r_idx[~kill]
            qc = q[~kill]
            if variant != "no-roulette-division":
                beta[cont] /= (1.0 - qc)[:, None]
            tol_b[cont] += dq[~kill] / (1.0 - qc) + 2.0 * EPS32
    keep = ~np.any([v for v in excl.values()], axis=0)
    return L, bound, keep, excl, info


def _walk_alt(mat, alpha, h, texel, u):
    """The local wi and f |cos| / pdf sample_f would give with si.wo (a sphere's normalize(o2w (-d))) in place of -ray.d."""
    wo = _local(h, h["wo"])
    if mat.kind == D.MAT_MATTE:
        wi, pdf = diffuse_sample(wo, u)[:2]
        f = mat.f(wo, wi, texel)[0]
    else:
        wi, _, pdf = ggx_sample(alpha, wo, u)[:3]
        with np.errstate(divide="ignore", invalid="ignore"):
            f = microfacet_f(alpha, _fresnel(mat), wo, wi)[0]
    with np.errstate(divide="ignore", invalid="ignore"):
        return wi, f * np.abs(wi[:, 2:3]) / pdf[:, None]


def _camera(sc, draws):
    from oracle import oracle as O
    w, h = sc.film.res
    spp = sc.sampler.samples_per_pixel()
    ys, xs = np.mgrid[0:h, 0:w]
    px = np.repeat(np.stack([xs.ravel(), ys.ravel()], -1).astype(F32), spp, axis=0)
    o, d = O.camera_rays(sc.cam, sc.film, px + draws[:, :2])
    return o.astype(np.float64), d.astype(np.float64)


@functools.lru_cache(maxsize=None)
def reference(case):
    sc = CASES[case]()
    draws, offs = _draws(sc)
    o, d = _camera(sc, draws)
    return sc, draws, offs, o, d, _walk(sc, o, d, draws, offs)


def _films(render, sc):
    """Per-sample films (N, 3), ordered (y, x, sample): an accumulating film onto zeros, one sample index at a time."""
    from oracle import oracle as O
    film = D.FilmSettings(sc.film.res, sc.film.tile_dim, accumulate=True)
    spp = sc.sampler.samples_per_pixel()
    w, h = film.res
    out = np.zeros((h, w, spp, 3), F32)
    base = O.film_tiles(film)
    for k in range(spp):
        tiles = base.copy()
        tiles["sample"] = k
        img = np.zeros((h, w, 3), F32)
        render(film, tiles, img)
        out[:, :, k] = img
    return out.reshape(-1, 3)


def _check(case, got):
    sc, _, _, _, _, (want, bound, keep, excl, info) = reference(case)
    got = got.astype(np.float64)
    err = np.abs(got - want)
    lim = bound + 8.0 * EPS32 * sc.depth * np.abs(want) + 1e-30
    bad = keep[:, None] & (err > lim)
    ratio = np.where(keep[:, None] & (want > 0), err / lim, 0.0)
    assert not bad.any(), (case, int(bad.any(-1).sum()), float(ratio.max()), np.flatnonzero(bad.any(-1))[:5].tolist())
    assert np.all(got[keep & (want.max(-1) == 0)] == 0.0), case
    assert keep.mean() >= 0.9, (case, {k: int(v.sum()) for k, v in excl.items()})
    return float(ratio.max())


# ---- the cases ------------------------------------------------------------------------------------------------------------
WALL_KD, BG = (0.6, 0.7, 0.5), (0.15, 0.2, 0.25)
PLANES_CAM = D.CameraParameters((0.3, -0.2, 3.0), (0.1, 0.0, 0.0), fov_axis=D.FOV_X, fov_deg=50.0)
SMALL_FILM = D.FilmSettings((24, 18), 8)
SAMPLERS = {"strat": D.SamplerType.stratified(2, 2), "uniform": D.SamplerType.uniform(4)}
_rot = lambda deg, axis: xf.rotation(float(F32(np.deg2rad(deg))), axis)


def _add_quad(s, corners, mat_index):
    s.meshes.append(D.Mesh(xf.identity(), np.array(corners, np.float32), np.array([0, 1, 2, 0, 2, 3], np.uint32), mat_index, uvs=QUAD_UV))
    return np.array(corners, np.float32)


def _matte(s, kd):
    zero = s.add_texture(D.Texture.constant(0.0))
    return s.add_material(D.Material(D.MAT_MATTE, (s.add_texture(D.Texture.constant(*kd)), zero)))


def _add_emitter(s, to_world, intensity, size):
    """A one-sided rect light (its -y normal) with its emissive quad, wound so that the quad's normal is the light's."""
    k = len(s.lights)
    s.lights.append(D.Light(D.LIGHT_RECT, to_world, intensity, size=size))
    hx, hz = size[0] / 2, size[1] / 2
    loc = np.array([(-hx, 0, -hz), (hx, 0, -hz), (hx, 0, hz), (-hx, 0, hz)], np.float32)
    world = np.array([xf.point(to_world, q) for q in loc], np.float32)
    s.meshes.append(D.Mesh(xf.identity(), world, np.array([0, 1, 2, 0, 2, 3], np.uint32), _matte(s, (0.0, 0.0, 0.0)), uvs=QUAD_UV, area_light=k))
    return world, k


def two_planes(mat_name, depth, smp, clamp=None):
    """The floor [-1, 1]^2 (z = 0) in the material under test, facing a large Matte wall (x = -1.2, normal +x) under a point
    light and a one-sided rect light aimed down, with a non-zero background."""
    mat = MATERIALS[mat_name]
    s = D.SceneDesc(background=BG)
    floor = _add_quad(s, [(-1, -1, 0), (1, -1, 0), (1, 1, 0), (-1, 1, 0)], mat.add_to(s))
    wall = _add_quad(s, [(-1.2, -2, 0), (-1.2, 2, 0), (-1.2, 2, 3), (-1.2, -2, 3)], _matte(s, WALL_KD))
    s.lights.append(D.Light(D.LIGHT_POINT, xf.translation((0.2, 0.3, 1.4)), (2.0, 1.8, 1.5)))
    s.lights.append(D.Light(D.LIGHT_RECT, xf.mul(xf.translation((-0.4, -0.2, 1.6)), _rot(90.0, (1.0, 0.0, 0.0))), (3.0, 3.0, 2.5), size=(0.5, 0.4)))
    surfaces = [Quad(floor, mat), Quad(wall, Mat("wall", D.MAT_MATTE, {"kd": WALL_KD, "sigma": 0.0}))]
    return Scene(s, PLANES_CAM, surfaces, SMALL_FILM, SAMPLERS[smp], depth, clamp)


SLAB_LIGHT_XF = xf.mul(xf.translation((-0.1, 0.3, 3.0)), _rot(90.0, (1.0, 0.0, 0.0)))


def glass_slab(wedge, depth, smp):
    """slab_scene (a Lambertian floor under a glass slab, a point light to the side) with an area light above: the camera
    sees it reflected in the slab's top, and the floor sees it through the slab."""
    s, corners = slab_scene(wedge)
    for m in s.meshes:
        m.uvs = QUAD_UV
    em, k = _add_emitter(s, SLAB_LIGHT_XF, (5.0, 4.5, 4.0), (1.2, 1.2))
    floor = Mat("floor", D.MAT_MATTE, {"kd": (0.6, 0.5, 0.4), "sigma": 0.0})
    surfaces = [Quad(corners[0], floor), Quad(corners[1], GLASS_MAT), Quad(corners[2], GLASS_MAT), Quad(em, None, emit=k)]
    return Scene(s, SLAB_CAM, surfaces, D.FilmSettings((24, 18), 8), SAMPLERS[smp], depth)


FLOOR_KD, CEIL_KD = (0.92, 0.75, 0.85), (0.85, 0.9, 0.8)
CORRIDOR_CAM = D.CameraParameters((0.0, -5.0, 0.5), (0.0, 0.0, 0.45), fov_axis=D.FOV_X, fov_deg=60.0)


def corridor(depth, smp, clamp=None):
    """Two facing high-albedo Matte planes, 1 apart and open at the sides, with point lights between them: paths pass
    bounces > 3 and meet Russian roulette; kd.g differs from kd.r."""
    s = D.SceneDesc(background=BG)
    fl = _add_quad(s, [(-1, -6, 0), (1, -6, 0), (1, 6, 0), (-1, 6, 0)], _matte(s, FLOOR_KD))
    ce = _add_quad(s, [(-1, -6, 1), (-1, 6, 1), (1, 6, 1), (1, -6, 1)], _matte(s, CEIL_KD))
    s.lights.append(D.Light(D.LIGHT_POINT, xf.translation((0.0, -2.0, 0.5)), (0.8, 0.8, 0.7)))
    s.lights.append(D.Light(D.LIGHT_POINT, xf.translation((0.3, 1.5, 0.6)), (0.6, 0.7, 0.8)))
    surfaces = [Quad(fl, Mat("floor", D.MAT_MATTE, {"kd": FLOOR_KD, "sigma": 0.0})), Quad(ce, Mat("ceiling", D.MAT_MATTE, {"kd": CEIL_KD, "sigma": 0.0}))]
    return Scene(s, CORRIDOR_CAM, surfaces, SMALL_FILM, SAMPLERS[smp], depth, clamp)


def spheres(sphere, mat_name, smp):
    """A rotated or non-uniformly scaled sphere above a lit Matte floor (z = -1.3), depth 2."""
    shape, mat = SPHERES[sphere], MATERIALS[mat_name]
    s = D.SceneDesc(background=BG)
    s.spheres.append(D.Sphere(shape.to_world, shape.r, mat.add_to(s)))
    fl = _add_quad(s, [(-3, -3, -1.3), (3, -3, -1.3), (3, 3, -1.3), (-3, 3, -1.3)], _matte(s, WALL_KD))
    s.lights.append(D.Light(D.LIGHT_POINT, xf.translation((0.4, 0.3, 2.8)), (6.0, 5.0, 4.0)))
    s.lights.append(D.Light(D.LIGHT_POINT, xf.translation((2.5, 0.5, 0.2)), (3.0, 3.0, 3.0)))
    surfaces = [Ball(shape, mat), Quad(fl, Mat("floor", D.MAT_MATTE, {"kd": WALL_KD, "sigma": 0.0}))]
    return Scene(s, PLANES_CAM, surfaces, SMALL_FILM, SAMPLERS[smp], 2)


def _case_table():
    t = {}
    for m in MATERIALS:
        t[f"planes-{m}-d2-strat"] = functools.partial(two_planes, m, 2, "strat")
        t[f"planes-{m}-d3-uniform"] = functools.partial(two_planes, m, 3, "uniform")
    for wedge in (False, True):
        for depth in (2, 3, 5):
            t[f"{'wedge' if wedge else 'slab'}-d{depth}-strat"] = functools.partial(glass_slab, wedge, depth, "strat")
        t[f"{'wedge' if wedge else 'slab'}-d5-uniform"] = functools.partial(glass_slab, wedge, 5, "uniform")
    for smp in SAMPLERS:
        t[f"corridor-d8-{smp}"] = functools.partial(corridor, 8, smp)
    t["clamp-planes-matte"] = functools.partial(two_planes, "matte", 3, "strat", 0.05)
    t["clamp-planes-copper-a0.3"] = functools.partial(two_planes, "copper-a0.3", 3, "uniform", 0.05)
    t["clamp-corridor"] = functools.partial(corridor, 8, "strat", 0.04)
    for sp in ("sphere-rotated", "sphere-scaled"):
        for m in ("matte", "oren-nayar-20", "copper-a0.3"):
            t[f"{sp}-{m}"] = functools.partial(spheres, sp, m, "strat")
    return t


CASES = _case_table()


def _claims(case):
    sc, draws, offs, o, d, (want, bound, keep, excl, info) = reference(case)
    N = len(want)
    assert np.isfinite(want).all()
    if case.startswith("planes") or case.startswith("clamp-planes"):
        second = keep & (info["vertices"] >= 2)
        assert second.sum() > 0.05 * N, int(second.sum())                      # a second vertex on the wall
        assert (keep & (info["bg"] > 0)).sum() > 0.1 * N                      # escaping bounces meet the background
        assert ((info["lit2"] & 1) > 0).sum() > 0.05 * N and ((info["lit2"] & 2) > 0).sum() > 0.05 * N   # both lights
        if "copper-a0.05" in case:
            assert info["far_mirror"].sum() > 0                                # GGX samples far from the mirror direction
    if case.startswith(("slab", "wedge")):
        assert (info["glass_r"] > 0).sum() > 0.05 * N and (info["glass_t"] > 0).sum() > 0.05 * N   # both lobe picks
        if sc.depth >= 2:
            assert (keep & (info["spec_emit"] > 0)).sum() > 0.02 * N           # emission after a specular bounce
        if sc.depth >= 2:   # beta once instead of twice on that emission would move those samples by far more than the bound
            alt = _walk(sc, o, d, draws, offs, variant="beta-once")[0]
            assert (keep & (np.abs(alt - want) > 10.0 * bound + 1e-6).any(-1)).sum() > 0.02 * N
        if case.startswith("wedge") and sc.depth >= 5:
            assert (info["tir"] > 0).sum() > 0                                 # total internal reflection ends paths
    if case.startswith("corridor") or case == "clamp-corridor":
        assert (info["rr_kill"] > 0).sum() > 0.02 * N and (info["rr_cont"] > 0).sum() > 0.02 * N
        alt = _walk(sc, o, d, draws, offs, variant="no-roulette-division")[0]   # 1 / (1 - q) shows in the film
        assert (keep & (np.abs(alt - want) > 10.0 * bound + 1e-6).any(-1)).sum() > 0.02 * N
    if case.startswith("clamp"):
        assert (keep & (info["clamped"] > 0)).sum() > 0.05 * N                # the clamp cuts later vertices ...
        assert (keep & (info["clamp0_over"] > 0)).sum() > 0.05 * N            # ... and would cut the first one
    if case.startswith("sphere"):
        sph = np.zeros(N, bool)
        for b, j, surf in info["vertex_mat"]:
            if isinstance(surf, Ball):
                sph[j] = True
        assert sph.sum() > 0.2 * N
        if not case.endswith("-matte"):   # Lambert's sample ignores wo but for its side, and its f is constant
            assert (keep & sph & (info["wo_matters"] > 0)).sum() > 0.5 * (keep & sph).sum()
    return {k: int(v.sum()) for k, v in excl.items()}


@pytest.mark.parametrize("case", list(CASES))
def test_oracle_path_samples_match_float64(oracle, case):
    sc = reference(case)[0]
    osc = oracle.OracleScene(sc.desc)
    got = _films(lambda film, tiles, img: osc.render(sc.cam, film, sc.sampler, sc.integ, tiles=tiles, film_out=img), sc)
    ratio = _check(case, got)
    excluded = _claims(case)
    print(case, "max err / bound", f"{ratio:.3g}", excluded)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_gpu_path_samples_match_float64_and_the_oracle(gpu_ctx, oracle, case):
    sc = reference(case)[0]
    osc = oracle.OracleScene(sc.desc)
    want = _films(lambda film, tiles, img: osc.render(sc.cam, film, sc.sampler, sc.integ, tiles=tiles, film_out=img), sc)
    dev = api.Scene(gpu_ctx, sc.desc)
    try:
        rn = api.Renderer(gpu_ctx)
        got = _films(lambda film, tiles, img: rn.render(dev, sc.cam, film, sc.sampler, sc.integ, tiles=tiles, film_out=img), sc)
    finally:
        dev.close()
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), case
    _check(case, got)


# ---- 3. bounce directions through debug_ray ------------------------------------------------------------------------------
DEBUG_CASES = ("planes-copper-a0.3-d2-strat", "planes-glossy-r0.2-d3-uniform", "planes-oren-nayar-60-d3-uniform", "slab-d5-strat",
               "wedge-d5-strat", "sphere-rotated-oren-nayar-20", "sphere-scaled-copper-a0.3")
DEBUG_SAMPLER = D.SamplerType.uniform(1, seed=0x2545F4914F6CDD1D)
DEBUG_PIXELS = [(x, y) for y in range(1, 18, 2) for x in range(1, 24, 2)]


def _debug_draws(sc, n):
    """The fresh clone's draws (window.rs:884-888): a uniform sampler never started on a pixel sample, Pcg32::new(seed, 0)."""
    from oracle import oracle as O
    return (O.pcg32_sequence(DEBUG_SAMPLER.seed, 0, 0, n) >> 8).astype(F32) * F32(2.0 ** -24)


def _sampled_directions(sc, o, d, u):
    """float64 world wi that sample_f draws at the first hit of the float32 rays (o, d) with draws u, its error bound (rad),
    and whether the sample is usable (a hit away from outlines and grazing angles, a sample, no decision within rounding)."""
    ts, near = zip(*[s.hit(o, d) for s in sc.surfaces])
    ts = np.stack(ts, 1)
    which = np.where(np.isfinite(ts).any(1), ts.argmin(1), -1)
    wi_w, err, use = np.zeros_like(o), np.zeros(len(o)), (which >= 0) & ~np.any(near, axis=0)
    for si, surf in enumerate(sc.surfaces):
        sel = which == si
        if not sel.any():
            continue
        h = surf.surface(o[sel], d[sel], ts[sel, si])
        wo = _local(h, -d[sel])
        c_in = np.abs((d[sel] * h["n"]).sum(-1)) / np.linalg.norm(d[sel], axis=-1)
        mat, good = surf.mat, c_in > COS_CUTOFF
        if mat == GLASS_MAT:
            wi, _, _, ok, comp, ct, near_c = glass_sample(wo, u[sel], np.asarray(GLASS_R), np.asarray(GLASS_T), GLASS_ETA)
            e = 16.0 * EPS32 / np.maximum(np.abs(ct), COS_T_CUTOFF)
            good &= ok & ~near_c
        elif isinstance(mat, Mat) and mat.kind == D.MAT_MATTE:
            wi, _, ok, e, band = diffuse_sample(wo, u[sel])
            good &= ok & ~band & (np.abs(wi[:, 2]) > COS_CUTOFF)
        elif isinstance(mat, Mat):
            alpha = mat.alpha(mat.scalar(_texel(mat, h["uv"])[0]))
            wi, _, _, ok, _, e, band = ggx_sample(alpha, wo, u[sel])
            good &= ok & ~band & (np.abs(wi[:, 2]) > COS_CUTOFF)
        else:
            continue
        wi_w[sel] = _world(h, wi)
        err[sel] = e + 2.0 * h["frame_err"] + 8.0 * EPS32
        use[sel] &= good
    return wi_w, err, use


def _debug_pairs(sc, rays_of):
    """(incoming o, d, draw u, logged outgoing d) of every vertex that continues, over DEBUG_PIXELS."""
    nl = len(sc.lights)
    draws = _debug_draws(sc, 2 + sc.depth * (2 * nl + 3))
    offs = np.cumsum([2] + [2 * nl + 2 + (1 if b > 3 else 0) for b in range(sc.depth)])
    out = []
    for px in DEBUG_PIXELS:
        rays = rays_of(px)
        bounce = rays[np.isin(rays["ray_type"], (0, 1, 2))]
        for b in range(len(bounce) - 1):
            u = draws[offs[b] + 2 * nl: offs[b] + 2 * nl + 2]
            out.append((bounce["o"][b], bounce["d"][b], u, bounce["d"][b + 1], bounce["ray_type"][b + 1]))
    o, d, u, wi, kind = (np.array([p[k] for p in out]) for k in range(5))
    return o.astype(np.float64), d.astype(np.float64), u.astype(np.float64), wi.astype(np.float64), kind


def _check_debug(case, rays_of):
    sc = CASES[case]()
    o, d, u, got, kind = _debug_pairs(sc, rays_of)
    want, err, use = _sampled_directions(sc, o, d, u)
    dev = np.linalg.norm(got - want, axis=-1)
    assert np.all(dev[use] <= err[use]), (case, int((dev[use] > err[use]).sum()), float((dev / err)[use].max()))
    assert use.sum() > 0.8 * len(use) and len(use) > 40, (case, int(use.sum()), len(use))
    if case.startswith(("slab", "wedge")):
        assert (use & (kind == 2)).sum() > 10 and (use & (kind == 1)).sum() > 10   # refraction and reflection rays
    return float((dev / err)[use].max())


@pytest.mark.parametrize("case", DEBUG_CASES)
def test_oracle_debug_ray_bounces_match_float64_sampling(oracle, case):
    sc = CASES[case]()
    osc = oracle.OracleScene(sc.desc)
    print(case, _check_debug(case, lambda px: osc.debug_ray(sc.cam, sc.film, DEBUG_SAMPLER, sc.integ, px)[0]))


@pytest.mark.gpu
@pytest.mark.parametrize("case", DEBUG_CASES)
def test_gpu_debug_ray_bounces_match_float64_sampling_and_the_oracle(gpu_ctx, oracle, case):
    sc = CASES[case]()
    osc = oracle.OracleScene(sc.desc)
    dev = api.Scene(gpu_ctx, sc.desc)
    try:
        rn = api.Renderer(gpu_ctx)
        for px in DEBUG_PIXELS[::7]:
            g = rn.debug_ray(dev, sc.cam, sc.film, DEBUG_SAMPLER, sc.integ, px)[0]
            assert g.tobytes() == osc.debug_ray(sc.cam, sc.film, DEBUG_SAMPLER, sc.integ, px)[0].tobytes(), (case, px)
        _check_debug(case, lambda px: rn.debug_ray(dev, sc.cam, sc.film, DEBUG_SAMPLER, sc.integ, px)[0])
    finally:
        dev.close()
