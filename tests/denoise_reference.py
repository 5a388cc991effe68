"""TEST INFRASTRUCTURE ONLY: numpy float32 restatement of `yk_denoise` (include/yuki_gpu.h), the edge-avoiding a-trous
filter that has no counterpart in the reference. The rule is written for bit-exact restatement (un-fused float32 operations
in a fixed order, IEEE division and square root), so the GPU is compared with `denoise` bit for bit."""
import numpy as np

F = np.float32

_H5 = (F(1 / 16), F(1 / 4), F(3 / 8), F(1 / 4), F(1 / 16))


def _shift(a, dy, dx, fill):
    """out[y, x] = a[y + dy, x + dx] where that lies inside the film, else `fill`."""
    h, w = a.shape[:2]
    out = np.full_like(a, fill)
    if abs(dy) < h and abs(dx) < w:
        out[max(0, -dy):h - max(0, dy), max(0, -dx):w - max(0, dx)] = a[max(0, dy):h - max(0, -dy), max(0, dx):w - max(0, -dx)]
    return out


def denoise(film, radiance_sq, spp=None, sample_counts=None, normals=None, iterations=5, sigma=2.0, eps=1e-4):
    """yk_denoise (include/yuki_gpu.h): the edge-avoiding a-trous filter with per-pixel variance from `radiance_sq` and the
    sample counts (or `spp` for every pixel), optionally guided by a normal companion film. Every operation is the header's
    float32 one in its order; a tap that does not count adds +0, which leaves the (never negative-zero) sums unchanged."""
    c = np.array(film, np.float32)
    sq = np.asarray(radiance_sq, np.float32)
    h, w, _ = c.shape
    n = np.full((h, w), spp, np.uint32) if sample_counts is None else np.asarray(sample_counts, np.uint32).reshape(h, w)
    filt = n >= 2
    s2, e = F(sigma) * F(sigma), F(eps)
    with np.errstate(all="ignore"):
        v = sq - c * c
        v = np.where(v < F(0), F(0), v)
        v = v / (n.astype(np.float32) - F(1))[..., None]
        var = np.where(filt, (v[..., 0] + v[..., 1]) + v[..., 2], F(0))
        nh = None
        if normals is not None:
            d = np.asarray(normals, np.float32) * F(2) - F(1)
            l2 = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
            nh = np.where(((l2 > F(0)) & filt)[..., None], d / np.sqrt(l2)[..., None], F(0))
        for it in range(iterations):
            step = 1 << it
            W = np.zeros((h, w), np.float32)
            C = np.zeros((h, w, 3), np.float32)
            V = np.zeros((h, w), np.float32)
            for ky in range(5):
                for kx in range(5):
                    dy, dx = step * (ky - 2), step * (kx - 2)
                    if ky == 2 and kx == 2:
                        wt, cq, vq, count = np.full((h, w), _H5[2] * _H5[2], np.float32), c, var, np.ones((h, w), bool)
                    else:
                        cq, vq, fq = _shift(c, dy, dx, F(0)), _shift(var, dy, dx, F(0)), _shift(filt, dy, dx, False)
                        dc = c - cq
                        num = (dc[..., 0] * dc[..., 0] + dc[..., 1] * dc[..., 1]) + dc[..., 2] * dc[..., 2]
                        den = s2 * (var + vq) + e
                        wc = den / (den + num)
                        wc = wc * wc
                        wn = np.ones((h, w), np.float32)
                        if nh is not None:
                            nq = _shift(nh, dy, dx, F(0))
                            t = (nh[..., 0] * nq[..., 0] + nh[..., 1] * nq[..., 1]) + nh[..., 2] * nq[..., 2]
                            wn = np.where(t > F(0), t, F(0))
                            for _ in range(7):
                                wn = wn * wn
                        wt = ((_H5[ky] * _H5[kx]) * wn) * wc
                        count = fq & (wt > F(0))
                    W = W + np.where(count, wt, F(0))
                    C = C + np.where(count[..., None], wt[..., None] * cq, F(0))
                    V = V + np.where(count, (wt * wt) * vq, F(0))
            c = np.where(filt[..., None], C / W[..., None], c)
            var = np.where(filt, V / (W * W), var)
    return c.astype(np.float32)
