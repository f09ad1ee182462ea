"""CPU restatement of rt_denoise_progressive (include/rt_core.h): spatial SVGF, an edge-avoiding a-trous filter guided by the
albedo and normal AOVs.  Vectorised over the image, float32 operation by operation in the kernels' order: every window is
summed tap by tap in row-major order (dy outer), and a tap outside the image or with weight 0 is skipped, not added as 0.
Only expf and sqrtf may then differ from the GPU (by an ulp or so)."""
import numpy as np

F = np.float32
B5 = (F(1 / 16), F(1 / 4), F(3 / 8), F(1 / 4), F(1 / 16))
H3 = (F(1 / 4), F(1 / 2), F(1 / 4))


def default_params():
    """(iterations, normal_exponent_log2, sigma_luminance, sigma_albedo): types.progressive_denoise_defaults()."""
    from dxrexperiments_b200 import types as T
    p = T.progressive_denoise_defaults()
    return p.iterations, p.normal_exponent_log2, p.sigma_luminance, p.sigma_albedo


def luminance(c):
    return (c[..., 0] * F(0.299) + c[..., 1] * F(0.587)) + c[..., 2] * F(0.114)


def _shift(img, dx, dy):
    """img[y + dy, x + dx] where that is inside the image (zeros elsewhere), and the in-image mask."""
    h, w = img.shape[:2]
    out = np.zeros_like(img)
    ok = np.zeros((h, w), bool)
    if abs(dx) >= w or abs(dy) >= h:
        return out, ok
    ys, yd = slice(max(dy, 0), h + min(dy, 0)), slice(max(-dy, 0), h + min(-dy, 0))
    xs, xd = slice(max(dx, 0), w + min(dx, 0)), slice(max(-dx, 0), w + min(-dx, 0))
    out[yd, xd] = img[ys, xs]
    ok[yd, xd] = True
    return out, ok


def _normal_weight(n, nq, nexp):
    d = np.maximum(F(0), (n[..., 0] * nq[..., 0] + n[..., 1] * nq[..., 1]) + n[..., 2] * nq[..., 2])
    for _ in range(nexp):
        d = d * d
    return d


def _half(v):
    return v.astype(np.float16).astype(np.float32)


def denoise(beauty, albedo, normal, iterations=5, normal_exponent_log2=7, sigma_luminance=4.0, sigma_albedo=0.1,
            half_targets=False):
    """(h, w, 4) float32 in, (h, w, 4) float32 out: the filter of rt_denoise_progressive."""
    beauty, albedo, normal = (np.ascontiguousarray(a, np.float32) for a in (beauty, albedo, normal))
    nexp, sig_l = int(normal_exponent_log2), F(sigma_luminance)
    inv_a = F(1) / F(sigma_albedo) if sigma_albedo > 0 else F(0)
    hit = normal[..., 3] != 0
    with np.errstate(all="ignore"):
        # variance pass: m1, m2 over the 7 x 7 window
        c = beauty[..., :3].copy()
        lum = luminance(c)
        s1, s2, sw = (np.zeros(c.shape[:2], np.float32) for _ in range(3))
        for dy in range(-3, 4):
            for dx in range(-3, 4):
                lq, ok = _shift(lum, dx, dy)
                if dx == 0 and dy == 0:
                    wn = np.ones_like(lum)
                else:
                    wn = _normal_weight(normal, _shift(normal, dx, dy)[0], nexp)
                    ok &= wn != 0
                s1 = np.where(ok, s1 + wn * lq, s1)
                s2 = np.where(ok, s2 + wn * (lq * lq), s2)
                sw = np.where(ok, sw + wn, sw)
        m1, m2 = s1 / sw, s2 / sw
        var = np.where(hit, np.maximum(F(0), m2 - m1 * m1), F(0)).astype(np.float32)
        for it in range(int(iterations)):
            step = 1 << it
            gs, gw = np.zeros_like(var), np.zeros_like(var)
            for dy in range(-1, 2):
                for dx in range(-1, 2):
                    vq, ok = _shift(var, dx, dy)
                    wn = np.ones_like(var) if dx == 0 and dy == 0 else _normal_weight(normal, _shift(normal, dx, dy)[0], nexp)
                    wg = (H3[dx + 1] * H3[dy + 1]) * wn
                    ok &= (wn != 0) & (wg != 0)
                    gs = np.where(ok, gs + wg * vq, gs)
                    gw = np.where(ok, gw + wg, gw)
            g = gs / gw
            inv_l = F(1) / (sig_l * np.sqrt(g) + F(1e-10))
            lp = luminance(c)
            acc = np.zeros_like(c)
            sv, sw = np.zeros_like(var), np.zeros_like(var)
            for dy in range(-2, 3):
                for dx in range(-2, 3):
                    cq, ok = _shift(c, step * dx, step * dy)
                    vq = _shift(var, step * dx, step * dy)[0]
                    if dx == 0 and dy == 0:
                        w = np.full(var.shape, B5[2] * B5[2], np.float32)
                    else:
                        wn = _normal_weight(normal, _shift(normal, step * dx, step * dy)[0], nexp)
                        aq = _shift(albedo, step * dx, step * dy)[0]
                        dl = np.abs(lp - luminance(cq))
                        da = (np.abs(albedo[..., 0] - aq[..., 0]) + np.abs(albedo[..., 1] - aq[..., 1])) + np.abs(albedo[..., 2] - aq[..., 2])
                        w = ((B5[dx + 2] * B5[dy + 2]) * wn) * np.exp(-(dl * inv_l + da * inv_a))
                        ok &= (wn != 0) & (w != 0)
                    acc = np.where(ok[..., None], acc + w[..., None] * cq, acc)
                    sv = np.where(ok, sv + (w * w) * vq, sv)
                    sw = np.where(ok, sw + w, sw)
            c = np.where(hit[..., None], acc / sw[..., None], c).astype(np.float32)
            var = np.where(hit, sv / (sw * sw), var).astype(np.float32)
    out = np.ones(beauty.shape, np.float32)
    out[..., :3] = _half(c) if half_targets else c
    return out


def synthetic_inputs(w, h, seed, sky_fraction=0.2):
    """Noisy beauty, piecewise albedo and unit normals from four directions, with random sky pixels (coverage 0, N = 0) and
    some partially covered ones: (beauty, albedo, normal), each (h, w, 4) float32."""
    rng = np.random.Generator(np.random.PCG64(seed))
    beauty = np.ones((h, w, 4), np.float32)
    beauty[..., :3] = rng.gamma(1.5, 0.4, size=(h, w, 3)).astype(np.float32)
    albedo = np.ones((h, w, 4), np.float32)
    albedo[..., :3] = rng.choice(np.array([[0.8, 0.2, 0.1], [0.3, 0.6, 0.9], [0.5, 0.5, 0.5]], np.float32), size=(h, w))
    dirs = np.array([[0, 0, 1], [1, 0, 0], [0, 1, 0], [0.6, 0, 0.8]], np.float32)
    normal = np.zeros((h, w, 4), np.float32)
    normal[..., :3] = dirs[(np.arange(w)[None, :] * 4 // max(w, 1) + np.arange(h)[:, None] * 2 // max(h, 1)) % 4]
    normal[..., 3] = 1
    part = rng.random((h, w)) < 0.1
    normal[part] *= np.float32(0.5)
    sky = rng.random((h, w)) < sky_fraction
    normal[sky] = 0
    return beauty, albedo, normal


def halves_inputs(w, h, seed):
    """Left half normal +z, right half +x: exactly perpendicular, so no tap crosses between the halves."""
    beauty, albedo, normal = synthetic_inputs(w, h, seed, sky_fraction=0.0)
    normal[...] = (0, 0, 1, 1)
    normal[:, w // 2:] = (1, 0, 0, 1)
    return beauty, albedo, normal
