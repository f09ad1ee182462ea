"""CPU restatement of rt_denoise_temporal (include/rt_core.h): SVGF's temporal pass (reproject through the position AOV,
bilinear history fetch with normal and position rejection, exponential blend of colour and luminance moments, variance
from the moments) in front of the a-trous stage of rt_denoise_progressive.  Vectorised over the image, float32 operation
by operation in the kernels' order (tests/progressive_denoise_reference.py does the same for the spatial filter, whose
helpers this file uses).  Also the position AOV's reference: P = o + t*d of the oracle's primary hits."""
import numpy as np

import progressive_denoise_reference as pdr
from dxrexperiments_b200 import types as T

F = np.float32
JITTER_SCALE = F(30.0)  # the progressive RayGen's (primary_ray's o = eye + jitters * 30)
HISTORY_CAP = F(32.0)


def default_params():
    """{keyword: value} of types.temporal_denoise_defaults(), in the keywords of denoise_temporal()."""
    return params_dict(T.temporal_denoise_defaults())


def params_dict(p):
    s = p.spatial
    return dict(iterations=s.iterations, normal_exponent_log2=s.normal_exponent_log2, sigma_luminance=s.sigma_luminance,
                sigma_albedo=s.sigma_albedo, alpha_color=p.alpha_color, alpha_moments=p.alpha_moments, normal_cos=p.normal_cos,
                position_tolerance=p.position_tolerance)


def make_params(iterations=5, normal_exponent_log2=7, sigma_luminance=4.0, sigma_albedo=0.1, alpha_color=0.2,
                alpha_moments=0.2, normal_cos=0.9, position_tolerance=0.02):
    return T.TemporalDenoiseParams(T.ProgressiveDenoiseParams(iterations, normal_exponent_log2, sigma_luminance, sigma_albedo),
                                   alpha_color, alpha_moments, normal_cos, position_tolerance)


def primary_positions(orc, otlas, frame, w, h):
    """(h, w, 4) float32: (P, 1) with P = o + t*d where the primary ray hits, 0 where it misses."""
    rays = orc.primary_rays(frame, w, h, float(JITTER_SCALE))
    hits = otlas.trace(rays, T.RAY_FLAG_CULL_BACK_FACING_TRIANGLES)
    out = np.zeros((w * h, 4), np.float32)
    hit = hits["primitive_index"] != T.NO_HIT
    out[hit, :3] = rays["origin"][hit] + hits["t"][hit, None] * rays["direction"][hit]
    out[hit, 3] = F(1)
    return out.reshape(h, w, 4)


def render_positions(orc, otlas, frames, w, h, half_targets=False):
    """The position AOV accumulated over `frames` exactly as rt_dispatch_rays accumulates it."""
    acc = np.zeros((h, w, 4), np.float32)
    for f in frames:
        if f.cameraParams.accumCount >= f.options.maxIterations:  # RayGen's early-out
            continue
        n = F(f.cameraParams.accumCount)
        acc = (n * acc + primary_positions(orc, otlas, f, w, h)) / F(f.cameraParams.accumCount + 1)
        if half_targets:
            acc = acc.astype(np.float16).astype(np.float32)
    return acc


def _dot(a, b):
    return (a[..., 0] * b[0] + a[..., 1] * b[1]) + a[..., 2] * b[2]


def reproject(normal, position, prev_camera):
    """(ok, fx, fy, r = P - o'): where pixel p's world position lands in the previous frame's image; `ok` marks the pixels that
    may take history at all (coverage 1, in front of the previous camera, (fx, fy) within (-1, w) x (-1, h))."""
    h, w = normal.shape[:2]
    cam = prev_camera
    eye, jit = np.array(cam.worldEyePos[:3], F), np.array(cam.jitters[:], F)
    o = np.array([eye[0] + jit[0] * JITTER_SCALE, eye[1] + jit[1] * JITTER_SCALE, eye[2] + F(0)], F)
    U, V, W = (np.array(v[:3], F) for v in (cam.U, cam.V, cam.W))
    r = position[..., :3] - o
    with np.errstate(all="ignore"):
        zc = _dot(r, W) / _dot(W, W)
        sx = (_dot(r, U) / _dot(U, U)) / zc
        sy = -((_dot(r, V) / _dot(V, V)) / zc)
        fx = ((sx + F(1)) * F(0.5)) * F(w) - F(0.5)
        fy = ((sy + F(1)) * F(0.5)) * F(h) - F(0.5)
        ok = (normal[..., 3] == F(1)) & (zc > F(0)) & (fx > F(-1)) & (fx < F(w)) & (fy > F(-1)) & (fy < F(h))
    return ok, np.where(ok, fx, F(0)), np.where(ok, fy, F(0)), r


def temporal_history(beauty, normal, position, prev_camera=None, prev_history=None, alpha_color=0.2, alpha_moments=0.2,
                     normal_cos=0.9, position_tolerance=0.02):
    """Steps 1-3 (reproject, bilinear fetch, blend): the (4, h, w, 4) float32 history rt_denoise_temporal writes."""
    beauty, normal, position = (np.ascontiguousarray(a, np.float32) for a in (beauty, normal, position))
    h, w = beauty.shape[:2]
    ch = np.zeros((h, w, 3), np.float32)
    nh, m1h, m2h = (np.zeros((h, w), np.float32) for _ in range(3))
    if prev_history is not None:
        prev = np.ascontiguousarray(prev_history, np.float32).reshape(4, h, w, 4)
        ok, fx, fy, r = reproject(normal, position, prev_camera)
        x0f, y0f = np.floor(fx), np.floor(fy)
        ax, ay = fx - x0f, fy - y0f
        x0, y0 = x0f.astype(np.int64), y0f.astype(np.int64)
        lim = F(position_tolerance) * np.sqrt((r[..., 0] * r[..., 0] + r[..., 1] * r[..., 1]) + r[..., 2] * r[..., 2])
        sw = np.zeros((h, w), np.float32)
        one = F(1)
        with np.errstate(all="ignore"):
            for dy in (0, 1):
                for dx in (0, 1):
                    qx, qy = x0 + dx, y0 + dy
                    wt = (ax if dx else one - ax) * (ay if dy else one - ay)
                    take = ok & (qx >= 0) & (qy >= 0) & (qx < w) & (qy < h) & (wt != 0)
                    qxc, qyc = np.clip(qx, 0, w - 1), np.clip(qy, 0, h - 1)
                    nq, pq = prev[2][qyc, qxc], prev[3][qyc, qxc]
                    take &= (nq[..., 3] == one) & ~((normal[..., 0] * nq[..., 0] + normal[..., 1] * nq[..., 1]) +
                                                     normal[..., 2] * nq[..., 2] < F(normal_cos))
                    e = pq[..., :3] - position[..., :3]
                    take &= ~(np.sqrt((e[..., 0] * e[..., 0] + e[..., 1] * e[..., 1]) + e[..., 2] * e[..., 2]) > lim)
                    cq, mq = prev[0][qyc, qxc], prev[1][qyc, qxc]
                    ch = np.where(take[..., None], ch + wt[..., None] * cq[..., :3], ch)
                    nh = np.where(take, nh + wt * cq[..., 3], nh)
                    m1h = np.where(take, m1h + wt * mq[..., 0], m1h)
                    m2h = np.where(take, m2h + wt * mq[..., 1], m2h)
                    sw = np.where(take, sw + wt, sw)
            some = sw > 0
            ch = np.where(some[..., None], ch / sw[..., None], ch)
            nh, m1h, m2h = (np.where(some, v / sw, v) for v in (nh, m1h, m2h))
    n = np.minimum(nh + F(1), HISTORY_CAP)
    a = np.maximum(F(1) / n, F(alpha_color))
    am = np.maximum(F(1) / n, F(alpha_moments))
    lum = pdr.luminance(beauty)
    hist = np.zeros((4, h, w, 4), np.float32)
    hist[0, ..., :3] = (F(1) - a)[..., None] * ch + a[..., None] * beauty[..., :3]
    hist[0, ..., 3] = n
    hist[1, ..., 0] = (F(1) - am) * m1h + am * lum
    hist[1, ..., 1] = (F(1) - am) * m2h + am * (lum * lum)
    hist[2], hist[3] = normal, position
    return hist


def window_variance(c, normal, nexp):
    """var0 of rt_denoise_progressive: max(0, m2 - m1^2) of L over the wN-weighted 7 x 7 window (0 on sky)."""
    lum = pdr.luminance(c)
    s1, s2, sw = (np.zeros(c.shape[:2], np.float32) for _ in range(3))
    with np.errstate(all="ignore"):
        for dy in range(-3, 4):
            for dx in range(-3, 4):
                lq, ok = pdr._shift(lum, dx, dy)
                if dx == 0 and dy == 0:
                    wn = np.ones_like(lum)
                else:
                    wn = pdr._normal_weight(normal, pdr._shift(normal, dx, dy)[0], nexp)
                    ok &= wn != 0
                s1 = np.where(ok, s1 + wn * lq, s1)
                s2 = np.where(ok, s2 + wn * (lq * lq), s2)
                sw = np.where(ok, sw + wn, sw)
        m1, m2 = s1 / sw, s2 / sw
        return np.where(normal[..., 3] != 0, np.maximum(F(0), m2 - m1 * m1), F(0)).astype(np.float32)


def atrous(c, var, albedo, normal, iterations, nexp, sigma_luminance, sigma_albedo, half_targets):
    """Step 5: rt_denoise_progressive's a-trous iterations on (C, var0), in progressive_denoise_reference's order."""
    sig_l = F(sigma_luminance)
    inv_a = F(1) / F(sigma_albedo) if sigma_albedo > 0 else F(0)
    hit = normal[..., 3] != 0
    B5, H3 = pdr.B5, pdr.H3
    with np.errstate(all="ignore"):
        for it in range(int(iterations)):
            step = 1 << it
            gs, gw = np.zeros_like(var), np.zeros_like(var)
            for dy in range(-1, 2):
                for dx in range(-1, 2):
                    vq, ok = pdr._shift(var, dx, dy)
                    wn = np.ones_like(var) if dx == 0 and dy == 0 else pdr._normal_weight(normal, pdr._shift(normal, dx, dy)[0], nexp)
                    wg = (H3[dx + 1] * H3[dy + 1]) * wn
                    ok &= (wn != 0) & (wg != 0)
                    gs = np.where(ok, gs + wg * vq, gs)
                    gw = np.where(ok, gw + wg, gw)
            g = gs / gw
            inv_l = F(1) / (sig_l * np.sqrt(g) + F(1e-10))
            lp = pdr.luminance(c)
            acc = np.zeros_like(c)
            sv, sw = np.zeros_like(var), np.zeros_like(var)
            for dy in range(-2, 3):
                for dx in range(-2, 3):
                    cq, ok = pdr._shift(c, step * dx, step * dy)
                    vq = pdr._shift(var, step * dx, step * dy)[0]
                    if dx == 0 and dy == 0:
                        w = np.full(var.shape, B5[2] * B5[2], np.float32)
                    else:
                        wn = pdr._normal_weight(normal, pdr._shift(normal, step * dx, step * dy)[0], nexp)
                        aq = pdr._shift(albedo, step * dx, step * dy)[0]
                        dl = np.abs(lp - pdr.luminance(cq))
                        da = (np.abs(albedo[..., 0] - aq[..., 0]) + np.abs(albedo[..., 1] - aq[..., 1])) + np.abs(albedo[..., 2] - aq[..., 2])
                        w = ((B5[dx + 2] * B5[dy + 2]) * wn) * np.exp(-(dl * inv_l + da * inv_a))
                        ok &= (wn != 0) & (w != 0)
                    acc = np.where(ok[..., None], acc + w[..., None] * cq, acc)
                    sv = np.where(ok, sv + (w * w) * vq, sv)
                    sw = np.where(ok, sw + w, sw)
            c = np.where(hit[..., None], acc / sw[..., None], c).astype(np.float32)
            var = np.where(hit, sv / (sw * sw), var).astype(np.float32)
    out = np.ones(c.shape[:2] + (4,), np.float32)
    out[..., :3] = pdr._half(c) if half_targets else c
    return out


def denoise_temporal(beauty, albedo, normal, position, prev_camera=None, prev_history=None, iterations=5, normal_exponent_log2=7,
                     sigma_luminance=4.0, sigma_albedo=0.1, alpha_color=0.2, alpha_moments=0.2, normal_cos=0.9,
                     position_tolerance=0.02, half_targets=False):
    """(h, w, 4) float32 images in (and the previous camera and history, or None for a first frame), (out (h, w, 4),
    history (4, h, w, 4)) float32 out: rt_denoise_temporal."""
    assert (prev_camera is None) == (prev_history is None)
    albedo, normal = (np.ascontiguousarray(a, np.float32) for a in (albedo, normal))
    hist = temporal_history(beauty, normal, position, prev_camera, prev_history, alpha_color, alpha_moments, normal_cos,
                            position_tolerance)
    c = hist[0, ..., :3].copy()
    nexp = int(normal_exponent_log2)
    var = np.where(hist[0, ..., 3] >= F(4), np.maximum(F(0), hist[1, ..., 1] - hist[1, ..., 0] * hist[1, ..., 0]),
                   window_variance(c, normal, nexp)).astype(np.float32)
    return atrous(c, var, albedo, normal, iterations, nexp, sigma_luminance, sigma_albedo, half_targets), hist


def orbit_frames(setup, w, h, frames, degrees, first_sample=0, jitter=None):
    """One-sample frames (accumCount 0) of a camera orbiting setup.camera's `at` by `degrees` per frame; frameCount runs
    from first_sample.  jitter: (frames, 2) or None for jitter-free frames."""
    import dataclasses

    from dxrexperiments_b200 import scenes
    out = []
    for f in range(frames):
        s = dataclasses.replace(setup, camera=scenes.orbit(setup.camera, f * degrees))
        out.append(scenes.make_frame(s, w, h, first_sample + f, 0, jitter=(0.0, 0.0) if jitter is None else jitter[f]))
    return out
