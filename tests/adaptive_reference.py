"""Float32 numpy restatement of adaptive sampling (include/rt_core.h, rt_set_adaptive_sampling / rt_adaptive_update).

A dispatch folds one sample into every active pixel with the pixel's own count n_p: v' = (n_p*v + s) / (n_p + 1), in the
kernels' operation order (the library is built with -fmad=false, so every float32 operation here rounds as the GPU's
does).  The random numbers are a pure function of (pixel, frameCount), so a pixel's k-th sample is the same value whichever
dispatches it takes part in: an adaptive render is composed exactly from a stack of one-sample frames (frameCount k,
accumCount 0) and the masks the update rule produces along the way.
"""
import numpy as np

F = np.float32
CONVERGED = np.uint32(0x80000000)
COUNT_MASK = np.uint32(0x7FFFFFFF)


def luminance(c):
    """(r*0.299f + g*0.587f) + b*0.114f of (..., >= 3) float32."""
    return (c[..., 0] * F(0.299) + c[..., 1] * F(0.587)) + c[..., 2] * F(0.114)


def to_half(a):
    return a.astype(np.float16).astype(np.float32)


def running_mean(prev, sample, n, half=False):
    """(n*prev + sample) / (n + 1) per pixel: prev and sample (..., C) float32, n (...) uint32 counts without bit 31."""
    fn = n.astype(F)[..., None]
    fn1 = (n + np.uint32(1)).astype(F)[..., None]
    out = (fn * prev + sample) / fn1
    return to_half(out) if half else out


def update_moments(moments, sample, n):
    """Fold the (already clamped) samples (..., >= 3) into the (..., 2) luminance moments with counts n."""
    l = luminance(sample)
    fn, fn1 = n.astype(F), (n + np.uint32(1)).astype(F)
    return np.stack([(fn * moments[..., 0] + l) / fn1, (fn * moments[..., 1] + l * l) / fn1], axis=-1)


def relative_error(counts, moments, floor):
    """e_p = sigma_p / (m1 + floor), sigma_p = sqrtf(fmaxf(0, m2 - m1*m1) / (n - 1)) for n >= 2, +inf below."""
    n = counts & COUNT_MASK
    m1, m2 = moments[..., 0], moments[..., 1]
    var = np.fmax(F(0), m2 - m1 * m1)  # fmaxf: a NaN difference gives 0
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        sigma = np.sqrt(var / np.maximum(n.astype(np.int64) - 1, 1).astype(F))
        e = sigma / (m1 + F(floor))
    return np.where(n >= 2, e, F(np.inf)).astype(F)


def update(counts, moments, threshold, floor, min_samples, max_samples):
    """rt_adaptive_update: (new counts, active count).  counts (h, w) uint32, moments (h, w, 2) float32."""
    counts = np.asarray(counts, np.uint32)
    h, w = counts.shape
    n = counts & COUNT_MASK
    with np.errstate(invalid="ignore"):
        ok = relative_error(counts, moments, floor) <= F(threshold)  # NaN fails
    padded = np.ones((h + 2, w + 2), bool)  # outside the image never holds a pixel back
    padded[1:-1, 1:-1] = ok
    window = np.ones((h, w), bool)
    for dy in range(3):
        for dx in range(3):
            window &= padded[dy:dy + h, dx:dx + w]
    conv = ((counts & CONVERGED) != 0) | (n >= max_samples) | ((n >= min_samples) & window)
    out = counts | np.where(conv, CONVERGED, np.uint32(0))
    return out, int((~conv).sum())


def compose(beauty, aovs=None, schedule=(), half=False, dispatches=None):
    """Compose an adaptive render from one-sample frames.

    beauty: (K, h, w, 4) float32, sample k of every pixel (gOutput of a dispatch with frameCount k and accumCount 0, fp32
    targets); aovs: dict name -> (K, h, w, 4) float32 one-sample AOV frames.  schedule: (after_dispatch, params) pairs;
    after dispatch number `after_dispatch` (1-based) the update runs with params = (threshold, floor, min_samples,
    max_samples).  half: the stores round through fp16 (moments stay fp32).  Returns a dict with "beauty", "aovs",
    "counts" (with bit 31), "moments", "active" (the active count after each update) and "dispatches"."""
    K, h, w, _ = beauty.shape
    dispatches = K if dispatches is None else dispatches
    aovs = aovs or {}
    out = np.zeros((h, w, 4), F)
    aout = {k: np.zeros((h, w, 4), F) for k in aovs}
    counts = np.zeros((h, w), np.uint32)
    moments = np.zeros((h, w, 2), F)
    plan = dict(schedule)
    active_log = []
    for k in range(dispatches):
        act = (counts & CONVERGED) == 0
        n = counts[act]
        out[act] = running_mean(out[act], beauty[k][act], n, half)
        for name, frames in aovs.items():
            aout[name][act] = running_mean(aout[name][act], frames[k][act], n, half)
        moments[act] = update_moments(moments[act], beauty[k][act], n)
        counts[act] = n + np.uint32(1)
        if k + 1 in plan:
            counts, active = update(counts, moments, *plan[k + 1])
            active_log.append(active)
    return {"beauty": out, "aovs": aout, "counts": counts, "moments": moments, "active": active_log, "dispatches": dispatches}


def every(k, params, dispatches):
    """An update after every k-th of `dispatches` dispatches."""
    return [(d, params) for d in range(k, dispatches + 1, k)]


def run_until_converged(beauty, params, update_every, aovs=None, half=False):
    """Dispatch and update every `update_every` dispatches until no pixel is active or the frames run out; returns
    compose()'s dict."""
    K = beauty.shape[0]
    res = compose(beauty, aovs, every(update_every, params, K), half)
    # the dispatches after the last active pixel converged change nothing; report how many were needed
    for i, a in enumerate(res["active"]):
        if a == 0:
            res["dispatches"] = (i + 1) * update_every
            break
    return res


def rel_mse(a, ref, eps=1e-2):
    """Mean relative squared error of the luminance, (a - ref)^2 / (ref^2 + eps): the error measure adaptive sampling's
    relative-error rule targets."""
    la, lr = luminance(a).astype(np.float64), luminance(ref).astype(np.float64)
    return float(np.mean((la - lr) ** 2 / (lr * lr + eps)))
