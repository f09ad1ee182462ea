"""CPU restatement of the previous-position AOV and of rt_denoise_temporal_motion (include/rt_core.h), float32 operation by
operation in the kernels' order.  The temporal pass itself is tests/temporal_denoise_reference.py's: the motion variant
is that pass with Q = previous_position.xyz in place of P in the reprojection and the position test, which is the same
as running it on Q and putting this frame's P back into history plane 3 (the only other place P goes)."""
import numpy as np

import temporal_denoise_reference as tdr
from dxrexperiments_b200 import types as T

F = np.float32


def motion_matrices(prev_transforms, transforms):
    """(n, 12) float32 world -> previous-world matrices prevObjectToWorld_i * inverse(objectToWorld_i), in float64 and
    rounded once (what Renderer.set_transforms binds)."""
    def four(t):
        t = np.asarray(t, np.float32).reshape(-1, 3, 4).astype(np.float64)
        m = np.zeros((t.shape[0], 4, 4))
        m[:, :3], m[:, 3, 3] = t, 1.0
        return m
    return (four(prev_transforms) @ np.linalg.inv(four(transforms)))[:, :3, :].reshape(-1, 12).astype(np.float32)


def apply_motion(position, inst, motion):
    """P' of every pixel: (..., 3) float32 P and (...) InstanceIndex(); each row ((m0*Px + m1*Py) + m2*Pz) + m3 in float32,
    and P itself (a copy) where there is no motion or inst >= n."""
    p = np.ascontiguousarray(position, np.float32)
    if motion is None or len(motion) == 0:
        return p.copy()
    m = np.asarray(motion, np.float32).reshape(-1, 3, 4)
    moved = inst < m.shape[0]
    rows = m[np.where(moved, inst, 0)]
    q = p.copy()
    with np.errstate(all="ignore"):
        for k in range(3):
            r = rows[..., k, :]
            v = ((r[..., 0] * p[..., 0] + r[..., 1] * p[..., 1]) + r[..., 2] * p[..., 2]) + r[..., 3]
            q[..., k] = np.where(moved, v, p[..., k])
    return q


def primary_previous_positions(orc, otlas, frame, w, h, motion):
    """(h, w, 4) float32: (P', 1) where the primary ray hits, 0 where it misses; P = o + t*d of the oracle's primary hit
    on the instance hits["instance_index"]."""
    rays = orc.primary_rays(frame, w, h, float(tdr.JITTER_SCALE))
    hits = otlas.trace(rays, T.RAY_FLAG_CULL_BACK_FACING_TRIANGLES)
    out = np.zeros((w * h, 4), np.float32)
    hit = hits["primitive_index"] != T.NO_HIT
    p = rays["origin"][hit] + hits["t"][hit, None] * rays["direction"][hit]
    out[hit, :3] = apply_motion(p, hits["instance_index"][hit], motion)
    out[hit, 3] = F(1)
    return out.reshape(h, w, 4)


def render_previous_positions(orc, otlas, frames, w, h, motion, half_targets=False):
    """The previous-position AOV accumulated over `frames` (one scene, one motion) as rt_dispatch_rays accumulates it."""
    acc = np.zeros((h, w, 4), np.float32)
    for f in frames:
        if f.cameraParams.accumCount >= f.options.maxIterations:
            continue
        n = F(f.cameraParams.accumCount)
        acc = (n * acc + primary_previous_positions(orc, otlas, f, w, h, motion)) / F(f.cameraParams.accumCount + 1)
        if half_targets:
            acc = acc.astype(np.float16).astype(np.float32)
    return acc


def temporal_history_motion(beauty, normal, position, previous_position, prev_camera=None, prev_history=None, **kw):
    """The (4, h, w, 4) history rt_denoise_temporal_motion writes."""
    hist = tdr.temporal_history(beauty, normal, previous_position, prev_camera, prev_history, **kw)
    hist[3] = np.ascontiguousarray(position, np.float32)
    return hist


def denoise_temporal_motion(beauty, albedo, normal, position, previous_position, prev_camera=None, prev_history=None, **kw):
    """(out (h, w, 4), history (4, h, w, 4)) float32 of rt_denoise_temporal_motion; keywords as
    temporal_denoise_reference.denoise_temporal."""
    out, hist = tdr.denoise_temporal(beauty, albedo, normal, previous_position, prev_camera, prev_history, **kw)
    hist[3] = np.ascontiguousarray(position, np.float32)
    return out, hist
