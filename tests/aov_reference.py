"""CPU reference for the AOV outputs of the progressive program (rt_set_aov_output), built from the unchanged oracle.

AOVs 0-4 are defined as what debug views show: AOV k is the oracle's beauty frame rendered with debug view k switched on,
from the same frames.  The normal AOV is the running mean of (N, 1) on a primary hit and (0, 0, 0, 0) on a miss, where N
is the normalised interpolated vertex normal shade() receives: the oracle's primary hit (same rays, flags and traversal as
PrimaryClosestHit) and the interpolation and normalisation of oracle_shade.cpp / oracle_internal.h restated in float32,
operation by operation.
"""
import numpy as np

from closed_form import camera_rays, const_env
from dxrexperiments_b200 import scenes, types as T
from helpers import SceneCase

VIEW_OF_AOV = {"direct": "showDirectLightingOnly", "indirect-diffuse": "showIndirectDiffuseOnly",
               "indirect-specular": "showIndirectSpecularOnly", "albedo": "showGBufferAlbedoOnly", "fresnel": "showFresnelTerm"}


def _store(v, half):
    return v.astype(np.float16).astype(np.float32) if half else v


def primary_normals(orc, otlas, meshes, frame, w, h):
    """(h, w, 4) float32: (N, 1) where the primary ray hits, 0 where it misses."""
    rays = orc.primary_rays(frame, w, h, 30.0)  # the progressive RayGen's jitter scale
    hits = otlas.trace(rays, T.RAY_FLAG_CULL_BACK_FACING_TRIANGLES)
    out = np.zeros((w * h, 4), np.float32)
    hit = hits["primitive_index"] != T.NO_HIT
    one = np.float32(1.0)
    for inst, mesh in enumerate(meshes):  # instance i carries the records of mesh i (hit group 2 i)
        sel = hit & (hits["instance_index"] == inst)
        if not sel.any():
            continue
        hs = hits[sel]
        idx = mesh.indices.reshape(-1, 3)[hs["primitive_index"]]
        nrm = mesh.vertices["normal"].astype(np.float32)
        n0, n1, n2 = nrm[idx[:, 0]], nrm[idx[:, 1]], nrm[idx[:, 2]]
        bu, bv = hs["bary"][:, 0], hs["bary"][:, 1]
        b0 = (one - bu) - bv
        n = (n0 * b0[:, None] + n1 * bu[:, None]) + n2 * bv[:, None]
        dot = (n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]) + n[:, 2] * n[:, 2]
        inv = one / np.sqrt(dot)
        out[sel, :3] = n * inv[:, None]
        out[sel, 3] = one
    return out.reshape(h, w, 4)


def render_aovs(orc, otlas, recs, meshes, env, frames, w, h, names=T.AOV_NAMES, half_targets=False, threads=8):
    """Accumulate the named AOVs over `frames` exactly as rt_dispatch_rays accumulates them.  The caller sets the oracle's
    render options (radiance depth, fp16 targets) to match the GPU side."""
    out = {}
    for name in names:
        acc = np.zeros((h, w, 4), np.float32)
        for f in frames:
            if name == "normal":
                if f.cameraParams.accumCount >= f.options.maxIterations:  # RayGen's early-out
                    continue
                n = np.float32(f.cameraParams.accumCount)
                acc = _store((n * acc + primary_normals(orc, otlas, meshes, f, w, h)) / np.float32(f.cameraParams.accumCount + 1),
                             half_targets)
            else:
                fv = T.PerFrameConstants.from_buffer_copy(bytes(f))
                setattr(fv.options, VIEW_OF_AOV[name], 1)
                orc.render_progressive(otlas, recs, env, fv, w, h, acc, threads=threads)
        out[name] = acc
    return out


def plane_case(w=96, h=64, half=1.0):
    """A square of normal +z under a black sky, its closed-form coverage: (case, on, off) with `on` / `off` the pixels whose
    jitter-free primary ray passes at least 1e-3 inside / outside the square's edge (nearer ones may go either way in
    float32)."""
    plane = scenes.quad((-half, -half, 0), (half, -half, 0), (half, half, 0), (-half, half, 0))
    mat = scenes.make_material(albedo=(0.5, 0.5, 0.5, 1.0), type=0, reflectivity=0.0, emissive=(0, 0, 0, 0))
    setup = scenes.FrameSetup(camera=scenes.Camera(eye=(0.3, -0.2, 4.0), at=(0.0, 0.0, 0.0)))
    case = SceneCase([plane], materials=[mat], setup=setup, env_size=0)
    case.env = const_env((0, 0, 0))
    o, d = camera_rays(setup, w, h)
    t = -o[..., 2] / d[..., 2]
    p = o + t[..., None] * d
    edge = np.max(np.abs(p[..., :2]), axis=-1)
    return case, edge < half - 1e-3, edge > half + 1e-3


def check_plane_normals(n, on, off):
    """x, y exactly 0 and coverage exactly 1 on the square; z within one ulp of 1, since the barycentric weights may sum to
    1 - 2^-24 before the normalisation; exactly 0 everywhere on the sky."""
    assert on.sum() > 0.2 * on.size and off.sum() > 0.2 * off.size
    np.testing.assert_array_equal(n[on][:, [0, 1, 3]], np.tile([0.0, 0.0, 1.0], (on.sum(), 1)))
    np.testing.assert_allclose(n[on][:, 2], 1.0, rtol=0, atol=1.2e-7)
    assert not n[off].any()
