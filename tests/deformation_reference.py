"""CPU restatement of the deformation term of the previous-position AOV (rt_set_instance_deformation, include/rt_core.h),
float32 operation by operation in the kernel's order, on the oracle's primary hits over the oracle's own refitted BLAS.
It composes with tests/motion_reference.py: P' = apply_motion(P) + Dw."""
import numpy as np

import motion_reference as mr
import temporal_denoise_reference as tdr
from dxrexperiments_b200 import types as T

F = np.float32


def refitted_blas(orc, rest_mesh, mesh=None):
    """The oracle's ALLOW_UPDATE BLAS of `rest_mesh`, refitted (orc_blas_update) to `mesh`'s vertices when given."""
    b = orc.Blas.from_mesh(rest_mesh, build_flags=T.BUILD_FLAG_ALLOW_UPDATE)
    if mesh is not None:
        b.update([dict(vertices=mesh.vertices, stride=24, indices=mesh.indices, flags=T.GEOMETRY_FLAG_OPAQUE)])
    return b


def descriptors(prev_positions, object_to_previous_world):
    """One (previous positions (V, 3) float32 or None, row-major 3x4 float32) per instance."""
    return [(None if p is None else np.asarray(p, np.float32).reshape(-1, 3), np.asarray(m, np.float32).reshape(12))
            for p, m in zip(prev_positions, object_to_previous_world)]


def displacement(hits, inst_meshes, descs):
    """(Dw (n, 3) float32, applied (n,) bool, invalid (n,) bool) of n primary hits: `hits` carries bary, primitive_index
    and instance_index; inst_meshes[i] is the mesh whose vertex and index buffers instance i's hit record holds (this
    frame's vertices); descs as descriptors() (len = the bound n).  Dw is applied only where the instance has a descriptor
    with previous positions and valid indices; `invalid` marks the hits that set the status bit."""
    n = hits.shape[0]
    dw = np.zeros((n, 3), F)
    applied, invalid = np.zeros(n, bool), np.zeros(n, bool)
    inst = hits["instance_index"].astype(np.int64)
    for i, (prev, m) in enumerate(descs):
        sel = np.nonzero(inst == i)[0]
        if prev is None or sel.size == 0:
            continue
        mesh = inst_meshes[i]
        tri = mesh.indices.reshape(-1, 3)[hits["primitive_index"][sel]].astype(np.int64)
        ok = (tri < prev.shape[0]).all(axis=1)
        invalid[sel[~ok]] = True
        sel, tri = sel[ok], tri[ok]
        applied[sel] = True
        bu, bv = hits["bary"][sel, 0].astype(F), hits["bary"][sel, 1].astype(F)
        b = ((F(1) - bu) - bv, bu, bv)
        cur = mesh.vertices["position"].astype(F)
        d = [prev[tri[:, k]] - cur[tri[:, k]] for k in range(3)]
        D = (d[0] * b[0][:, None] + d[1] * b[1][:, None]) + d[2] * b[2][:, None]
        r = m.reshape(3, 4)
        for k in range(3):
            dw[sel, k] = (r[k, 0] * D[:, 0] + r[k, 1] * D[:, 1]) + r[k, 2] * D[:, 2]
    return dw, applied, invalid


def primary_previous_positions(orc, otlas, frame, w, h, motion, inst_meshes, descs):
    """(h, w, 4) float32: (P', 1) where the primary ray hits, 0 where it misses, with P' = apply_motion(P) + Dw."""
    rays = orc.primary_rays(frame, w, h, float(tdr.JITTER_SCALE))
    hits = otlas.trace(rays, T.RAY_FLAG_CULL_BACK_FACING_TRIANGLES)
    out = np.zeros((w * h, 4), np.float32)
    hit = hits["primitive_index"] != T.NO_HIT
    p = rays["origin"][hit] + hits["t"][hit, None] * rays["direction"][hit]
    q = mr.apply_motion(p, hits["instance_index"][hit], motion)
    dw, applied, _ = displacement(hits[hit], inst_meshes, descs)
    out[hit, :3] = np.where(applied[:, None], q + dw, q)
    out[hit, 3] = F(1)
    return out.reshape(h, w, 4)


def render_previous_positions(orc, otlas, frames, w, h, motion, inst_meshes, descs, half_targets=False):
    """The previous-position AOV accumulated over `frames` (one scene, one binding) as rt_dispatch_rays accumulates it."""
    acc = np.zeros((h, w, 4), np.float32)
    for f in frames:
        if f.cameraParams.accumCount >= f.options.maxIterations:
            continue
        n = F(f.cameraParams.accumCount)
        acc = (n * acc + primary_previous_positions(orc, otlas, f, w, h, motion, inst_meshes, descs)) / F(f.cameraParams.accumCount + 1)
        if half_targets:
            acc = acc.astype(np.float16).astype(np.float32)
    return acc
