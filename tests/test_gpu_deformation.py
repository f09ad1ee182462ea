"""GPU: the deformation term of the previous-position AOV (rt_set_instance_deformation) and Renderer.set_vertices against
their CPU restatement (tests/deformation_reference.py), their exact properties, argument checks, and the history they
keep on a deforming mesh."""
import ctypes as C

import numpy as np
import pytest

import deformation_reference as dr
import motion_reference as mr
import temporal_denoise_reference as tdr
from dxrexperiments_b200 import scenes, types as T
from helpers import SceneCase
from test_deformation_reference import check_quality, quality, sheet_frame_case
from test_gpu_instance_motion import bunny_instances
from test_gpu_temporal_denoise import _check_history, _check_out, _kw

pytestmark = pytest.mark.gpu
RT_ERR_INVALID_ARG = -1
POS, PREV = T.AOV_POSITION_NAME, T.AOV_PREVIOUS_POSITION_NAME
GUIDES = ("albedo", "normal", POS, PREV)
BUNNY_SHEAR = (1.5, 0.5, -1.0)  # the bunny's top moves by this (object space) between the two frames


def _renderer(rt, ctx, case, w, h, aovs, instance_mesh=None, deforming=(0,), **kw):
    return rt.Renderer(ctx, case.meshes, case.transforms, case.materials, case.env, rt.PROGRESSIVE, w, h, aovs=aovs,
                       instance_mesh=instance_mesh, deforming=deforming, **kw)


def _frames(case, w, h, spp, seed=31):
    jit = scenes.jitter_sequence(seed, spp, w, h)
    return [scenes.make_frame(case.setup, w, h, s, s, jitter=jit[s]) for s in range(spp)]


def _deformed(kind):
    """(case at rest, deformed mesh 0, case after a rigid motion, instance_mesh) of a deforming scene: the waving sheet
    from frame 2 to 3 (moved as a whole by 0.1 along x when rigid motion is added), or eight instances of one bunny
    sheared by BUNNY_SHEAR (moved by bunny_instances' next transforms)."""
    if kind == "cornell":
        rest = sheet_frame_case(2)
        moved = sheet_frame_case(2)
        moved.transforms = [np.array([1, 0, 0, 0.1, 0, 1, 0, 0, 0, 0, 1, 0], np.float32), moved.transforms[1]]
        return rest, sheet_frame_case(3).meshes[0], moved, None
    rest, moved = bunny_instances(10), bunny_instances(11)
    moved.meshes = rest.meshes
    m = rest.meshes[0]
    v = m.vertices.copy()
    v["position"] = scenes.sheared_positions(v["position"], BUNNY_SHEAR)
    return rest, scenes.Mesh(v, m.indices), moved, [0] * 8


def _deform(r, mesh):
    r.set_vertices(0, mesh.vertices["position"], mesh.vertices["normal"])


def _oracle(orc, rest, mesh, case, instance_mesh):
    """(oracle TLAS over the refitted BLAS of mesh 0 and the other meshes, per-instance meshes, descriptors)."""
    blases = [dr.refitted_blas(orc, rest.meshes[0], mesh)] + [orc.Blas.from_mesh(m) for m in rest.meshes[1:]]
    im = instance_mesh or list(range(len(rest.meshes)))
    meshes = [mesh] + rest.meshes[1:]
    prev = [rest.meshes[0].vertices["position"] if k == 0 else None for k in im]
    return orc.Tlas([blases[k] for k in im], case.transforms), [meshes[k] for k in im], dr.descriptors(prev, rest.transforms)


def _setup(rt, ctx, kind, motion, w, h, aovs=(POS, PREV), **kw):
    rest, mesh, moved, im = _deformed(kind)
    r = _renderer(rt, ctx, rest, w, h, aovs, im, **kw)
    if motion:
        r.set_transforms(moved.transforms)
    _deform(r, mesh)
    return r, rest, mesh, (moved if motion else rest), im


# ---------------------------------------------------------------------------------------------------- the AOV
@pytest.mark.parametrize("motion", [False, True])
@pytest.mark.parametrize("kind", ["cornell", "bunny"])
def test_one_sample_is_the_restatement_of_the_gpus_own_hits_exactly(kind, motion, ctx, rt):
    """At one sample with fp32 targets the AOV is the rule applied to the GPU's own P, barycentrics, primitive and
    instance (from the debug capture), bit for bit on every pixel."""
    w, h = 96, 64
    r, rest, mesh, case, im = _setup(rt, ctx, kind, motion, w, h)
    ctx.enable_debug_capture(True)
    try:
        r.dispatch(_frames(case, w, h, 1)[0])
        ph, rec = ctx.debug_array("primary_hits"), ctx.debug_array("primary_records")
    finally:
        ctx.enable_debug_capture(False)
    ctx.status()
    got, pos = r.aov(PREV).reshape(-1, 4), r.aov(POS).reshape(-1, 4)
    hit = pos[:, 3] == 1
    hits = np.zeros(int(hit.sum()), T.HIT_DTYPE)
    hits["bary"][:, 0], hits["bary"][:, 1] = ph["u"][hit], ph["v"][hit]
    hits["primitive_index"], hits["instance_index"] = ph["prim"][hit], rec[hit] // 2  # hit group i * 2 + ray type 0
    meshes = [mesh if k == 0 else rest.meshes[k] for k in (im or range(len(rest.meshes)))]
    prev = [rest.meshes[0].vertices["position"] if k == 0 else None for k in (im or range(len(rest.meshes)))]
    q = mr.apply_motion(pos[hit, :3], hits["instance_index"], r.motion)
    dw, applied, invalid = dr.displacement(hits, meshes, dr.descriptors(prev, r.prev_transforms))
    assert applied.mean() > 0.2 and not invalid.any()
    want = np.where(applied[:, None], q + dw, q)
    np.testing.assert_array_equal(got[hit, :3].view(np.uint32), want.view(np.uint32))
    assert not got[~hit].any()
    assert np.abs(got[hit, :3] - pos[hit, :3]).max() > 0.01  # the deformation moved something


@pytest.mark.parametrize("motion", [False, True])
@pytest.mark.parametrize("half", [False, True])
@pytest.mark.parametrize("kind,w,h,spp", [("cornell", 96, 96, 3), ("bunny", 120, 72, 2)])
def test_previous_position_aov_matches_the_oracle_restatement(kind, w, h, spp, half, motion, ctx, rt, orc):
    ctx.set_render_options(1, half)
    try:
        r, rest, mesh, case, im = _setup(rt, ctx, kind, motion, w, h)
        frames = _frames(case, w, h, spp)
        for f in frames:
            r.dispatch(f)
        ctx.status()
        got, pos = r.aov(PREV), r.aov(POS)
    finally:
        ctx.set_render_options(1, False)
    otlas, meshes, descs = _oracle(orc, rest, mesh, case, im)
    want = dr.render_previous_positions(orc, otlas, frames, w, h, r.motion, meshes, descs, half_targets=half)
    assert (want[..., 3] > 0).mean() > 0.1
    np.testing.assert_array_equal(got[..., 3], want[..., 3])
    np.testing.assert_array_equal(got[..., 3], pos[..., 3])
    scale = np.maximum(np.abs(want[..., :3]).max(axis=-1), 1e-6)
    rel = np.abs(got[..., :3].astype(np.float64) - want[..., :3]).max(axis=-1) / scale
    tol = 4e-6 if not half else 1e-3
    print(f"previous-position AOV: largest relative deviation {rel.max():.2e}, share within {tol:g}: {(rel <= tol).mean():.6f}")
    assert (rel <= tol).mean() >= 0.9999


def test_refitted_hits_equal_the_oracles_including_growth_past_the_old_bounds(ctx, rt, orc):
    """After set_vertices the primary hits are the oracle's on its refitted tree, also when the mesh grows past its old
    box: the rebuilt TLAS picks up the refitted BLAS's new box."""
    w, h = 128, 96
    rest = sheet_frame_case(0)
    r = _renderer(rt, ctx, rest, w, h, ())
    grown = rest.meshes[0].vertices.copy()
    grown["position"] = scenes.sheared_positions(grown["position"], (0.0, 0.6, 0.0))  # the top edge rises 0.6 above its box
    for mesh in (sheet_frame_case(3).meshes[0], scenes.Mesh(grown, rest.meshes[0].indices)):
        _deform(r, mesh)
        otlas, _, _ = _oracle(orc, rest, mesh, rest, None)
        rays = orc.primary_rays(scenes.make_frame(rest.setup, w, h, 0, 0), w, h)
        want = otlas.trace(rays, T.RAY_FLAG_CULL_BACK_FACING_TRIANGLES)
        got = ctx.trace(r.tlas, rays, T.RAY_FLAG_CULL_BACK_FACING_TRIANGLES)
        same = (got["primitive_index"] == want["primitive_index"]) & (got["instance_index"] == want["instance_index"])
        print(f"hit agreement {same.mean():.6f}")
        assert same.mean() >= 0.9999
        hit = same & (want["primitive_index"] != T.NO_HIT)
        np.testing.assert_allclose(got["t"][hit], want["t"][hit], rtol=1e-5)
    top = mesh.vertices["position"][:, 1].max()
    p = rays["origin"] + want["t"][:, None] * rays["direction"]
    above = (want["instance_index"] == 0) & (want["primitive_index"] != T.NO_HIT) & (p[:, 1] > 0.45 + 0.05)
    assert top > 1.0 and above.sum() > 100  # the sheet is hit above its old top edge (y = 0.45)


def _bind_and_dispatch(rt, ctx, r, frame, descs_ptr, n):
    """Renderer.dispatch with a caller-chosen deformation binding (and no motion)."""
    rt.check(rt.lib.rt_set_output(ctx.handle, 0, r.out[0].ptr, 16 * r.width))
    for name, k in rt._AOV_IDS.items():
        buf = r.aovs.get(name)
        rt.check(rt.lib.rt_set_aov_output(ctx.handle, k, buf.ptr if buf is not None else None, 16 * r.width if buf is not None else 0))
    rt.check(rt.lib.rt_set_tlas(ctx.handle, r.tlas.result.ptr))
    rt.check(rt.lib.rt_set_frame_constants(ctx.handle, C.byref(frame)))
    ctx.set_instance_motion(None, 0)
    ctx.set_adaptive_sampling(None, None)
    ctx.set_instance_deformation(descs_ptr, n)
    rt.check(rt.lib.rt_dispatch_rays(ctx.handle, r.program.handle, r.width, r.height, 1))


def _null_descs(ctx, n):
    d = (T.DeformationDesc * n)()
    for k in range(n):
        d[k].stride_bytes, d[k].vertex_count = 24, 1
    return ctx.upload(np.frombuffer(d, np.uint8))


@pytest.mark.parametrize("half", [False, True])
def test_equal_positions_null_and_unmatched_instances_give_the_unbound_aov(half, ctx, rt):
    """With the sheet deformed (room first, so the sheet is instance 1): a NULL binding, NULL pointers and n = 1 (the
    sheet's i = 1 >= n) all give the unbound AOV bit for bit; previous positions equal to the current ones give it by
    value (a -0 coordinate may come out +0)."""
    w, h = 80, 64
    rest, after = sheet_frame_case(2), sheet_frame_case(3)
    case = SceneCase(rest.meshes[::-1], transforms=rest.transforms, setup=rest.setup)
    ctx.set_render_options(1, half)
    try:
        r = _renderer(rt, ctx, case, w, h, (POS, PREV), deforming=(1,))
        r.set_vertices(1, after.meshes[0].vertices["position"], after.meshes[0].vertices["normal"])
        null = _null_descs(ctx, 2)
        aovs = {}
        for name, ptr, n in (("unbound", None, 0), ("null", null.ptr, 2), ("unmatched", r._deform_buf.ptr, 1),
                             ("bound", r._deform_buf.ptr, 2)):
            for b in (*r.out, *r.aovs.values()):
                b.zero()
            for f in _frames(after, w, h, 3):
                _bind_and_dispatch(rt, ctx, r, f, ptr, n)
            ctx.status()
            aovs[name] = r.aov(PREV)
        want = aovs["unbound"]
        np.testing.assert_array_equal(want.view(np.uint32), r.aov(POS).view(np.uint32))
        for name in ("null", "unmatched"):
            np.testing.assert_array_equal(aovs[name].view(np.uint32), want.view(np.uint32))
        assert np.abs(aovs["bound"] - want).max() > 0.01
        # equal positions: set the same vertices again, so the previous positions are the current ones
        r.set_vertices(1, after.meshes[0].vertices["position"], after.meshes[0].vertices["normal"])
        for b in (*r.out, *r.aovs.values()):
            b.zero()
        for f in _frames(after, w, h, 3):
            _bind_and_dispatch(rt, ctx, r, f, r._deform_buf.ptr, 2)
        ctx.status()
        np.testing.assert_array_equal(r.aov(PREV), want)
        ctx.set_instance_deformation(None, 0)
    finally:
        ctx.set_render_options(1, False)


def test_binding_leaves_everything_else_alone(ctx, rt):
    """Beauty, every other AOV and the ray counts are bit-identical with and without the deformation bound."""
    w, h, spp = 80, 56, 3
    aovs = T.AOV_NAMES + (POS, PREV)
    r, rest, mesh, case, im = _setup(rt, ctx, "cornell", True, w, h, aovs)
    outs = []
    for bound in (True, False):
        for b in (*r.out, *r.aovs.values()):
            b.zero()
        ctx.ray_counts(reset=True)
        saved = r._deform_buf
        if not bound:
            r._deform_buf = None  # dispatch() then unbinds the deformation
        try:
            for f in _frames(case, w, h, spp):
                r.dispatch(f)
        finally:
            r._deform_buf = saved
        ctx.status()
        c = ctx.ray_counts(reset=True)
        outs.append(([r.image(0)] + [r.aov(a) for a in T.AOV_NAMES + (POS,)], (c.primary, c.secondary, c.shadow), r.aov(PREV)))
    for a, b in zip(outs[0][0], outs[1][0]):
        np.testing.assert_array_equal(a.view(np.uint32), b.view(np.uint32))
    assert outs[0][1] == outs[1][1]
    assert np.abs(outs[0][2] - outs[1][2]).max() > 0.01


def test_a_deforming_renderers_first_frame_is_a_plain_renderers(ctx, rt):
    """BUILD_FLAG_ALLOW_UPDATE on the deforming meshes changes nothing a dispatch writes."""
    w, h = 80, 56
    rest = sheet_frame_case(0)
    imgs = []
    for deforming in ((), (0,)):
        r = _renderer(rt, ctx, rest, w, h, T.AOV_NAMES + (POS, PREV), deforming=deforming)
        r.dispatch(_frames(rest, w, h, 1)[0])
        ctx.status()
        imgs.append([r.image(0)] + [r.aov(a) for a in T.AOV_NAMES + (POS, PREV)])
    for a, b in zip(*imgs):
        np.testing.assert_array_equal(a.view(np.uint32), b.view(np.uint32))


def test_region_strip_stats_capture_and_adaptive_dispatches_equal_the_full_frame(ctx, rt):
    w, h = 96, 64
    rs = {mode: _setup(rt, ctx, "bunny", True, w, h, ("normal", POS, PREV), adaptive=(mode == "adaptive"))[0]
          for mode in ("full", "tiled", "strips", "stats", "capture", "adaptive")}
    case = _deformed("bunny")[2]
    for f in _frames(case, w, h, 2, seed=5):
        for mode, r in rs.items():
            if mode == "tiled":
                for region in ((0, 0, 40, 24), (40, 0, w, 24), (0, 24, w, h)):
                    r.dispatch(f, region=region)
            elif mode == "strips":
                for g in range(2):
                    r.dispatch(f, strips=(8, 2, g))
            else:
                ctx.enable_trace_stats(mode == "stats")
                ctx.enable_debug_capture(mode == "capture")
                try:
                    r.dispatch(f)
                finally:
                    ctx.enable_trace_stats(False)
                    ctx.enable_debug_capture(False)
    ctx.status()
    want = rs["full"].aov(PREV)
    assert np.abs(want - rs["full"].aov(POS)).max() > 0.01
    for mode, r in rs.items():
        np.testing.assert_array_equal(r.aov(PREV).view(np.uint32), want.view(np.uint32), err_msg=mode)


def _shear(frame, step=(0.08, 0.0, 0.0)):
    """sheared_box(frame)'s deformation as an instance transform: sliding_box(0)'s transform times the shear."""
    s = np.eye(4)
    s[:3, 1] += frame * np.asarray(step) / 0.3
    t = np.eye(4)
    t[:3] = np.asarray(scenes.sliding_box(0)[1][0], np.float64).reshape(3, 4)
    return (t @ s)[:3].reshape(12).astype(np.float32)


def test_sheared_box_by_vertices_agrees_with_the_same_shear_as_an_instance_transform(ctx, rt):
    """Independent of the restatement: the box sheared by set_vertices (frame 1 -> 2) and the rest box moved by the
    equivalent instance transforms (set_transforms, frame 1 -> 2) give the same previous positions, within 2e-5 (fp32
    rounding of two different evaluations of a point near 1 in size), on the box pixels where both hit the same point
    (within 1e-5)."""
    w, h = 96, 96
    meshes, transforms = scenes.sliding_box(0)
    base = SceneCase(meshes, transforms=transforms, setup=sheet_frame_case(0).setup)
    a = _renderer(rt, ctx, base, w, h, (POS, PREV))
    for f in (1, 2):
        m = scenes.sheared_box(f)[0][0]
        _deform(a, m)
    b = _renderer(rt, ctx, SceneCase(meshes, transforms=[_shear(1), transforms[1]], setup=base.setup), w, h, (POS, PREV), deforming=())
    b.set_transforms([_shear(2), transforms[1]])
    frame = _frames(base, w, h, 1)[0]
    for r in (a, b):
        r.dispatch(frame)
    ctx.status()
    pa, pb, qa, qb = a.aov(POS), b.aov(POS), a.aov(PREV), b.aov(PREV)
    box = (pa[..., 3] == 1) & (pb[..., 3] == 1) & (np.abs(qa - pa).max(axis=-1) > 0) & (np.abs(pa - pb).max(axis=-1) <= 1e-5)
    moved = (pa[..., 3] == 1) & (np.abs(qa - pa).max(axis=-1) > 0)
    assert box.sum() >= 200 and box.sum() >= 0.97 * moved.sum(), (box.sum(), moved.sum())
    err = np.abs(qa[box] - qb[box]).max()
    print(f"sheared box: {box.sum()} pixels, largest |P'_vertices - P'_transform| {err:.2e}")
    assert err <= 2e-5


def test_deforming_sequences_match_the_reference(ctx, rt):
    """Eight frames of the waving sheet through Renderer.denoise_temporal (rt_denoise_temporal_motion) against the
    restatement run on the GPU's own inputs: within 1e-5 relative RMSE."""
    w, h = 96, 96
    for p in (dict(iterations=0), dict(iterations=5)):
        r = _renderer(rt, ctx, sheet_frame_case(0), w, h, GUIDES)
        jit = scenes.jitter_sequence(3, 8, w, h)
        params = tdr.make_params(**_kw(p))
        prev_cam = prev_hist = None
        for k in range(8):
            m = sheet_frame_case(k).meshes[0]
            if k:
                _deform(r, m)
            f = scenes.make_frame(sheet_frame_case(0).setup, w, h, 100 + k, 0, jitter=jit[k])
            r.dispatch(f)
            inputs = (r.image(0), r.aov("albedo"), r.aov("normal"), r.aov(POS), r.aov(PREV))
            g = r.denoise_temporal(params)
            gh = r.temporal_history()
            ref, rh = mr.denoise_temporal_motion(*inputs, prev_cam, prev_hist, **_kw(p))
            _check_out(g, ref, False)
            _check_history(gh, rh, (None, None, inputs[2], inputs[3]))
            prev_cam, prev_hist = f.cameraParams, gh
        ctx.status()
        assert gh[0, ..., 3].max() > 4


def test_an_out_of_range_index_sets_the_status(ctx, rt):
    w, h = 48, 40
    r, rest, mesh, case, im = _setup(rt, ctx, "cornell", False, w, h)
    d = (T.DeformationDesc * 2)()
    d[0].previous_positions, d[0].stride_bytes, d[0].vertex_count = r._prev_vb[0].ptr, 24, 10  # most indices are >= 10
    d[0].object_to_previous_world[:] = scenes.IDENTITY_3X4.tolist()
    bad = ctx.upload(np.frombuffer(d, np.uint8))
    for buf in (bad, _null_descs(ctx, 2)):
        _bind_and_dispatch(rt, ctx, r, _frames(case, w, h, 1)[0], buf.ptr, 2)
        if buf is bad:
            assert rt.lib.rt_get_status(ctx.handle) == RT_ERR_INVALID_ARG
    ctx.status()  # the status does not stick
    d[0].vertex_count, d[0].stride_bytes = mesh.vertices.shape[0], 14  # a stride that is not a multiple of 4
    bad = ctx.upload(np.frombuffer(d, np.uint8))
    _bind_and_dispatch(rt, ctx, r, _frames(case, w, h, 1)[0], bad.ptr, 2)
    assert rt.lib.rt_get_status(ctx.handle) == RT_ERR_INVALID_ARG
    ctx.set_instance_deformation(None, 0)


def test_invalid_arguments_and_renderer_misuse(ctx, rt):
    assert C.sizeof(T.DeformationDesc) == 64
    d = ctx.alloc(64 * 4)
    for args in ((None, 1), (d.ptr, 0), (d.ptr + 4, 1), (d.ptr + 8, 1), (d.ptr, 1 << 24), (d.ptr, 0xFFFFFFFF)):
        assert rt.lib.rt_set_instance_deformation(ctx.handle, *args) == RT_ERR_INVALID_ARG, args
    assert rt.lib.rt_set_instance_deformation(None, d.ptr, 1) == RT_ERR_INVALID_ARG
    rt.check(rt.lib.rt_set_instance_deformation(ctx.handle, d.ptr + 16, (1 << 24) - 1))  # bound, never read
    rt.check(rt.lib.rt_set_instance_deformation(ctx.handle, None, 0))
    rest, w, h = sheet_frame_case(0), 16, 16
    with pytest.raises(ValueError):
        _renderer(rt, ctx, rest, w, h, (), deforming=(2,))
    r = _renderer(rt, ctx, rest, w, h, GUIDES)
    v = rest.meshes[0].vertices
    with pytest.raises(ValueError):  # the room is not deforming
        r.set_vertices(1, rest.meshes[1].vertices["position"], rest.meshes[1].vertices["normal"])
    with pytest.raises(ValueError):
        r.set_vertices(0, v["position"][:-1], v["normal"][:-1])
    with pytest.raises(ValueError):
        r.set_vertices(0, v["position"], v["normal"][:, :2])
    bad = v["position"].copy()
    bad[0, 0] = np.nan
    with pytest.raises(ValueError):
        r.set_vertices(0, bad, v["normal"])
    assert r._deform_buf is None
    with pytest.raises(ValueError):
        _renderer(rt, ctx, rest, w, h, (), deforming=()).set_vertices(0, v["position"], v["normal"])


def test_quality_on_gpu_renders(ctx, rt):
    w = h = 96
    frames = 16
    last = sheet_frame_case(frames - 1)
    ref = _renderer(rt, ctx, last, w, h, (), deforming=())
    for s in range(1024):
        ref.dispatch(scenes.make_frame(last.setup, w, h, s, s))
    r = _renderer(rt, ctx, sheet_frame_case(0), w, h, GUIDES)
    ins = []
    for f in range(frames):
        if f:
            _deform(r, sheet_frame_case(f).meshes[0])
        fr = scenes.make_frame(last.setup, w, h, 5000 + f, 0)
        r.dispatch(fr)
        ins.append((r.image(0), r.aov("albedo"), r.aov("normal"), r.aov(POS), r.aov(PREV), fr.cameraParams))
    ctx.status()
    # the sheet's pixels in the last frame: where the deformation moved the position
    sheet = (ins[-1][3][..., 3] == 1) & (np.abs(ins[-1][4] - ins[-1][3]).max(axis=-1) > 0)
    assert sheet.sum() >= 1000
    q = quality(ins, ref.image(0), sheet)
    print("GPU renders, sheet pixels: with history %.4f / %.4f; temporal pass with deformation / noisy %.4f, without %.4f; "
          "with the a-trous iterations %.4f / %.4f" % q)
    check_quality(q)
