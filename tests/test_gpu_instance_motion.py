"""GPU: the previous-position AOV (rt_set_instance_motion) and rt_denoise_temporal_motion against their CPU restatements
(tests/motion_reference.py), their exact properties, argument checks, and the history they keep on a moving instance."""
import ctypes as C

import numpy as np
import pytest

import motion_reference as mr
import temporal_denoise_reference as tdr
from dxrexperiments_b200 import scenes, types as T
from helpers import SceneCase, cornell_case
from test_gpu_temporal_denoise import PARAMS, _check_history, _check_out, _kw
from test_motion_reference import (box_ratio, check_quality, run_sequence, sliding_case)

pytestmark = pytest.mark.gpu
RT_ERR_INVALID_ARG = -1
POS, PREV = T.AOV_POSITION_NAME, T.AOV_PREVIOUS_POSITION_NAME
GUIDES = ("albedo", "normal", POS, PREV)


def _renderer(rt, ctx, case, w, h, aovs, instance_mesh=None):
    return rt.Renderer(ctx, case.meshes, case.transforms, case.materials, case.env, rt.PROGRESSIVE, w, h, aovs=aovs,
                       instance_mesh=instance_mesh)


def bunny_instances(seed):
    """Eight instances of one bunny mesh under scenes.random_rigid_transforms, seen from far enough to cover them."""
    tr = scenes.random_rigid_transforms(8, seed=seed, extent=25.0, scale=(0.5, 1.5))
    return SceneCase([scenes.bunny_scale(3)], transforms=list(tr), camera=scenes.Camera(eye=(0.0, 40.0, 110.0), at=(0.0, 0.0, 0.0)))


def _moved(kind):
    """(case before, case after, instance_mesh) of a moving scene."""
    if kind == "cornell":
        return sliding_case(2), sliding_case(3), None
    a, b = bunny_instances(10), bunny_instances(11)
    b.meshes = a.meshes
    return a, b, [0] * 8


def _frames(case, w, h, spp, seed=31):
    jit = scenes.jitter_sequence(seed, spp, w, h)
    return [scenes.make_frame(case.setup, w, h, s, s, jitter=jit[s]) for s in range(spp)]


def _oracle_tlas(orc, case, instance_mesh):
    blases = [orc.Blas.from_mesh(m) for m in case.meshes]
    im = instance_mesh or list(range(len(case.meshes)))
    return orc.Tlas([blases[k] for k in im], case.transforms)


# ---------------------------------------------------------------------------------------------------- the AOV
@pytest.mark.parametrize("half", [False, True])
@pytest.mark.parametrize("kind,w,h,spp", [("cornell", 96, 96, 3), ("bunny", 120, 72, 2)])
def test_previous_position_aov_matches_the_restatement(kind, w, h, spp, half, ctx, rt, orc):
    before, after, im = _moved(kind)
    ctx.set_render_options(1, half)
    try:
        r = _renderer(rt, ctx, before, w, h, (POS, PREV), im)
        r.set_transforms(after.transforms)
        frames = _frames(after, w, h, spp)
        for f in frames:
            r.dispatch(f)
        ctx.status()
        got, pos = r.aov(PREV), r.aov(POS)
    finally:
        ctx.set_render_options(1, False)
    motion = mr.motion_matrices(before.transforms, after.transforms)
    np.testing.assert_array_equal(r.motion, motion)
    otlas = _oracle_tlas(orc, after, im)
    want = mr.render_previous_positions(orc, otlas, frames, w, h, motion, half_targets=half)
    assert (want[..., 3] > 0).mean() > 0.1
    np.testing.assert_array_equal(got[..., 3], want[..., 3])
    np.testing.assert_array_equal(got[..., 3], pos[..., 3])
    scale = np.maximum(np.abs(want[..., :3]).max(axis=-1), 1e-6)
    rel = np.abs(got[..., :3].astype(np.float64) - want[..., :3]).max(axis=-1) / scale
    tol = 4e-6 if not half else 1e-3
    print(f"previous-position AOV: largest relative deviation {rel.max():.2e}, share within {tol:g}: {(rel <= tol).mean():.6f}")
    assert (rel <= tol).mean() >= 0.9999
    assert np.abs(got - pos).max() > 0.01  # the motion moved something


@pytest.mark.parametrize("kind", ["cornell", "bunny"])
def test_one_sample_is_the_motion_of_the_gpus_own_position_exactly(kind, ctx, rt, orc):
    """At one sample with fp32 targets the AOV is M_i * P of the GPU's own P, bit for bit, with i the oracle's instance."""
    w, h = 96, 64
    before, after, im = _moved(kind)
    r = _renderer(rt, ctx, before, w, h, (POS, PREV), im)
    r.set_transforms(after.transforms)
    f = _frames(after, w, h, 1)[0]
    r.dispatch(f)
    got, pos = r.aov(PREV), r.aov(POS)
    hits = _oracle_tlas(orc, after, im).trace(orc.primary_rays(f, w, h, float(tdr.JITTER_SCALE)), T.RAY_FLAG_CULL_BACK_FACING_TRIANGLES)
    inst = hits["instance_index"].reshape(h, w)
    want = mr.apply_motion(pos[..., :3], inst, r.motion)
    hit = pos[..., 3] == 1
    same = np.all(got[..., :3].view(np.uint32) == want.view(np.uint32), axis=-1)
    print(f"bit-identical pixels: {same[hit].mean():.6f}")
    assert same[hit].mean() >= 0.999
    assert not got[~hit].any()


def _bind_and_dispatch(rt, ctx, r, frame, motion_ptr, n):
    """Renderer.dispatch with a caller-chosen motion binding."""
    rt.check(rt.lib.rt_set_output(ctx.handle, 0, r.out[0].ptr, 16 * r.width))
    for name, k in rt._AOV_IDS.items():
        buf = r.aovs.get(name)
        rt.check(rt.lib.rt_set_aov_output(ctx.handle, k, buf.ptr if buf is not None else None, 16 * r.width if buf is not None else 0))
    rt.check(rt.lib.rt_set_tlas(ctx.handle, r.tlas.result.ptr))
    rt.check(rt.lib.rt_set_frame_constants(ctx.handle, C.byref(frame)))
    rt.check(rt.lib.rt_set_instance_motion(ctx.handle, motion_ptr, n))
    rt.check(rt.lib.rt_dispatch_rays(ctx.handle, r.program.handle, r.width, r.height, 1))


@pytest.mark.parametrize("half", [False, True])
def test_no_motion_identity_and_unmatched_instances_copy_the_position(half, ctx, rt):
    case, w, h = sliding_case(4), 80, 64
    ctx.set_render_options(1, half)
    try:
        eye = ctx.upload(np.tile(scenes.IDENTITY_3X4, 2))
        shift = ctx.upload(np.array([1, 0, 0, 0.5, 0, 1, 0, 0, 0, 0, 1, 0], np.float32))  # moves instance 0 only; the room is 1 >= n
        for ptr, n, exact in ((None, 0, True), (eye.ptr, 2, False), (shift.ptr, 1, None)):
            r = _renderer(rt, ctx, case, w, h, (POS, PREV))
            for f in _frames(case, w, h, 3):
                _bind_and_dispatch(rt, ctx, r, f, ptr, n)
            ctx.status()
            got, pos = r.aov(PREV), r.aov(POS)
            if exact is None:  # the box moved, every other pixel is a copy
                box = np.abs(got - pos).max(axis=-1) > 0
                assert box.sum() > 50
                np.testing.assert_array_equal(got[~box].view(np.uint32), pos[~box].view(np.uint32))
            elif exact:
                np.testing.assert_array_equal(got.view(np.uint32), pos.view(np.uint32))
            else:
                np.testing.assert_array_equal(got, pos)  # values: only a -0 coordinate may come out +0
        ctx.set_instance_motion(None, 0)
    finally:
        ctx.set_render_options(1, False)


def test_binding_previous_position_leaves_everything_else_alone(ctx, rt):
    before, after, _ = _moved("cornell")
    w, h, spp = 80, 56, 3
    outs = []
    for aovs in (T.AOV_NAMES + (POS,), T.AOV_NAMES + (POS, PREV)):
        r = _renderer(rt, ctx, before, w, h, aovs)
        r.set_transforms(after.transforms)
        ctx.ray_counts(reset=True)
        for f in _frames(after, w, h, spp):
            r.dispatch(f)
        ctx.status()
        c = ctx.ray_counts(reset=True)
        outs.append(([r.image(0)] + [r.aov(a) for a in T.AOV_NAMES + (POS,)], (c.primary, c.secondary, c.shadow)))
    for a, b in zip(outs[0][0], outs[1][0]):
        np.testing.assert_array_equal(a.view(np.uint32), b.view(np.uint32))
    assert outs[0][1] == outs[1][1]


def test_region_and_strip_dispatches_equal_the_full_frame(ctx, rt):
    before, after, im = _moved("bunny")
    w, h = 96, 64
    full, tiled, strips = (_renderer(rt, ctx, before, w, h, ("normal", POS, PREV), im) for _ in range(3))
    for r in (full, tiled, strips):
        r.set_transforms(after.transforms)
    for f in _frames(after, w, h, 2, seed=5):
        full.dispatch(f)
        for region in ((0, 0, 40, 24), (40, 0, w, 24), (0, 24, w, h)):
            tiled.dispatch(f, region=region)
        for g in range(2):
            strips.dispatch(f, strips=(8, 2, g))
    ctx.status()
    for r in (tiled, strips):
        np.testing.assert_array_equal(r.aov(PREV), full.aov(PREV))


def test_trace_stats_and_debug_capture_fill_the_instance_index(ctx, rt):
    before, after, im = _moved("bunny")
    w, h = 96, 64
    imgs = []
    for mode in ("plain", "stats", "capture"):
        r = _renderer(rt, ctx, before, w, h, (POS, PREV), im)
        r.set_transforms(after.transforms)
        if mode == "stats":
            ctx.enable_trace_stats(True)
        if mode == "capture":
            ctx.enable_debug_capture(True)
        try:
            for f in _frames(after, w, h, 2):
                r.dispatch(f)
            ctx.status()
        finally:
            ctx.enable_trace_stats(False)
            ctx.enable_debug_capture(False)
        imgs.append(r.aov(PREV))
    for g in imgs[1:]:
        np.testing.assert_array_equal(g.view(np.uint32), imgs[0].view(np.uint32))


# ---------------------------------------------------------------------------------------------------- rt_denoise_temporal_motion
def _sliding_renders(rt, ctx, w, h, frames, aovs=GUIDES, jitter_seed=3):
    r = _renderer(rt, ctx, sliding_case(0), w, h, aovs)
    jit = scenes.jitter_sequence(jitter_seed, frames, w, h)
    fs = [scenes.make_frame(sliding_case(0).setup, w, h, 100 + f, 0, jitter=jit[f]) for f in range(frames)]
    return r, fs


def test_previous_position_equal_to_position_is_the_temporal_pass(ctx, rt):
    w, h = 72, 56
    r, fs = _sliding_renders(rt, ctx, w, h, 4)
    prev_cam = hm = hp = None
    for k, f in enumerate(fs):
        if k:
            r.set_transforms(sliding_case(k).transforms)
        r.dispatch(f)
        ins = (r.image(0), r.aov("albedo"), r.aov("normal"), r.aov(POS))
        om, hm2 = ctx.denoise_temporal_motion(*ins, ins[3], prev_cam, hm)
        op, hp2 = ctx.denoise_temporal(*ins, prev_cam, hp)
        np.testing.assert_array_equal(om.view(np.uint32), op.view(np.uint32))
        np.testing.assert_array_equal(hm2.view(np.uint32), hp2.view(np.uint32))
        prev_cam, hm, hp = f.cameraParams, hm2, hp2


@pytest.mark.parametrize("half", [False, True])
def test_moving_sequences_match_the_reference(half, ctx, rt):
    w, h = 96, 96
    ctx.set_render_options(1, half)
    try:
        for p in PARAMS[:6]:
            r, fs = _sliding_renders(rt, ctx, w, h, 8)
            params = tdr.make_params(**_kw(p))
            prev_cam = prev_hist = None
            for k, f in enumerate(fs):
                if k:
                    r.set_transforms(sliding_case(k).transforms)
                r.dispatch(f)
                inputs = (r.image(0), r.aov("albedo"), r.aov("normal"), r.aov(POS), r.aov(PREV))
                before = ctx.launches()
                g = r.denoise_temporal(params)
                assert ctx.launches() - before == 2 + params.spatial.iterations
                gh = r.temporal_history()
                ref, rh = mr.denoise_temporal_motion(*inputs, prev_cam, prev_hist, **_kw(p), half_targets=half)
                _check_out(g, ref, half)
                _check_history(gh, rh, (None, None, inputs[2], inputs[3]))
                prev_cam, prev_hist = f.cameraParams, gh
            assert gh[0, ..., 3].max() > 4
    finally:
        ctx.set_render_options(1, False)


def test_inputs_and_prev_history_are_only_read(ctx, rt):
    w, h = 48, 40
    r, fs = _sliding_renders(rt, ctx, w, h, 2)
    r.dispatch(fs[0])
    r.denoise_temporal()
    r.set_transforms(sliding_case(1).transforms)
    r.dispatch(fs[1])
    ins = [r.out[0], r.aovs["albedo"], r.aovs["normal"], r.aovs[POS], r.aovs[PREV], r._temporal[0]]
    before = [b.download(np.float32) for b in ins]
    r.denoise_temporal()
    ctx.status()
    for b, want in zip(ins, before):
        np.testing.assert_array_equal(b.download(np.float32), want)


def test_invalid_arguments(ctx, rt):
    w, h = 16, 8
    img = 16 * w * h
    pool = ctx.alloc(16 * img + 64)  # beauty, albedo, normal, position, previous position, prev (4), history (4), tmp (2), out
    base = pool.ptr
    beauty, albedo, normal, position, prevpos, prev, hist, tmp, out = (base + k * img for k in (0, 1, 2, 3, 4, 5, 9, 13, 15))
    cam = T.CameraParams()
    cam.W[:] = (0.0, 0.0, -1.0, 0.0)
    good = tdr.make_params(iterations=2)

    def call(b=beauty, a=albedo, n=normal, ps=position, q=prevpos, pc=C.byref(cam), pv=prev, hs=hist, t=tmp, o=out, ww=w, hh=h,
             p=good, handle=ctx.handle):
        return rt.lib.rt_denoise_temporal_motion(handle, b, a, n, ps, q, pc, pv, hs, t, o, ww, hh, C.byref(p) if p is not None else None)

    rt.check(call())
    rt.check(call(pc=None, pv=None))
    rt.check(call(q=position))  # Q = P is allowed: both are only read
    ctx.status()
    before = ctx.launches()
    bad = [dict(handle=None), dict(b=None), dict(ps=None), dict(q=None), dict(p=None), dict(pc=None), dict(pv=None),
           dict(q=prevpos + 4), dict(q=prevpos + 8), dict(b=beauty + 4), dict(ww=0),
           dict(p=tdr.make_params(iterations=6)), dict(p=tdr.make_params(alpha_color=0.0)),
           dict(hs=prevpos), dict(hs=prevpos - 3 * img), dict(t=prevpos), dict(t=prevpos - img + 16), dict(o=prevpos),
           dict(o=prevpos + 16), dict(hs=beauty), dict(o=hist + img), dict(t=out - img)]
    for kw in bad:
        assert call(**kw) == RT_ERR_INVALID_ARG, kw
    assert ctx.launches() == before
    # rt_set_instance_motion
    m = ctx.alloc(48 * 4)
    for args in ((None, 1), (m.ptr, 0), (m.ptr + 4, 1), (m.ptr + 8, 1), (m.ptr, 1 << 24), (m.ptr, 0xFFFFFFFF)):
        assert rt.lib.rt_set_instance_motion(ctx.handle, *args) == RT_ERR_INVALID_ARG, args
    assert rt.lib.rt_set_instance_motion(None, m.ptr, 1) == RT_ERR_INVALID_ARG
    rt.check(rt.lib.rt_set_instance_motion(ctx.handle, m.ptr, (1 << 24) - 1))  # bound, never read: no dispatch follows
    rt.check(rt.lib.rt_set_instance_motion(ctx.handle, None, 0))
    # the previous-position AOV follows rt_set_aov_output's rules: not for a realtime program, not in the AO view
    case, w, h = cornell_case(), 16, 16
    buf = ctx.alloc(16 * w * h)
    rtr = rt.Renderer(ctx, case.meshes, case.transforms, case.materials, case.env, rt.REALTIME, w, h)
    f = scenes.make_frame(case.setup, w, h, 0, 0)
    rt.check(rt.lib.rt_set_output(ctx.handle, 0, rtr.out[0].ptr, 16 * w))
    rt.check(rt.lib.rt_set_output(ctx.handle, 1, rtr.out[1].ptr, 16 * w))
    for k in range(T.AOV_COUNT):
        rt.check(rt.lib.rt_set_aov_output(ctx.handle, k, None, 0))
    rt.check(rt.lib.rt_set_aov_output(ctx.handle, T.AOV_PREVIOUS_POSITION, buf.ptr, 16 * w))
    rt.check(rt.lib.rt_set_tlas(ctx.handle, rtr.tlas.result.ptr))
    rt.check(rt.lib.rt_set_frame_constants(ctx.handle, C.byref(f)))
    assert rt.lib.rt_dispatch_rays(ctx.handle, rtr.program.handle, w, h, 1) == RT_ERR_INVALID_ARG
    prog = _renderer(rt, ctx, case, w, h, ())
    rt.check(rt.lib.rt_set_output(ctx.handle, 0, prog.out[0].ptr, 16 * w))
    ao = scenes.make_frame(case.setup, w, h, 0, 0)
    ao.options.showAmbientOcclusionOnly = 1
    rt.check(rt.lib.rt_set_frame_constants(ctx.handle, C.byref(ao)))
    assert rt.lib.rt_dispatch_rays(ctx.handle, prog.program.handle, w, h, 1) == RT_ERR_INVALID_ARG
    assert rt.lib.rt_set_aov_output(ctx.handle, T.AOV_COUNT, buf.ptr, 16 * w) == RT_ERR_INVALID_ARG
    rt.check(rt.lib.rt_set_aov_output(ctx.handle, T.AOV_PREVIOUS_POSITION, None, 0))


def test_renderer_misuse_raises_value_error(ctx, rt):
    case, w, h = sliding_case(0), 16, 16
    r = _renderer(rt, ctx, case, w, h, GUIDES)
    assert r.motion is None
    with pytest.raises(ValueError):
        r.set_transforms(case.transforms[:1])
    with pytest.raises(ValueError):
        r.set_transforms([np.zeros(12, np.float32), scenes.IDENTITY_3X4])  # not invertible
    with pytest.raises(ValueError):
        r.set_transforms([np.full(12, np.nan, np.float32), scenes.IDENTITY_3X4])
    assert r.motion is None
    with pytest.raises(ValueError):  # the motion variant still needs the position AOV
        r2 = _renderer(rt, ctx, case, w, h, ("albedo", "normal", PREV))
        r2.dispatch(scenes.make_frame(case.setup, w, h, 0, 0))
        r2.denoise_temporal()
    r.set_transforms(sliding_case(1).transforms)
    np.testing.assert_array_equal(r.motion, mr.motion_matrices(case.transforms, sliding_case(1).transforms))


def test_quality_on_gpu_renders(ctx, rt):
    w = h = 96
    frames = 16
    last = sliding_case(frames - 1)
    ref = _renderer(rt, ctx, last, w, h, ())
    for s in range(1024):
        ref.dispatch(scenes.make_frame(last.setup, w, h, s, s))
    r = _renderer(rt, ctx, sliding_case(0), w, h, GUIDES)
    ins = []
    for f in range(frames):
        if f:
            r.set_transforms(sliding_case(f).transforms)
        fr = scenes.make_frame(last.setup, w, h, 5000 + f, 0)
        r.dispatch(fr)
        ins.append((r.image(0), r.aov("albedo"), r.aov("normal"), r.aov(POS), r.aov(PREV), fr.cameraParams))
    ctx.status()
    truth = ref.image(0)
    # the box's pixels in the last frame: where the instance motion moved the position
    box = (ins[-1][3][..., 3] == 1) & (np.abs(ins[-1][4] - ins[-1][3]).max(axis=-1) > 0)
    assert box.sum() >= 200
    noisy = ins[-1][0]
    om, hm, op, hp = run_sequence(ins, 0)
    m, pl = box_ratio(om, noisy, truth, box), box_ratio(op, noisy, truth, box)
    share = (hm[0, ..., 3][box] > 1).mean()
    fm = box_ratio(run_sequence(ins, 5)[0], noisy, truth, box)
    print(f"GPU renders, box pixels: temporal pass with motion / noisy {m:.4f}, without {pl:.4f}; with history {share:.4f}; "
          f"with the a-trous iterations {fm:.4f}")
    check_quality(m, pl, share, fm)
    # the GPU's own filter on the same frames gives the same ratio as the restatement run on its inputs
    r2 = _renderer(rt, ctx, sliding_case(0), w, h, GUIDES)
    for f in range(frames):
        if f:
            r2.set_transforms(sliding_case(f).transforms)
        r2.dispatch(scenes.make_frame(last.setup, w, h, 5000 + f, 0))
        g = r2.denoise_temporal(tdr.make_params(iterations=0))
    assert abs(box_ratio(g, noisy, truth, box) - m) <= 1e-3 * m
