"""GPU: the position AOV and rt_denoise_temporal against their CPU restatements (tests/temporal_denoise_reference.py), their
exact properties, argument checks, and the temporal filter's quality on a moving camera."""
import ctypes as C
import dataclasses

import numpy as np
import pytest

import aov_reference
import temporal_denoise_reference as tdr
from conftest import rel_rmse
from dxrexperiments_b200 import scenes, types as T
from helpers import bunny_case, cornell_case, two_material_case
from test_temporal_denoise_reference import check_quality, quality_ratios

pytestmark = pytest.mark.gpu
RT_ERR_INVALID_ARG = -1
POS = T.AOV_POSITION_NAME
GUIDES = ("albedo", "normal", POS)

PARAMS = [dict(iterations=i) for i in range(6)] + [
    dict(iterations=3, normal_exponent_log2=4, sigma_luminance=2.0, sigma_albedo=0.0, alpha_color=0.5, alpha_moments=0.1,
         normal_cos=0.5, position_tolerance=0.05),
    dict(iterations=2, normal_exponent_log2=0, sigma_luminance=8.0, sigma_albedo=0.5, alpha_color=1.0, alpha_moments=1.0,
         normal_cos=-1.0, position_tolerance=0.0),
    dict(iterations=5, normal_exponent_log2=8, sigma_luminance=1.0, sigma_albedo=0.3, alpha_color=0.05, alpha_moments=0.3,
         normal_cos=0.99, position_tolerance=0.1)]


def _kw(p):
    return dict(tdr.default_params(), **p)


def _renderer(rt, ctx, case, w, h, aovs):
    return rt.Renderer(ctx, case.meshes, case.transforms, case.materials, case.env, rt.PROGRESSIVE, w, h, aovs=aovs)


def _accumulate(r, case, w, h, spp, seed=31):
    jit = scenes.jitter_sequence(seed, spp, w, h)
    frames = [scenes.make_frame(case.setup, w, h, s, s, jitter=jit[s]) for s in range(spp)]
    for f in frames:
        r.dispatch(f)
    return frames


# ---------------------------------------------------------------------------------------------------- position AOV
@pytest.mark.parametrize("half", [False, True])
@pytest.mark.parametrize("case_fn,w,h,spp", [(cornell_case, 96, 96, 4), (bunny_case, 120, 72, 2), (two_material_case, 104, 64, 3)])
def test_position_aov_matches_the_oracle(case_fn, w, h, spp, half, ctx, rt, orc):
    case = case_fn()
    ctx.set_render_options(1, half)
    try:
        r = _renderer(rt, ctx, case, w, h, (POS,))
        frames = _accumulate(r, case, w, h, spp)
        ctx.status()
        got = r.aov(POS)
    finally:
        ctx.set_render_options(1, False)
    otlas, _ = case.oracle(orc)
    want = tdr.render_positions(orc, otlas, frames, w, h, half_targets=half)
    np.testing.assert_array_equal(got[..., 3], want[..., 3])  # coverage
    scale = np.maximum(np.abs(want[..., :3]).max(axis=-1), 1e-6)
    rel = np.abs(got[..., :3].astype(np.float64) - want[..., :3]).max(axis=-1) / scale
    tol = 1e-6 if not half else 1e-3  # fp16 targets: a running mean one fp16 rounding apart
    print(f"position AOV: largest relative deviation {rel.max():.2e}, share within {tol:g}: {(rel <= tol).mean():.6f}")
    assert (rel <= tol).mean() >= 0.9999


def test_position_aov_on_the_closed_form_plane(ctx, rt):
    w, h = 96, 64
    case, on, off = aov_reference.plane_case(w, h)
    r = _renderer(rt, ctx, case, w, h, (POS,))
    r.dispatch(scenes.make_frame(case.setup, w, h, 0, 0))
    ctx.status()
    p = r.aov(POS)
    assert on.sum() > 0.2 * on.size and off.sum() > 0.2 * off.size
    assert np.abs(p[on][:, 2]).max() <= 1e-6
    assert np.all(p[on][:, 3] == 1.0) and np.all(np.abs(p[on][:, :2]) <= 1.0)
    assert not p[off].any()


def test_binding_position_leaves_everything_else_alone(ctx, rt):
    case, w, h, spp = cornell_case(), 80, 56, 3
    outs = []
    for aovs in (T.AOV_NAMES, T.AOV_NAMES + (POS,)):
        r = _renderer(rt, ctx, case, w, h, aovs)
        ctx.ray_counts(reset=True)
        _accumulate(r, case, w, h, spp)
        ctx.status()
        c = ctx.ray_counts(reset=True)
        outs.append(([r.image(0)] + [r.aov(a) for a in T.AOV_NAMES], (c.primary, c.secondary, c.shadow)))
    for a, b in zip(outs[0][0], outs[1][0]):
        np.testing.assert_array_equal(a, b)
    assert outs[0][1] == outs[1][1]


def test_position_region_and_strip_dispatches_equal_the_full_frame(ctx, rt):
    case, w, h = two_material_case(), 96, 64
    jit = scenes.jitter_sequence(5, 2, w, h)
    frames = [scenes.make_frame(case.setup, w, h, s, s, jitter=jit[s]) for s in range(2)]
    full, tiled, strips = (_renderer(rt, ctx, case, w, h, ("normal", POS)) for _ in range(3))
    for f in frames:
        full.dispatch(f)
        for region in ((0, 0, 40, 24), (40, 0, w, 24), (0, 24, w, h)):
            tiled.dispatch(f, region=region)
        for g in range(2):
            strips.dispatch(f, strips=(8, 2, g))
    ctx.status()
    for r in (tiled, strips):
        np.testing.assert_array_equal(r.aov(POS), full.aov(POS))


# ---------------------------------------------------------------------------------------------------- rt_denoise_temporal
def _check_out(g, ref, half):
    """fp32 targets: relative RMSE <= 1e-5.  fp16 targets: every value equals the restatement's or is one fp16 ulp from it
    (an ulp of expf can cross an fp16 rounding boundary), on at most 0.2 % of the values or one value, whichever is more."""
    assert np.isfinite(g).all()
    if not half:
        assert rel_rmse(g, ref) <= 1e-5, rel_rmse(g, ref)
        return
    g16, r16 = g.astype(np.float16), ref.astype(np.float16)
    np.testing.assert_array_equal(g16.astype(np.float32), g)
    ulp = np.maximum(np.abs(np.spacing(g16)), np.abs(np.spacing(r16))).astype(np.float32)
    differ = g != ref
    assert np.all(np.abs(g - ref)[differ] <= ulp[differ])
    assert differ.sum() <= max(1.0, 2e-3 * differ.size), differ.sum()


def _check_history(g, ref, inputs):
    np.testing.assert_array_equal(g[2], inputs[2])
    np.testing.assert_array_equal(g[3], inputs[3])
    assert rel_rmse(g[0, ..., :3], ref[0, ..., :3]) <= 1e-5
    assert rel_rmse(g[1], ref[1]) <= 1e-5
    assert (g[0, ..., 3] == ref[0, ..., 3]).mean() >= 0.999


def _orbit(case, w, h, frames=8, degrees=0.5, seed=3):
    jit = scenes.jitter_sequence(seed, frames, w, h)
    return tdr.orbit_frames(case.setup, w, h, frames, degrees, first_sample=100, jitter=jit)


@pytest.mark.parametrize("half", [False, True])
@pytest.mark.parametrize("case_fn,w,h", [(cornell_case, 96, 96), (bunny_case, 120, 72), (cornell_case, 33, 17), (cornell_case, 3, 2),
                                         (cornell_case, 1, 1), (two_material_case, 2, 40)])
def test_orbit_matches_the_reference(case_fn, w, h, half, ctx, rt):
    case = case_fn()
    ctx.set_render_options(1, half)
    try:
        r = _renderer(rt, ctx, case, w, h, GUIDES)
        frames = _orbit(case, w, h)
        for p in PARAMS if (w, h) in ((96, 96), (33, 17)) else PARAMS[-3:]:
            params = tdr.make_params(**_kw(p))
            r.reset_temporal()
            prev_cam = prev_hist = None
            for f in frames:
                r.dispatch(f)
                inputs = (r.image(0), r.aov("albedo"), r.aov("normal"), r.aov(POS))
                before = ctx.launches()
                g = r.denoise_temporal(params)
                assert ctx.launches() - before == 2 + params.spatial.iterations
                gh = r.temporal_history()
                ref, rh = tdr.denoise_temporal(*inputs, prev_cam, prev_hist, **_kw(p), half_targets=half)
                _check_out(g, ref, half)
                _check_history(gh, rh, (None, None, inputs[2], inputs[3]))
                prev_cam, prev_hist = f.cameraParams, gh  # the GPU's own history, so that each step is checked alone
            if _kw(p)["position_tolerance"] > 0 and min(w, h) >= 16:  # (in a 2-pixel-wide image a pixel is half the view)
                assert gh[0, ..., 3].max() > 1  # the orbit kept some history
    finally:
        ctx.set_render_options(1, False)


@pytest.mark.parametrize("half", [False, True])
@pytest.mark.parametrize("iterations", range(6))
def test_without_history_equals_the_spatial_denoiser(iterations, half, ctx, rt):
    case, w, h = cornell_case(), 72, 56
    ctx.set_render_options(1, half)
    try:
        r = _renderer(rt, ctx, case, w, h, GUIDES)
        r.dispatch(scenes.make_frame(case.setup, w, h, 7, 0, jitter=(0.01, -0.02)))
        ins = (r.image(0), r.aov("albedo"), r.aov("normal"), r.aov(POS))
        p = tdr.make_params(iterations=iterations)
        out, hist = ctx.denoise_temporal(*ins, params=p)
        np.testing.assert_array_equal(out, ctx.denoise_progressive(ins[0], ins[1], ins[2], p.spatial))
        np.testing.assert_array_equal(out, r.denoise_temporal(p))
        np.testing.assert_array_equal(hist[0, ..., 3], 1)
    finally:
        ctx.set_render_options(1, False)


def test_inputs_and_prev_history_are_only_read(ctx, rt):
    case, w, h = cornell_case(), 48, 40
    r = _renderer(rt, ctx, case, w, h, GUIDES)
    frames = _orbit(case, w, h, frames=2)
    r.dispatch(frames[0])
    r.denoise_temporal()
    r.dispatch(frames[1])
    prev = r._temporal[0]
    ins = [r.out[0], r.aovs["albedo"], r.aovs["normal"], r.aovs[POS], prev]
    before = [b.download(np.float32) for b in ins]
    r.denoise_temporal()
    ctx.status()
    for b, want in zip(ins, before):
        np.testing.assert_array_equal(b.download(np.float32), want)


def test_invalid_arguments(ctx, rt):
    w, h = 16, 8
    img = 16 * w * h
    pool = ctx.alloc(15 * img + 64)  # beauty, albedo, normal, position, prev (4), history (4), tmp (2), out, slack
    base = pool.ptr
    beauty, albedo, normal, position, prev, hist, tmp, out = (base + k * img for k in (0, 1, 2, 3, 4, 8, 12, 14))
    cam = T.CameraParams()
    cam.W[:] = (0.0, 0.0, -1.0, 0.0)
    good = tdr.make_params(iterations=2)

    def params(**kw):
        return tdr.make_params(**dict(tdr.params_dict(good), **kw))

    def call(b=beauty, a=albedo, n=normal, ps=position, pc=C.byref(cam), pv=prev, hs=hist, t=tmp, o=out, ww=w, hh=h, p=good,
             handle=ctx.handle):
        return rt.lib.rt_denoise_temporal(handle, b, a, n, ps, pc, pv, hs, t, o, ww, hh, C.byref(p) if p is not None else None)

    rt.check(call())  # the eight images touch end to end, which is not an overlap
    rt.check(call(pc=None, pv=None))
    ctx.status()
    before = ctx.launches()
    nan, inf = float("nan"), float("inf")
    bad = [dict(handle=None), dict(b=None), dict(a=None), dict(n=None), dict(ps=None), dict(hs=None), dict(t=None), dict(o=None),
           dict(p=None), dict(pc=None), dict(pv=None),
           dict(b=beauty + 4), dict(a=albedo + 8), dict(n=normal + 12), dict(ps=position + 4), dict(pv=prev + 8), dict(hs=hist + 4),
           dict(t=tmp + 4), dict(o=out + 8), dict(ww=0), dict(hh=0),
           dict(p=params(iterations=6)), dict(p=params(normal_exponent_log2=9)), dict(p=params(sigma_luminance=0.0)),
           dict(p=params(sigma_luminance=nan)), dict(p=params(sigma_albedo=-0.1)),
           dict(p=params(alpha_color=0.0)), dict(p=params(alpha_color=1.5)), dict(p=params(alpha_color=nan)),
           dict(p=params(alpha_moments=0.0)), dict(p=params(alpha_moments=-1.0)), dict(p=params(alpha_moments=nan)),
           dict(p=params(normal_cos=1.01)), dict(p=params(normal_cos=-1.5)), dict(p=params(normal_cos=nan)),
           dict(p=params(position_tolerance=-0.01)), dict(p=params(position_tolerance=inf)), dict(p=params(position_tolerance=nan)),
           # history, tmp and out against the inputs, prev_history and each other
           dict(hs=beauty), dict(hs=position + 16), dict(hs=prev + 3 * img), dict(hs=tmp - 4 * img + 16), dict(hs=out),
           dict(t=albedo), dict(t=prev + 16), dict(t=hist + 2 * img), dict(t=out - img),
           dict(o=normal), dict(o=prev + 3 * img + 16), dict(o=hist + img), dict(o=tmp + img)]
    for kw in bad:
        assert call(**kw) == RT_ERR_INVALID_ARG, kw
    assert ctx.launches() == before


def test_renderer_denoise_temporal_needs_its_guides_and_one_sample_frames(ctx, rt):
    case, w, h = cornell_case(), 16, 16
    for aovs in ((), ("albedo", "normal"), ("albedo", POS), ("normal", POS)):
        r = _renderer(rt, ctx, case, w, h, aovs)
        r.dispatch(scenes.make_frame(case.setup, w, h, 0, 0))
        with pytest.raises(ValueError):
            r.denoise_temporal()
    r = _renderer(rt, ctx, case, w, h, GUIDES)
    with pytest.raises(ValueError):  # nothing dispatched yet
        r.denoise_temporal()
    r.dispatch(scenes.make_frame(case.setup, w, h, 0, 0))
    r.dispatch(scenes.make_frame(case.setup, w, h, 1, 1))  # accumulating
    with pytest.raises(ValueError):
        r.denoise_temporal()
    with pytest.raises(ValueError):
        rt.Renderer(ctx, case.meshes, case.transforms, case.materials, case.env, rt.PROGRESSIVE, w, h, aovs=("depth",))


def test_quality_on_gpu_renders(ctx, rt):
    w = h = 96
    case = cornell_case()
    frames = tdr.orbit_frames(case.setup, w, h, 16, 0.5, first_sample=5000)
    last = dataclasses.replace(case.setup, camera=scenes.orbit(case.setup.camera, 15 * 0.5))
    ref = _renderer(rt, ctx, case, w, h, ())
    for s in range(1024):
        ref.dispatch(scenes.make_frame(last, w, h, s, s))
    r = _renderer(rt, ctx, case, w, h, GUIDES)
    for f in frames:
        r.dispatch(f)
        out = r.denoise_temporal()
    ctx.status()
    t, s = quality_ratios(out, r.denoise(), r.image(0), ref.image(0))
    print(f"temporal / noisy {t:.4f}, spatial / noisy {s:.4f} (rel RMSE against 1024 spp, GPU renders)")
    check_quality(t, s)
