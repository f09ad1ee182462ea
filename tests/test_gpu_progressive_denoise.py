"""GPU: rt_denoise_progressive against its CPU restatement (tests/progressive_denoise_reference.py), its exact properties,
its argument checks and its quality on GPU renders."""
import ctypes as C

import numpy as np
import pytest

import progressive_denoise_reference as pdr
from conftest import rel_rmse
from dxrexperiments_b200 import scenes, types as T
from helpers import bunny_case, cornell_case, two_material_case
from test_progressive_denoise_reference import QUALITY_RATIO_BOUND, cornell_quality_frames

pytestmark = pytest.mark.gpu
RT_ERR_INVALID_ARG = -1

PARAMS = [(i, 7, 4.0, 0.1) for i in range(6)] + [(3, 4, 2.0, 0.0), (2, 0, 8.0, 0.5), (5, 8, 1.0, 0.3), (4, 2, 0.5, 2.0)]


def _params(p):
    return T.ProgressiveDenoiseParams(*p)


def _renderer(rt, ctx, case, w, h, spp, aovs=("albedo", "normal"), seed=31):
    r = rt.Renderer(ctx, case.meshes, case.transforms, case.materials, case.env, rt.PROGRESSIVE, w, h, aovs=aovs)
    jit = scenes.jitter_sequence(seed, spp, w, h)
    for s in range(spp):
        r.dispatch(scenes.make_frame(case.setup, w, h, s, s, jitter=jit[s]))
    ctx.status()
    return r


def _check_against_reference(g, inputs, p, half):
    """fp32 targets: relative RMSE <= 1e-5 (measured <= 1e-7).  fp16 targets: an ulp of expf in fp32 now and then moves a value
    across an fp16 rounding boundary, a step of one fp16 ulp (~1e-3 relative), so a few such steps alone can exceed 1e-5 on a
    small frame; there every value must equal the restatement's or be one fp16 ulp from it, on at most 0.2 % of the values."""
    ref = pdr.denoise(*inputs, *p, half_targets=half)
    assert np.isfinite(g).all()
    err = rel_rmse(g, ref)
    dev = float(np.max(np.abs(g.astype(np.float64) - ref) / np.maximum(np.abs(ref), 1e-6)))
    print(f"params {p} half {half}: rel RMSE {err:.2e}, largest per-pixel relative deviation {dev:.2e}")
    if not half:
        assert err <= 1e-5, (p, err)
        return
    g16, r16 = g.astype(np.float16), ref.astype(np.float16)
    np.testing.assert_array_equal(g16.astype(np.float32), g)  # the stores are fp16 values
    ulp = np.maximum(np.abs(np.spacing(g16)), np.abs(np.spacing(r16))).astype(np.float32)
    differ = g != ref
    assert np.all(np.abs(g - ref)[differ] <= ulp[differ]), p
    assert differ.mean() <= 2e-3, (p, differ.mean())


@pytest.mark.parametrize("half", [False, True])
@pytest.mark.parametrize("case_fn,w,h,spp", [(cornell_case, 96, 96, 4), (bunny_case, 120, 72, 2), (two_material_case, 104, 64, 3),
                                             (two_material_case, 640, 512, 1)])
def test_matches_reference_on_renders(case_fn, w, h, spp, half, ctx, rt):
    ctx.set_render_options(1, half)
    try:
        r = _renderer(rt, ctx, case_fn(), w, h, spp)
        inputs = (r.image(0), r.aov("albedo"), r.aov("normal"))
        for p in PARAMS:
            before = ctx.launches()
            g = r.denoise(_params(p))
            assert ctx.launches() - before == 1 + p[0]
            _check_against_reference(g, inputs, p, half)
        # the inputs are only read
        for got, want in zip((r.image(0), r.aov("albedo"), r.aov("normal")), inputs):
            np.testing.assert_array_equal(got, want)
    finally:
        ctx.set_render_options(1, False)


@pytest.mark.parametrize("w,h", [(1, 1), (3, 2), (33, 17), (2, 40)])
@pytest.mark.parametrize("half", [False, True])
def test_matches_reference_on_ragged_sizes(w, h, half, ctx, rt):
    inputs = pdr.synthetic_inputs(w, h, 11 + w * h, sky_fraction=0.1)
    ctx.set_render_options(1, half)
    try:
        for p in PARAMS:
            _check_against_reference(ctx.denoise_progressive(*inputs, _params(p)), inputs, p, half)
    finally:
        ctx.set_render_options(1, False)


def test_zero_iterations_return_the_beauty_frame(ctx, rt):
    b, a, n = pdr.synthetic_inputs(37, 23, 1)
    out = ctx.denoise_progressive(b, a, n, _params((0, 7, 4.0, 0.1)))
    np.testing.assert_array_equal(out[..., :3], b[..., :3])
    assert np.all(out[..., 3] == 1.0)


@pytest.mark.parametrize("iterations", [1, 3, 5])
def test_constant_image_is_a_fixed_point(iterations, ctx, rt):
    h, w = 40, 52
    b = np.tile(np.array([0.7, 0.3, 0.2, 1.0], np.float32), (h, w, 1))
    a = np.tile(np.array([0.5, 0.4, 0.3, 1.0], np.float32), (h, w, 1))
    n = np.tile(np.array([0.0, 0.6, 0.8, 1.0], np.float32), (h, w, 1))
    out = ctx.denoise_progressive(b, a, n, _params((iterations, 7, 4.0, 0.1)))
    np.testing.assert_allclose(out, b, rtol=1e-6, atol=0)


@pytest.mark.parametrize("iterations", [0, 2, 5])
def test_sky_is_copied_and_never_read(iterations, ctx, rt):
    b, a, n = pdr.synthetic_inputs(45, 31, 2)
    sky = n[..., 3] == 0
    p = _params((iterations, 7, 4.0, 0.1))
    out = ctx.denoise_progressive(b, a, n, p)
    np.testing.assert_array_equal(out[sky][:, :3], b[sky][:, :3])
    b2, a2 = b.copy(), a.copy()
    b2[sky] = np.float32(1e4)
    a2[sky] = np.float32(7.0)
    np.testing.assert_array_equal(ctx.denoise_progressive(b2, a2, n, p)[~sky], out[~sky])


@pytest.mark.parametrize("iterations", range(6))
def test_perpendicular_halves_do_not_mix(iterations, ctx, rt):
    w, h = 48, 20
    b, a, n = pdr.halves_inputs(w, h, 3)
    p = _params((iterations, 7, 4.0, 0.1))
    out = ctx.denoise_progressive(b, a, n, p)
    b2 = b.copy()
    b2[:, w // 2:, :3] = np.float32(50.0) * b2[:, w // 2:, :3] + np.float32(3.0)
    np.testing.assert_array_equal(ctx.denoise_progressive(b2, a, n, p)[:, :w // 2], out[:, :w // 2])


def test_quality_on_gpu_renders(ctx, rt):
    w = h = 96
    case, ref_frames = cornell_quality_frames(w, h, 1024, 0)
    _, frames = cornell_quality_frames(w, h, 4, 5000)
    ref = rt.Renderer(ctx, case.meshes, case.transforms, case.materials, case.env, rt.PROGRESSIVE, w, h)
    for f in ref_frames:
        ref.dispatch(f)
    r = rt.Renderer(ctx, case.meshes, case.transforms, case.materials, case.env, rt.PROGRESSIVE, w, h, aovs=("albedo", "normal"))
    for f in frames:
        r.dispatch(f)
    ctx.status()
    truth = ref.image(0)[..., :3]
    ratio = rel_rmse(r.denoise()[..., :3], truth) / rel_rmse(r.image(0)[..., :3], truth)
    print(f"denoised / noisy rel RMSE against 1024 spp on the GPU: {ratio:.4f}")
    assert ratio <= QUALITY_RATIO_BOUND, ratio


def test_invalid_arguments(ctx, rt):
    w, h = 16, 8
    img = 16 * w * h
    pool = ctx.alloc(8 * img + 64)  # beauty, albedo, normal, tmp (2 images), out, slack
    base = pool.ptr
    beauty, albedo, normal, tmp, out = base, base + img, base + 2 * img, base + 3 * img, base + 5 * img
    good = _params((2, 7, 4.0, 0.1))

    def call(b=beauty, a=albedo, n=normal, t=tmp, o=out, ww=w, hh=h, p=good, handle=ctx.handle):
        return rt.lib.rt_denoise_progressive(handle, b, a, n, t, o, ww, hh, C.byref(p) if p is not None else None)

    rt.check(call())  # the five images touch end to end, which is not an overlap
    ctx.status()
    before = ctx.launches()
    bad = [dict(handle=None), dict(b=None), dict(a=None), dict(n=None), dict(t=None), dict(o=None), dict(p=None),
           dict(b=beauty + 4), dict(a=albedo + 8), dict(n=normal + 12), dict(t=tmp + 4), dict(o=out + 8),
           dict(ww=0), dict(hh=0),
           dict(p=_params((6, 7, 4.0, 0.1))), dict(p=_params((2, 9, 4.0, 0.1))), dict(p=_params((2, 7, 0.0, 0.1))),
           dict(p=_params((2, 7, -1.0, 0.1))), dict(p=_params((2, 7, float("nan"), 0.1))), dict(p=_params((2, 7, float("inf"), 0.1))),
           dict(p=_params((2, 7, 4.0, -0.1))), dict(p=_params((2, 7, 4.0, float("nan")))),
           dict(o=beauty), dict(o=albedo + 16 * w), dict(o=normal - 16), dict(o=tmp + img), dict(o=tmp - img + 16),
           dict(t=beauty), dict(t=albedo), dict(t=albedo + 16), dict(t=out - 2 * img + 16), dict(t=out)]
    for kw in bad:
        assert call(**kw) == RT_ERR_INVALID_ARG, kw
    assert ctx.launches() == before


def test_renderer_denoise_needs_the_guides(ctx, rt):
    case = cornell_case()
    for aovs in ((), ("albedo",), ("normal",), ("direct", "fresnel")):
        r = _renderer(rt, ctx, case, 16, 16, 1, aovs=aovs)
        with pytest.raises(ValueError):
            r.denoise()
