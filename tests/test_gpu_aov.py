"""GPU: the AOV outputs of the progressive program (rt_set_aov_output).

AOV k is what debug view k shows, accumulated from the same rays as the beauty frame.  Random numbers depend only on
(pixel, frameCount) and the debug views only change the final selection in k_resolve, so a render with the AOVs bound and
a render with view k switched on trace identical rays: AOV k must equal that render's beauty output bit for bit.
"""
import ctypes as C

import numpy as np
import pytest

import aov_reference
from conftest import rel_rmse
from dxrexperiments_b200 import scenes, sharding, types as T
from helpers import bunny_case, cornell_case, two_material_case

pytestmark = pytest.mark.gpu

VIEW_OF_AOV = aov_reference.VIEW_OF_AOV
# name: (DebugOptions overrides, max_radiance_ray_depth, half_render_targets)
CONFIGS = {"default": ({}, 1, False), "radiance_depth_2": ({}, 2, False), "half_targets": ({}, 1, True),
           "one_light_sampling": ({"debug": 2}, 1, False), "uniform_hemisphere": ({"cosineHemisphereSampling": 0}, 1, False)}


def _options(overrides):
    opt = scenes.default_options()
    for k, v in overrides.items():
        setattr(opt, k, v)
    return opt


def _frames(case, w, h, spp, overrides, seed=31):
    jit = scenes.jitter_sequence(seed, spp, w, h)
    return [scenes.make_frame(case.setup, w, h, frame_count=s, accum_count=s, jitter=jit[s], options=_options(overrides))
            for s in range(spp)]


def _renderer(rt, ctx, case, w, h, aovs=()):
    return rt.Renderer(ctx, case.meshes, case.transforms, case.materials, case.env, rt.PROGRESSIVE, w, h, aovs=aovs)


def _render(rt, ctx, case, w, h, spp, overrides, aovs=()):
    r = _renderer(rt, ctx, case, w, h, aovs)
    ctx.ray_counts(reset=True)
    for f in _frames(case, w, h, spp, overrides):
        r.dispatch(f)
    ctx.status()
    return r, ctx.ray_counts()


def _check_debug_view_identity(rt, ctx, case, w, h, spp, config):
    overrides, depth, half = CONFIGS[config]
    ctx.set_render_options(depth, half)
    try:
        with_aovs, counts = _render(rt, ctx, case, w, h, spp, overrides, T.AOV_NAMES)
        plain, plain_counts = _render(rt, ctx, case, w, h, spp, overrides)
        # binding AOVs changes neither the beauty output nor the rays traced
        np.testing.assert_array_equal(with_aovs.image(0), plain.image(0))
        assert (counts.primary, counts.secondary, counts.shadow) == (plain_counts.primary, plain_counts.secondary, plain_counts.shadow)
        for name, view in VIEW_OF_AOV.items():
            ref, _ = _render(rt, ctx, case, w, h, spp, {**overrides, view: 1})
            np.testing.assert_array_equal(with_aovs.aov(name), ref.image(0), err_msg=name)
        n = with_aovs.aov("normal")
        assert 0.0 < n[..., 3].mean() <= 1.0
        assert not n[n[..., 3] == 0.0].any()
    finally:
        ctx.set_render_options(1, False)


@pytest.mark.parametrize("config", sorted(CONFIGS))
@pytest.mark.parametrize("case_fn,w,h,spp", [(cornell_case, 96, 96, 4), (bunny_case, 120, 72, 2), (two_material_case, 104, 64, 3)])
def test_aovs_equal_debug_views(case_fn, w, h, spp, config, ctx, rt):
    _check_debug_view_identity(rt, ctx, case_fn(), w, h, spp, config)


@pytest.mark.parametrize("config", ["default", "half_targets"])
def test_aovs_equal_debug_views_two_band_dispatch(config, ctx, rt):
    """640x512 is large enough for a dispatch to run as two pixel bands on their own streams."""
    _check_debug_view_identity(rt, ctx, two_material_case(), 640, 512, 1, config)


def test_aovs_single_sample_cornell(ctx, rt):
    _check_debug_view_identity(rt, ctx, cornell_case(), 64, 48, 1, "default")


@pytest.mark.parametrize("config", ["default", "half_targets"])
@pytest.mark.parametrize("case_fn,w,h,spp", [(cornell_case, 128, 128, 3), (two_material_case, 160, 96, 2), (bunny_case, 160, 90, 2)])
def test_aovs_match_oracle(case_fn, w, h, spp, config, ctx, rt, orc):
    """Against the CPU reference built from the oracle (tests/aov_reference.py): AOVs 0-4 within the north-star tolerance,
    the normal AOV exact on >= 99.99 % of the pixels (the rest: pixels whose primary hit differs in float32)."""
    overrides, depth, half = CONFIGS[config]
    case = case_fn()
    otlas, recs = case.oracle(orc)
    frames = _frames(case, w, h, spp, overrides)
    ctx.set_render_options(depth, half)
    orc.set_render_options(depth, half)
    try:
        r = _renderer(rt, ctx, case, w, h, T.AOV_NAMES)
        for f in frames:
            r.dispatch(f)
        ctx.status()
        ref = aov_reference.render_aovs(orc, otlas, recs, case.meshes, case.env, frames, w, h, half_targets=half)
    finally:
        ctx.set_render_options(1, False)
        orc.set_render_options(1, False)
    for name in T.AOV_NAMES:
        g = r.aov(name)
        assert np.isfinite(g).all(), name
        if not np.any(ref[name][..., :3]):  # e.g. no reflective material in view
            assert not g[..., :3].any(), name
            continue
        assert rel_rmse(g, ref[name]) <= 1e-3, name
    exact = np.all(r.aov("normal") == ref["normal"], axis=-1)
    assert exact.mean() >= 0.9999, f"normal AOV exact on {exact.mean():.6f} of the pixels"


def test_normal_aov_of_a_plane_against_closed_form(ctx, rt):
    """A square of normal +z under a black sky: (0, 0, 1, 1) on the square, (0, 0, 0, 0) on the sky."""
    w, h = 96, 64
    case, on, off = aov_reference.plane_case(w, h)
    r = _renderer(rt, ctx, case, w, h, ("normal",))
    for s in range(3):
        r.dispatch(scenes.make_frame(case.setup, w, h, s, s))
    ctx.status()
    aov_reference.check_plane_normals(r.aov("normal"), on, off)


def test_region_dispatch_aovs_equal_full_frame(ctx, rt):
    case = two_material_case()
    w, h = 100, 76
    full = _renderer(rt, ctx, case, w, h, T.AOV_NAMES)
    tiled = _renderer(rt, ctx, case, w, h, T.AOV_NAMES)
    for f in _frames(case, w, h, 2, {}):
        full.dispatch(f)
        for reg in [(0, 0, 37, 40), (37, 0, w, 40), (0, 40, 64, h), (64, 40, w, h)]:
            tiled.dispatch(f, region=reg)
    ctx.status()
    np.testing.assert_array_equal(tiled.image(0), full.image(0))
    for name in T.AOV_NAMES:
        np.testing.assert_array_equal(tiled.aov(name), full.aov(name), err_msg=name)


@pytest.mark.parametrize("world,strip_groups", [(2, 2), (4, 2), (2, 1)])
def test_sharded_aovs_sum_to_the_full_frame(world, strip_groups, ctx, rt):
    """Strip-interleaved and sample shards (sharding.plan), each rank's buffers weighted as rt_accum_reduce weights them
    and summed: every AOV equals the single-dispatch frame up to the fp32 summation order."""
    case = bunny_case(4)
    w, h, spp = 200, 150, 4
    frames = _frames(case, w, h, spp, {})
    full = _renderer(rt, ctx, case, w, h, T.AOV_NAMES)
    for f in frames:
        full.dispatch(f)
    total = {a: np.zeros((h, w, 4), np.float32) for a in ("beauty",) + T.AOV_NAMES}
    for rank in range(world):
        p = sharding.plan(rank, world, spp, strip_groups=strip_groups, strip_rows=32)
        r = _renderer(rt, ctx, case, w, h, T.AOV_NAMES)
        for local, s in enumerate(p.samples):
            f = frames[s]
            f.cameraParams.accumCount = local
            r.dispatch(f, strips=(32, strip_groups, p.strip_group))
            f.cameraParams.accumCount = s
        total["beauty"] += np.float32(p.weight) * r.image(0)
        for a in T.AOV_NAMES:
            total[a] += np.float32(p.weight) * r.aov(a)
    ctx.status()
    assert rel_rmse(total["beauty"], full.image(0)) <= 1e-6
    for a in T.AOV_NAMES:
        assert rel_rmse(total[a], full.aov(a)) <= 1e-6, a


def test_aov_errors_and_unbinding(ctx, rt):
    case = cornell_case()
    w, h = 64, 48
    r = _renderer(rt, ctx, case, w, h, ("albedo",))
    buf = r.aovs["albedo"]
    with pytest.raises(rt.RtError):
        rt.check(rt.lib.rt_set_aov_output(ctx.handle, T.AOV_COUNT, buf.ptr, 16 * w))
    with pytest.raises(rt.RtError):
        rt.check(rt.lib.rt_set_aov_output(ctx.handle, 0xFFFFFFFF, None, 0))
    f = scenes.make_frame(case.setup, w, h, 0, 0)
    # pitch too small for the launch width: set by hand after the Renderer's own binding
    rt.check(lib_dispatch_prepare(rt, ctx, r, f))
    rt.check(rt.lib.rt_set_aov_output(ctx.handle, T.AOV_ALBEDO, buf.ptr, 16 * (w - 1)))
    with pytest.raises(rt.RtError):
        rt.check(rt.lib.rt_dispatch_rays(ctx.handle, r.program.handle, w, h, 1))
    # the ambient-occlusion view traces AO rays instead of lighting
    with pytest.raises(rt.RtError):
        r.dispatch(scenes.make_frame(case.setup, w, h, 0, 0, options=_options({"showAmbientOcclusionOnly": 1})))
    # a realtime program's outputs already are AOVs
    rtr = rt.Renderer(ctx, case.meshes, case.transforms, case.materials, case.env, rt.REALTIME, w, h)
    rtr.dispatch(f)  # binds no AOV: fine
    rt.check(rt.lib.rt_set_aov_output(ctx.handle, T.AOV_ALBEDO, buf.ptr, 16 * w))
    with pytest.raises(rt.RtError):
        rt.check(rt.lib.rt_dispatch_rays(ctx.handle, rtr.program.handle, w, h, 1))
    # unbinding with NULL returns to the plain path: the same image as a Renderer that never had AOVs
    rt.check(rt.lib.rt_set_aov_output(ctx.handle, T.AOV_ALBEDO, None, 0))
    plain = _renderer(rt, ctx, case, w, h)
    rt.check(lib_dispatch_prepare(rt, ctx, plain, f))
    rt.check(rt.lib.rt_dispatch_rays(ctx.handle, plain.program.handle, w, h, 1))
    ref = _renderer(rt, ctx, case, w, h)
    ref.dispatch(f)
    ctx.status()
    np.testing.assert_array_equal(plain.image(0), ref.image(0))
    assert not buf.download(np.float32).any()  # every failed dispatch above left the AOV untouched


def lib_dispatch_prepare(rt, ctx, r, frame):
    """Bind the Renderer's output, TLAS and frame constants, but no AOV."""
    rt.check(rt.lib.rt_set_output(ctx.handle, 0, r.out[0].ptr, 16 * r.width))
    rt.check(rt.lib.rt_set_tlas(ctx.handle, r.tlas.result.ptr))
    return rt.lib.rt_set_frame_constants(ctx.handle, C.byref(frame))


def test_max_iterations_leaves_aovs_untouched(ctx, rt):
    case = cornell_case()
    w, h = 64, 64
    opt = _options({"maxIterations": 1})
    r = _renderer(rt, ctx, case, w, h, T.AOV_NAMES)
    r.dispatch(scenes.make_frame(case.setup, w, h, 0, 0, options=opt))
    first = {a: r.aov(a).copy() for a in T.AOV_NAMES}
    assert first["albedo"].any()
    r.dispatch(scenes.make_frame(case.setup, w, h, 1, 1, options=opt))
    ctx.status()
    for a in T.AOV_NAMES:
        np.testing.assert_array_equal(r.aov(a), first[a], err_msg=a)


def test_renderer_rejects_unknown_aov_name(ctx, rt):
    case = cornell_case()
    with pytest.raises(ValueError):
        _renderer(rt, ctx, case, 16, 16, ("depth",))
