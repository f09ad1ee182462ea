"""GPU: adaptive sampling of the progressive program (rt_set_adaptive_sampling, rt_adaptive_update).

Random numbers depend only on (pixel, frameCount), so pixel p's k-th sample is the same value whichever dispatches it
takes part in.  The closed-loop tests render one-sample frames (frameCount k, accumCount 0) with the plain pipeline, compose
the adaptive render from them with the float32 restatement (tests/adaptive_reference.py), and hold the GPU's adaptive
render to it bit for bit: beauty, every AOV, the moments and the counts.
"""
import ctypes as C

import numpy as np
import pytest

import adaptive_reference as ar
from dxrexperiments_b200 import scenes, types as T
from helpers import bunny_case, cornell_case, two_material_case

pytestmark = pytest.mark.gpu

ALL_AOVS = (*T.AOV_NAMES, T.AOV_POSITION_NAME, T.AOV_PREVIOUS_POSITION_NAME)


def _options(**kw):
    opt = scenes.default_options()
    for k, v in kw.items():
        setattr(opt, k, v)
    return opt


def _frame(case, w, h, k, accum, options=None, jitter=None):
    jit = scenes.jitter_sequence(31, k + 1, w, h)[k] if jitter is None else jitter
    return scenes.make_frame(case.setup, w, h, frame_count=k, accum_count=accum, jitter=jit, options=options or scenes.default_options())


def _renderer(rt, ctx, case, w, h, aovs=(), adaptive=False):
    return rt.Renderer(ctx, case.meshes, case.transforms, case.materials, case.env, rt.PROGRESSIVE, w, h, aovs=aovs, adaptive=adaptive)


@pytest.fixture
def opts(ctx):
    yield ctx.set_render_options
    ctx.set_render_options(1, False)


@pytest.mark.parametrize("half", [False, True])
@pytest.mark.parametrize("depth", [1, 2])
@pytest.mark.parametrize("view", ["beauty", "debug2", "indirect", "ao"])
def test_bound_without_updates_is_the_plain_pipeline(rt, ctx, opts, half, depth, view):
    case, w, h, K = cornell_case(), 40, 33, 3
    options = {"beauty": _options(), "debug2": _options(debug=2), "indirect": _options(showIndirectDiffuseOnly=1),
               "ao": _options(showAmbientOcclusionOnly=1)}[view]
    aovs = () if view == "ao" else ALL_AOVS
    # the moments are those of gOutput's clamped fp32 samples (the debug view's, or the AO view's): one-sample frames
    samples = []
    opts(depth, False)
    one = _renderer(rt, ctx, case, w, h)
    for k in range(K):
        one.dispatch(_frame(case, w, h, k, 0, options))
        samples.append(one.image())
    opts(depth, half)
    plain, adapt = _renderer(rt, ctx, case, w, h, aovs), _renderer(rt, ctx, case, w, h, aovs, adaptive=True)
    counts = []
    for r in (plain, adapt):
        ctx.ray_counts(reset=True)
        for k in range(K):
            r.dispatch(_frame(case, w, h, k, k, options))
        ctx.status()
        c = ctx.ray_counts()
        counts.append((c.primary, c.secondary, c.shadow))
    assert counts[0] == counts[1]
    np.testing.assert_array_equal(adapt.image(), plain.image())
    for a in aovs:
        np.testing.assert_array_equal(adapt.aov(a), plain.aov(a), err_msg=a)
    n, conv = adapt.sample_counts()
    assert np.all(n == K) and not conv.any()
    res = ar.compose(np.stack(samples))
    np.testing.assert_array_equal(adapt.moments(), res["moments"])


def _one_sample_frames(rt, ctx, case, w, h, K, options=None):
    """K one-sample frames (frameCount k, accumCount 0) of the beauty output and every AOV, fp32 targets."""
    r = _renderer(rt, ctx, case, w, h, ALL_AOVS)
    beauty, aovs = [], {a: [] for a in ALL_AOVS}
    for k in range(K):
        r.dispatch(_frame(case, w, h, k, 0, options))
        beauty.append(r.image())
        for a in ALL_AOVS:
            aovs[a].append(r.aov(a))
    return np.stack(beauty), {a: np.stack(v) for a, v in aovs.items()}


@pytest.mark.parametrize("half", [False, True])
@pytest.mark.parametrize("name", ["cornell", "two-material", "bunny"])
def test_closed_loop_equals_the_restatement(rt, ctx, opts, name, half):
    case = {"cornell": cornell_case, "two-material": two_material_case, "bunny": bunny_case}[name]()
    w, h, K, every = 61, 47, 24, 4
    params = (0.15, 0.1, 4, 20)
    beauty, aovs = _one_sample_frames(rt, ctx, case, w, h, K)
    want = ar.compose(beauty, aovs, ar.every(every, params, K), half=half)
    opts(1, half)
    r = _renderer(rt, ctx, case, w, h, ALL_AOVS, adaptive=True)
    active = []
    for k in range(K):
        r.dispatch(_frame(case, w, h, k, 0))
        if (k + 1) % every == 0:
            active.append(r.adaptive_update(T.AdaptiveParams(*params)))
    ctx.status()
    assert active == want["active"]
    assert any(0 < a < w * h for a in want["active"]), "the case converges some pixels before others"
    n, conv = r.sample_counts()
    np.testing.assert_array_equal(n | np.where(conv, ar.CONVERGED, np.uint32(0)), want["counts"])
    np.testing.assert_array_equal(r.moments(), want["moments"])
    np.testing.assert_array_equal(r.image(), want["beauty"])
    for a in ALL_AOVS:
        np.testing.assert_array_equal(r.aov(a), want["aovs"][a], err_msg=a)


@pytest.mark.parametrize("shape", [(1, 1), (1, 17), (13, 1), (15, 16), (16, 17), (33, 47), (200, 200), (129, 75)])
def test_update_kernel_equals_the_restatement(ctx, shape):
    h, w = shape
    rng = np.random.default_rng(h * 1000 + w)
    counts = rng.integers(0, 12, (h, w)).astype(np.uint32)
    counts[rng.random((h, w)) < 0.15] |= ar.CONVERGED
    m1 = (rng.random((h, w)) * 2).astype(np.float32)
    m2 = (m1 * m1 * (1 + rng.random((h, w)) * 0.05)).astype(np.float32)
    m2.reshape(-1)[:: 7] = (m1 * m1).reshape(-1)[:: 7]  # zero variance
    m2.reshape(-1)[3:: 11] = np.nan
    mom = np.stack([m1, m2], -1).astype(np.float32)
    for params in [(0.02, 0.1, 2, 10), (0.3, 0.05, 4, 11), (0.0, 1.0, 1, 1), (1e30, 0.1, 3, 2 ** 31 - 1)]:
        d_counts, d_mom, d_act = ctx.upload(counts), ctx.upload(mom), ctx.alloc(4)
        ctx.adaptive_update(d_mom, d_counts, w, h, T.AdaptiveParams(*params), d_act)
        got = d_counts.download(np.uint32, h * w).reshape(h, w)
        want, active = ar.update(counts, mom, *params)
        np.testing.assert_array_equal(got, want, err_msg=str(params))
        assert int(d_act.download(np.uint32, 1)[0]) == active
        np.testing.assert_array_equal(d_mom.download(np.float32, h * w * 2).reshape(h, w, 2), mom)
        ctx.adaptive_update(d_mom, d_counts, w, h, T.AdaptiveParams(*params), None)  # no active count: same update again
        np.testing.assert_array_equal(d_counts.download(np.uint32, h * w).reshape(h, w), want)


def _mask(h, w, seed=5):
    m = np.random.default_rng(seed).random((h, w)) < 0.4
    m[: h // 4, : w // 3] = True  # a whole converged block: some shading tiles have no active pixel
    return m


def _preset(r, mask, sentinel=0x3F00DEAD):
    """Fill every bound buffer with a sentinel pattern and mark `mask` converged (count 5 everywhere)."""
    h, w = mask.shape
    counts = np.full((h, w), 5, np.uint32) | np.where(mask, ar.CONVERGED, np.uint32(0))
    r.adaptive[0].upload(counts)
    r.adaptive[1].upload(np.full(h * w * 2, sentinel, np.uint32))
    for b in (*r.out, *r.aovs.values()):
        b.upload(np.full(h * w * 4, sentinel, np.uint32))
    return counts


def _bytes(r):
    h, w = r.height, r.width
    out = {"out": r.out[0].download(np.uint32).reshape(h, w, 4), "counts": r.adaptive[0].download(np.uint32).reshape(h, w),
           "moments": r.adaptive[1].download(np.uint32).reshape(h, w, 2)}
    out.update({a: b.download(np.uint32).reshape(h, w, 4) for a, b in r.aovs.items()})
    return out


@pytest.mark.parametrize("mode", ["full", "region", "strips", "two-band", "stats", "capture"])
def test_skipped_pixels_are_untouched(rt, ctx, mode):
    case = cornell_case()
    w, h = (640, 480) if mode == "two-band" else (70, 52)
    mask = _mask(h, w)
    r = _renderer(rt, ctx, case, w, h, ALL_AOVS, adaptive=True)
    before = _preset(r, mask)
    inside = np.ones((h, w), bool)
    region = strips = None
    if mode == "region":
        region = (9, 5, 61, 44)
        inside[:] = False
        inside[5:44, 9:61] = True
    if mode == "strips":
        strips = (4, 3, 1)
        rows = np.arange(h)
        inside[:] = ((rows // 4) % 3 == 1)[:, None]
    if mode == "stats":
        ctx.enable_trace_stats(True)
    if mode == "capture":
        ctx.enable_debug_capture(True)
    ctx.ray_counts(reset=True)
    ctx.trace_stats(reset=True)
    try:
        r.dispatch(_frame(case, w, h, 3, 0), region=region, strips=strips)
        ctx.status()
        counts = ctx.ray_counts()
        prim = ctx.trace_stats()[0].rays
        if mode == "capture":  # the hit slots are the active pixels' hits only
            assert ctx.debug_counts()["slots"] <= int((~mask & inside).sum())
            assert not np.any(mask.reshape(-1)[ctx.debug_array("slot_info")["pixel"]])
    finally:
        ctx.enable_trace_stats(False)
        ctx.enable_debug_capture(False)
    act = ~mask & inside
    assert counts.primary == int(act.sum()), "one primary ray per active pixel"
    if mode == "stats":
        assert prim == int(act.sum())
    got = _bytes(r)
    skipped = ~act
    sentinel = np.uint32(0x3F00DEAD)
    assert np.array_equal(got["counts"][skipped], before[skipped])
    assert np.all(got["counts"][act] == 6)
    for k, v in got.items():
        if k != "counts":
            assert np.all(v[skipped] == sentinel), k
            assert not np.any(np.all(v[act] == sentinel, axis=-1)), k


def test_two_band_dispatch_equals_one_band(rt, ctx):
    case, w, h = two_material_case(), 640, 448  # >= 2^18 pixels: two bands unless captured
    mask = _mask(h, w, 9)
    res = []
    for capture in (False, True):
        r = _renderer(rt, ctx, case, w, h, ("albedo", "normal"), adaptive=True)
        _preset(r, mask)
        ctx.enable_debug_capture(capture)
        try:
            for k in range(3):
                r.dispatch(_frame(case, w, h, k, 0))
            ctx.status()
        finally:
            ctx.enable_debug_capture(False)
        res.append(_bytes(r))
    for k in res[0]:
        np.testing.assert_array_equal(res[0][k], res[1][k], err_msg=k)


def test_argument_checks(rt, ctx):
    lib = rt.lib
    a, b = ctx.alloc(4096), ctx.alloc(8192)
    assert lib.rt_set_adaptive_sampling(ctx.handle, a.ptr, None) != 0
    assert lib.rt_set_adaptive_sampling(ctx.handle, None, b.ptr) != 0
    assert lib.rt_set_adaptive_sampling(ctx.handle, a.ptr + 2, b.ptr) != 0
    assert lib.rt_set_adaptive_sampling(ctx.handle, a.ptr, b.ptr + 4) != 0
    assert lib.rt_set_adaptive_sampling(ctx.handle, a.ptr, b.ptr) == 0
    assert lib.rt_set_adaptive_sampling(ctx.handle, None, None) == 0
    good = T.adaptive_defaults()

    def upd(m, c, w=32, h=32, p=good, act=None):
        return lib.rt_adaptive_update(ctx.handle, m, c, w, h, C.byref(p) if p is not None else None, act)
    assert upd(b.ptr, a.ptr) == 0
    assert upd(None, a.ptr) != 0 and upd(b.ptr, None) != 0 and upd(b.ptr, a.ptr, p=None) != 0
    assert upd(b.ptr, a.ptr, w=0) != 0 and upd(b.ptr, a.ptr, h=0) != 0
    assert upd(b.ptr + 4, a.ptr) != 0 and upd(b.ptr, a.ptr + 2) != 0 and upd(b.ptr, a.ptr, act=a.ptr + 4098) != 0
    assert upd(b.ptr, b.ptr + 4096) != 0, "counts overlapping moments"
    assert upd(b.ptr, a.ptr, act=a.ptr + 64) != 0 and upd(b.ptr, a.ptr, act=b.ptr + 8) != 0
    for bad in [(-0.1, 0.1, 2, 4), (float("nan"), 0.1, 2, 4), (float("inf"), 0.1, 2, 4), (0.1, 0.0, 2, 4), (0.1, float("nan"), 2, 4),
                (0.1, 0.1, 0, 4), (0.1, 0.1, 5, 4), (0.1, 0.1, 2, 2 ** 31)]:
        assert upd(b.ptr, a.ptr, p=T.AdaptiveParams(*bad)) != 0, bad


def test_realtime_program_is_rejected(rt, ctx):
    case, w, h = cornell_case(), 32, 32
    r = rt.Renderer(ctx, case.meshes, case.transforms, case.materials, case.env, rt.REALTIME, w, h)
    counts, moments = ctx.alloc(4 * w * h).zero(), ctx.alloc(8 * w * h).zero()
    r.dispatch(_frame(case, w, h, 0, 0))  # binds nothing adaptive: fine
    ctx.set_adaptive_sampling(counts, moments)
    try:
        with pytest.raises(rt.RtError):
            rt.check(rt.lib.rt_dispatch_rays(ctx.handle, r.program.handle, w, h, 1))
    finally:
        ctx.set_adaptive_sampling(None, None)
    with pytest.raises(ValueError):
        rt.Renderer(ctx, case.meshes, case.transforms, case.materials, case.env, rt.REALTIME, w, h, adaptive=True)


def test_renderer_misuse_and_reset(rt, ctx):
    case, w, h = cornell_case(), 24, 20
    plain = _renderer(rt, ctx, case, w, h)
    for call in (lambda: plain.adaptive_update(), plain.sample_counts, plain.moments, plain.reset_adaptive):
        with pytest.raises(ValueError):
            call()
    r = _renderer(rt, ctx, case, w, h, ("albedo", "normal", "position"), adaptive=True)
    r.dispatch(_frame(case, w, h, 0, 0))
    with pytest.raises(ValueError):
        r.denoise_temporal()
    assert r.denoise().shape == (h, w, 4)  # the AOVs are per-pixel means: the spatial filter takes them as they are
    assert r.adaptive_update(T.AdaptiveParams(0.1, 0.1, 1, 1)) == 0
    r.dispatch(_frame(case, w, h, 1, 1))
    assert np.all(r.sample_counts()[0] == 1)
    r.reset_adaptive()
    n, conv = r.sample_counts()
    assert not n.any() and not conv.any() and not r.moments().any() and not r.image().any() and not r.aov("albedo").any()
    # another Renderer's dispatch unbinds the adaptive buffers
    plain.dispatch(_frame(case, w, h, 0, 0))
    ctx.status()
    assert not r.sample_counts()[0].any()


def test_gpu_quality_matches_the_cpu_figure(rt, ctx, orc):
    """The closed loop on the GPU reproduces the restatement's quality figure on jitter-free Cornell: the same one-sample
    frames as the oracle's (to the oracle's parity tolerance), so the same ratio to three decimals."""
    import test_adaptive_reference as tar
    case, w, h, K = cornell_case(), 96, 96, 256
    frames = []
    r = _renderer(rt, ctx, case, w, h)
    for k in range(K):
        r.dispatch(_frame(case, w, h, 5000 + k, 0, jitter=(0.0, 0.0)))
        frames.append(r.image())
    frames = np.stack(frames)
    ref = tar.stack(case, w, h, 0, 1024, orc).mean(axis=0, dtype=np.float64).astype(np.float32)
    res = ar.run_until_converged(frames, (0.1, 0.1, 8, K), 4)
    spp = float((res["counts"] & ar.COUNT_MASK).sum()) / (w * h)
    uniform = frames[:max(1, int(round(spp)))].mean(axis=0, dtype=np.float64).astype(np.float32)
    from conftest import rel_rmse
    ratio = rel_rmse(res["beauty"][..., :3], ref[..., :3]) / rel_rmse(uniform[..., :3], ref[..., :3])
    print(f"GPU frames: {spp:.1f} spp, adaptive / uniform rel RMSE {ratio:.3f}")
    assert abs(ratio - tar.QUALITY["cornell"]["rmse"]) <= 0.01
