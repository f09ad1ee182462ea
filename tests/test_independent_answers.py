"""Answers that do not come from the oracle (VERDICT r1, weak #1 i): closed-form radiance values, an independent numpy
statement of the RNG recurrences and of the denoiser, and the reference's own denoiser inputs.

CPU tests pin the ORACLE with them; the `gpu` tests hold the CUDA path to the very same numbers through the C ABI.
"""
import os

import numpy as np
import pytest

import closed_form as cf
from dxrexperiments_b200 import scenes, types as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


# ---------------------------------------------------------------------------------------------- RNG
def tea16(v0, v1):
    """The 16-round TEA hash with the published constants (delta 0x9e3779b9; keys 0xa341316c, 0xc8013ea4, 0xad90777d,
    0x7e95761e), vectorised over uint32 arrays with wrap-around arithmetic in uint64."""
    M = np.uint64(0xFFFFFFFF)
    v0, v1, s = v0.astype(np.uint64), v1.astype(np.uint64), np.uint64(0)
    for _ in range(16):
        s = (s + np.uint64(0x9E3779B9)) & M
        v0 = (v0 + ((((v1 << np.uint64(4)) & M) + np.uint64(0xA341316C) & M) ^ ((v1 + s) & M) ^ (((v1 >> np.uint64(5)) + np.uint64(0xC8013EA4)) & M))) & M
        v1 = (v1 + ((((v0 << np.uint64(4)) & M) + np.uint64(0xAD90777D) & M) ^ ((v0 + s) & M) ^ (((v0 >> np.uint64(5)) + np.uint64(0x7E95761E)) & M))) & M
    return v0.astype(np.uint32)


def test_rng_matches_an_independent_numpy_statement(orc):
    rng = np.random.Generator(np.random.PCG64(99))
    pix = np.concatenate([np.arange(64, dtype=np.uint32), rng.integers(0, 3840 * 2160, 4000, dtype=np.uint32), [0xFFFFFFFF, 0x80000000]]).astype(np.uint32)
    frm = np.concatenate([np.zeros(64, np.uint32), rng.integers(0, 1 << 20, 4000, dtype=np.uint32), [0xFFFFFFFF, 7]]).astype(np.uint32)
    want = tea16(pix, frm)
    for p, f, w in zip(pix.tolist(), frm.tolist(), want.tolist()):
        assert orc.init_rand(p, f) == w
    # LCG: s <- 1664525 s + 1013904223 (mod 2^32); value = (s & 0xFFFFFF) / 2^24 — exactly representable in fp32
    for seed in want[:200].tolist():
        s = seed
        for _ in range(4):
            v, s_o = orc.next_rand(s)
            s = (1664525 * s + 1013904223) & 0xFFFFFFFF
            assert s_o == s and np.float32(v) == np.float32((s & 0xFFFFFF) / 16777216.0)


# ---------------------------------------------------------------------------------------------- closed-form shading
def _oracle_render(orc, case):
    blases = [orc.Blas.from_mesh(m) for m in case.meshes]
    tlas = orc.Tlas(blases, [scenes.IDENTITY_3X4] * len(blases))
    recs = orc.Records(case.meshes, case.materials)
    if case.realtime:
        return orc.render_realtime(tlas, recs, case.env, case.frame(0), case.w, case.h, threads=4)
    acc = np.zeros((case.h, case.w, 4), np.float32)
    for s in range(case.spp):
        orc.render_progressive(tlas, recs, case.env, case.frame(s), case.w, case.h, acc, threads=4)
    return acc, None


def _cuda_render(rt, ctx, case):
    r = rt.Renderer(ctx, case.meshes, [scenes.IDENTITY_3X4] * len(case.meshes), case.materials, case.env,
                    rt.REALTIME if case.realtime else rt.PROGRESSIVE, case.w, case.h)
    for s in range(case.spp):
        r.dispatch(case.frame(s))
    ctx.status()
    return r.image(0), (r.image(1) if case.realtime else None)


@pytest.mark.parametrize("make", cf.CASES, ids=lambda f: f.__name__)
def test_oracle_reproduces_closed_form_radiance(make, orc):
    case = make()
    a, b = _oracle_render(orc, case)
    case.check(a, "oracle")
    if case.realtime:
        assert not np.asarray(b)[..., :3].any()  # no reflection: the indirect-specular AOV is black


def test_oracle_furnace_is_invariant_under_accumulation_and_converges_with_uniform_sampling(orc):
    cf.furnace(spp=5).check(_oracle_render(orc, cf.furnace(spp=5))[0], "oracle, 5 spp running mean")
    # uniform hemisphere sampling: radiance * NoL / pdf (ProgressiveRaytracing.hlsl:71-75) has expectation E * pi as well;
    # a 48-spp image mean must land on the same closed form
    c = cf.furnace(w=48, h=36, spp=48, uniform=True)
    img = np.asarray(_oracle_render(orc, c)[0], np.float64)[..., :3]
    ratio = img[c.mask].mean(axis=0) / c.expected[c.mask].mean(axis=0)
    np.testing.assert_allclose(ratio, 1.0, atol=5e-3)


@pytest.mark.gpu
@pytest.mark.parametrize("make", cf.CASES, ids=lambda f: f.__name__)
def test_cuda_reproduces_closed_form_radiance(make, ctx, rt):
    case = make()
    a, b = _cuda_render(rt, ctx, case)
    case.check(a, "cuda")
    if case.realtime:
        assert not np.asarray(b)[..., :3].any()


@pytest.mark.gpu
def test_cuda_furnace_accumulation_and_uniform_sampling(ctx, rt):
    cf.furnace(spp=5).check(_cuda_render(rt, ctx, cf.furnace(spp=5))[0], "cuda, 5 spp running mean")
    c = cf.furnace(w=48, h=36, spp=48, uniform=True)
    img = np.asarray(_cuda_render(rt, ctx, c)[0], np.float64)[..., :3]
    ratio = img[c.mask].mean(axis=0) / c.expected[c.mask].mean(axis=0)
    np.testing.assert_allclose(ratio, 1.0, atol=5e-3)


# ---------------------------------------------------------------------------------------------- denoiser
def _random_aovs(h, w, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    direct = np.ones((h, w, 4), np.float32)
    spec = np.ones((h, w, 4), np.float32)
    base = rng.random((h // 8 + 1, w // 8 + 1, 3), dtype=np.float32)  # blocky joint image: real edges for the range weight
    direct[..., :3] = np.kron(base, np.ones((8, 8, 1), np.float32))[:h, :w] * 0.5 + rng.random((h, w, 3), dtype=np.float32) * 0.02
    spec[..., :3] = rng.random((h, w, 3), dtype=np.float32)
    return direct, spec


@pytest.mark.parametrize("k,mode,tonemap,gamma", [(12, 0, 1, 0), (5, 0, 1, 1), (20, 1, 0, 0), (1, 3, 0, 0), (12, 0, 0, 1)])
def test_oracle_denoiser_matches_the_independent_statement(k, mode, tonemap, gamma, orc):
    direct, spec = _random_aovs(70, 93, 5 + k)
    out, tmp = orc.denoise(direct, spec, T.DenoiserParams(1.25, 2.2, tonemap, gamma, k, mode))
    hp, final = cf.denoise_reference(direct, spec, k=k, exposure=1.25, tonemap=bool(tonemap), gamma_correct=bool(gamma), mode=mode)
    np.testing.assert_allclose(tmp[..., :3], hp, rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(out[..., :3], final, rtol=3e-5, atol=3e-6)


def _mock_crop():
    """A 192 x 128 crop of the reference's own mock denoiser inputs (src/DenoiseCompositor.cpp:52-60, 1922 x 1126 8-bit
    PNGs), as WIC decodes them: 8-bit UNORM -> float / 255."""
    g = np.load(os.path.join(GOLDEN, "denoise_mock_crop.npz"))
    return g["direct_u8"].astype(np.float32) / np.float32(255.0), g["spec_u8"].astype(np.float32) / np.float32(255.0)


def test_oracle_denoiser_on_the_committed_crop_of_the_reference_inputs(orc):
    direct, spec = _mock_crop()
    out, _ = orc.denoise(direct, spec, T.DenoiserParams(1.0, 2.2, 1, 0, 12, 0))
    _, final = cf.denoise_reference(direct, spec, k=12)
    ok = np.isfinite(final).all(axis=-1)
    np.testing.assert_allclose(out[..., :3][ok], final[ok], rtol=3e-5, atol=3e-6)


@pytest.mark.gpu
def test_cuda_denoiser_on_reference_inputs_and_at_their_full_size(ctx, orc):
    direct, spec = _mock_crop()
    out, _ = ctx.denoise(direct, spec, T.DenoiserParams(1.0, 2.2, 1, 0, 12, 0))
    _, final = cf.denoise_reference(direct, spec, k=12)
    ok = np.isfinite(final).all(axis=-1)
    np.testing.assert_allclose(out[..., :3][ok], final[ok], rtol=3e-5, atol=3e-6)
    # the reference's mock size (1922 x 1126: neither dimension a multiple of the tiles), tiled from the crop
    H, W = 1126, 1922
    reps = (H // direct.shape[0] + 1, W // direct.shape[1] + 1, 1)
    D, S = np.tile(direct, reps)[:H, :W].copy(), np.tile(spec, reps)[:H, :W].copy()
    got, gtmp = ctx.denoise(D, S, T.DenoiserParams(1.0, 2.2, 1, 0, 12, 0))
    want, wtmp = orc.denoise(D, S, T.DenoiserParams(1.0, 2.2, 1, 0, 12, 0), threads=16)
    ok = np.isfinite(want).all(axis=-1)
    np.testing.assert_allclose(gtmp[..., :3][ok], wtmp[..., :3][ok], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(got[..., :3][ok], want[..., :3][ok], rtol=1e-5, atol=1e-6)
