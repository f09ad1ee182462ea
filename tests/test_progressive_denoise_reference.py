"""CPU: the restatement of rt_denoise_progressive (tests/progressive_denoise_reference.py) that the GPU is held to has the
filter's exact properties, and it removes most of the Monte Carlo noise of a 4-spp oracle frame."""
import numpy as np
import pytest

import aov_reference
import progressive_denoise_reference as pdr
from conftest import rel_rmse
from dxrexperiments_b200 import scenes
from helpers import cornell_case

# rel RMSE(denoised 4 spp) / rel RMSE(4 spp), both against 1024 spp, Cornell 96 x 96, default parameters.  Measured 0.346
# with this restatement (0.33-0.35 for 3-5 iterations at sigma_luminance 4, 0.38-0.42 at 8, 0.70 at 1).
QUALITY_RATIO_MEASURED, QUALITY_RATIO_BOUND = 0.346, 0.45


def test_zero_iterations_return_the_beauty_frame():
    b, a, n = pdr.synthetic_inputs(37, 23, 1)
    out = pdr.denoise(b, a, n, iterations=0)
    np.testing.assert_array_equal(out[..., :3], b[..., :3])
    assert np.all(out[..., 3] == 1.0)


@pytest.mark.parametrize("iterations", [1, 3, 5])
def test_constant_image_is_a_fixed_point(iterations):
    h, w = 40, 52
    b = np.tile(np.array([0.7, 0.3, 0.2, 1.0], np.float32), (h, w, 1))
    a = np.tile(np.array([0.5, 0.4, 0.3, 1.0], np.float32), (h, w, 1))
    n = np.tile(np.array([0.0, 0.6, 0.8, 1.0], np.float32), (h, w, 1))
    out = pdr.denoise(b, a, n, iterations)
    np.testing.assert_allclose(out, b, rtol=1e-6, atol=0)


@pytest.mark.parametrize("iterations", [0, 2, 5])
def test_sky_is_copied_and_never_read(iterations):
    b, a, n = pdr.synthetic_inputs(45, 31, 2)
    sky = n[..., 3] == 0
    out = pdr.denoise(b, a, n, iterations)
    np.testing.assert_array_equal(out[sky][:, :3], b[sky][:, :3])
    b2, a2 = b.copy(), a.copy()
    b2[sky] = np.float32(1e4)
    a2[sky] = np.float32(7.0)
    out2 = pdr.denoise(b2, a2, n, iterations)
    np.testing.assert_array_equal(out2[~sky], out[~sky])


@pytest.mark.parametrize("iterations", range(6))
def test_perpendicular_halves_do_not_mix(iterations):
    w, h = 48, 20
    b, a, n = pdr.halves_inputs(w, h, 3)
    out = pdr.denoise(b, a, n, iterations)
    b2 = b.copy()
    b2[:, w // 2:, :3] = np.float32(50.0) * b2[:, w // 2:, :3] + np.float32(3.0)
    out2 = pdr.denoise(b2, a, n, iterations)
    np.testing.assert_array_equal(out2[:, :w // 2], out[:, :w // 2])
    if iterations:
        assert not np.array_equal(out2[:, w // 2:], out[:, w // 2:])


def cornell_quality_frames(w, h, spp, first_sample):
    """Jitter-free frames: the progressive RayGen's jitter (up to 15 pixels at jitterScale 30) makes a 4-spp frame a few
    displaced copies of the scene, an error no spatial filter can undo (the ratio is 0.80 with jittered frames); without
    it, what remains between 4 and 1024 spp is the Monte Carlo noise the filter is for.  Samples first_sample ..
    first_sample + spp - 1, so that the noisy frame and the reference draw different random numbers."""
    case = cornell_case()
    return case, [scenes.make_frame(case.setup, w, h, first_sample + s, s, jitter=(0.0, 0.0)) for s in range(spp)]


def test_quality_on_the_oracle(orc):
    w = h = 96
    case, ref_frames = cornell_quality_frames(w, h, 1024, 0)
    _, frames = cornell_quality_frames(w, h, 4, 5000)
    otlas, recs = case.oracle(orc)
    ref, noisy = np.zeros((h, w, 4), np.float32), np.zeros((h, w, 4), np.float32)
    for f in ref_frames:
        orc.render_progressive(otlas, recs, case.env, f, w, h, ref, threads=8)
    for f in frames:
        orc.render_progressive(otlas, recs, case.env, f, w, h, noisy, threads=8)
    aov = aov_reference.render_aovs(orc, otlas, recs, case.meshes, case.env, frames, w, h, names=("albedo", "normal"))
    out = pdr.denoise(noisy, aov["albedo"], aov["normal"], *pdr.default_params())
    ratio = rel_rmse(out[..., :3], ref[..., :3]) / rel_rmse(noisy[..., :3], ref[..., :3])
    print(f"denoised / noisy rel RMSE against 1024 spp: {ratio:.4f}")
    assert ratio <= QUALITY_RATIO_BOUND, ratio
