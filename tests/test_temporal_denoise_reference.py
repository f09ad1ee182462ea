"""CPU: the restatement of rt_denoise_temporal (tests/temporal_denoise_reference.py) that the GPU is held to has the temporal
pass's exact properties, and on a moving camera it leaves clearly less Monte Carlo noise than the spatial filter alone."""
import dataclasses

import numpy as np
import pytest

import aov_reference
import progressive_denoise_reference as pdr
import temporal_denoise_reference as tdr
from closed_form import camera_rays
from conftest import rel_rmse
from dxrexperiments_b200 import scenes, types as T
from helpers import cornell_case

F = np.float32

# Cornell 96 x 96, a 16-frame orbit of 0.5 degrees per frame, one jitter-free sample per frame, last frame against 1024
# jitter-free samples at the last camera; rel RMSE of the filtered frame over that of the noisy 1-spp frame, default
# parameters.  Measured with this restatement: temporal 0.138, spatial (rt_denoise_progressive) 0.224.
TEMPORAL_RATIO_MEASURED, SPATIAL_RATIO_MEASURED = 0.138, 0.224
TEMPORAL_RATIO_BOUND = 0.17   # and at most this fraction of the spatial ratio:
TEMPORAL_OVER_SPATIAL_BOUND = 0.75


def dyadic_camera(eye_x, jitter=(0.0, 0.0)):
    """CameraParams with U = +x, V = +y, W = -z, eye (eye_x, 0, 1): every quantity of the reprojection of a plane z = 0 or
    z = 0.5 is a short dyadic fraction, so it is exact in float32."""
    c = T.CameraParams()
    c.worldEyePos[:] = (eye_x, 0.0, 1.0, 1.0)
    c.U[:] = (1.0, 0.0, 0.0, 0.0)
    c.V[:] = (0.0, 1.0, 0.0, 0.0)
    c.W[:] = (0.0, 0.0, -1.0, 0.0)
    c.jitters[:] = jitter
    return c


def dyadic_planes(w, h, cam, front_x=None):
    """(normal, position) of the camera's primary hits on the plane z = 0 and, where x < front_x, on a plane z = 0.5 in
    front of it (normals +z, coverage 1)."""
    sx = ((np.arange(w, dtype=F) + F(0.5)) / F(w)) * F(2) - F(1)
    sy = ((np.arange(h, dtype=F) + F(0.5)) / F(h)) * F(2) - F(1)
    ex = F(cam.worldEyePos[0])
    pos = np.zeros((h, w, 4), F)
    pos[..., 0] = ex + sx[None, :]
    pos[..., 1] = -sy[:, None]
    pos[..., 3] = 1
    if front_x is not None:  # z = 0.5: half the distance, half the offset from the eye
        fx = ex + F(0.5) * sx[None, :] + np.zeros((h, 1), F)
        front = fx < F(front_x)
        pos[front, 0] = fx[front]
        pos[front, 1] = (F(-0.5) * sy[:, None] + np.zeros((1, w), F))[front]
        pos[front, 2] = F(0.5)
    normal = np.zeros((h, w, 4), F)
    normal[..., 2] = 1
    normal[..., 3] = 1
    return normal, pos


def synthetic_position(w, h, seed):
    """A position AOV to go with progressive_denoise_reference.synthetic_inputs: random points, coverage of its normal."""
    b, a, n = pdr.synthetic_inputs(w, h, seed)
    rng = np.random.Generator(np.random.PCG64(seed + 1))
    p = np.zeros((h, w, 4), F)
    p[..., :3] = rng.uniform(-1, 1, size=(h, w, 3)).astype(F)
    p[..., 3] = n[..., 3]
    p[n[..., 3] == 0] = 0
    return b, a, n, p


@pytest.mark.parametrize("iterations", range(6))
def test_without_history_equals_the_spatial_filter(iterations):
    b, a, n, p = synthetic_position(41, 27, 5)
    kw = dict(tdr.default_params(), iterations=iterations)
    out, hist = tdr.denoise_temporal(b, a, n, p, **kw)
    np.testing.assert_array_equal(out, pdr.denoise(b, a, n, iterations, kw["normal_exponent_log2"], kw["sigma_luminance"],
                                                   kw["sigma_albedo"]))
    np.testing.assert_array_equal(hist[0, ..., :3], b[..., :3])
    assert np.all(hist[0, ..., 3] == 1)
    np.testing.assert_array_equal(hist[2], n)
    np.testing.assert_array_equal(hist[3], p)


def test_static_camera_reprojects_onto_the_pixel_centres():
    w, h = 96, 64
    case, on, _ = aov_reference.plane_case(w, h)
    o, d = camera_rays(case.setup, w, h)
    t = -o[..., 2] / d[..., 2]
    pos = np.zeros((h, w, 4), F)
    pos[..., :3] = (o + t[..., None] * d).astype(F)
    pos[..., 3] = 1
    normal = np.zeros((h, w, 4), F)
    normal[..., 2:] = 1
    cam = scenes.make_frame(case.setup, w, h, 0, 0).cameraParams
    ok, fx, fy, _ = tdr.reproject(normal, pos, cam)
    px, py = np.meshgrid(np.arange(w), np.arange(h))
    assert ok[on].all()
    assert np.abs(fx - px)[on].max() <= 1e-3 and np.abs(fy - py)[on].max() <= 1e-3


@pytest.mark.parametrize("k", [1, 3])
def test_a_pan_of_k_pixels_shifts_the_history_by_k(k):
    w, h = 64, 32
    prev_cam, cam = dyadic_camera(0.0), dyadic_camera(k * 2.0 / w)
    n0, p0 = dyadic_planes(w, h, prev_cam)
    n1, p1 = dyadic_planes(w, h, cam)
    rng = np.random.Generator(np.random.PCG64(k))
    b0, b1 = (np.concatenate([rng.random((h, w, 3), F), np.ones((h, w, 1), F)], axis=-1) for _ in range(2))
    _, h0 = tdr.denoise_temporal(b0, b0, n0, p0, iterations=0)
    ok, fx, fy, _ = tdr.reproject(n1, p1, prev_cam)
    px, py = np.meshgrid(np.arange(w), np.arange(h))
    np.testing.assert_array_equal(fx[:, :w - k], (px + k)[:, :w - k])
    np.testing.assert_array_equal(fy[:, :w - k], py[:, :w - k])
    _, h1 = tdr.denoise_temporal(b1, b1, n1, p1, prev_cam, h0, iterations=0)
    np.testing.assert_array_equal(h1[0, :, :w - k, 3], 2)
    np.testing.assert_array_equal(h1[0, :, w - k:, 3], 1)  # the newly exposed columns
    # history weight 1/2 from pixel x + k of the previous frame
    want = F(0.5) * b0[:, k:, :3] + F(0.5) * b1[:, :w - k, :3]
    np.testing.assert_array_equal(h1[0, :, :w - k, :3], want)
    np.testing.assert_array_equal(h1[0, :, w - k:, :3], b1[:, w - k:, :3])


def test_a_disocclusion_rejects_the_history():
    """A plane z = 0.5 in front of x < 0 moves twice as far across the image as the background under a pan: the background
    it uncovers reprojects onto it in the previous frame, and the position test drops that history."""
    w, h, k = 64, 16, 4
    prev_cam, cam = dyadic_camera(0.0), dyadic_camera(k * 2.0 / w)
    n0, p0 = dyadic_planes(w, h, prev_cam, front_x=0.0)
    n1, p1 = dyadic_planes(w, h, cam, front_x=0.0)
    b = np.ones((h, w, 4), F)
    _, h0 = tdr.denoise_temporal(b, b, n0, p0, iterations=0)
    _, h1 = tdr.denoise_temporal(b, b, n1, p1, prev_cam, h0, iterations=0)
    back1, front0 = p1[..., 2] == 0, p0[..., 2] == F(0.5)
    px = np.arange(w)
    src = np.clip(px + k, 0, w - 1)  # background pixels reproject k pixels to the right
    uncovered = back1 & front0[:, src] & (px + k < w)[None, :]
    assert uncovered.sum() >= h * k
    np.testing.assert_array_equal(h1[0, ..., 3][uncovered], 1)
    kept = back1 & ~front0[:, src] & (px + k < w)[None, :]
    assert kept.sum() > w * h // 4
    np.testing.assert_array_equal(h1[0, ..., 3][kept], 2)


def test_a_constant_frame_is_a_fixed_point():
    w, h = 64, 32
    cam = dyadic_camera(0.0)
    n, p = dyadic_planes(w, h, cam)
    b = np.tile(np.array([0.7, 0.3, 0.2, 1.0], F), (h, w, 1))
    a = np.tile(np.array([0.5, 0.4, 0.3, 1.0], F), (h, w, 1))
    prev = hist = None
    for _ in range(8):
        out, hist = tdr.denoise_temporal(b, a, n, p, prev, hist)
        prev = cam
        np.testing.assert_allclose(out, b, rtol=1e-6, atol=0)
        np.testing.assert_allclose(hist[0, ..., :3], b[..., :3], rtol=1e-6, atol=0)
    assert np.all(hist[0, ..., 3] == 8)


def test_integrated_variance_approaches_alpha_over_two_minus_alpha():
    w, h, frames, sigma = 64, 64, 48, 0.1
    cam = dyadic_camera(0.0)
    n, p = dyadic_planes(w, h, cam)
    rng = np.random.Generator(np.random.PCG64(3))
    prev = hist = None
    for _ in range(frames):
        b = np.ones((h, w, 4), F)
        b[..., :3] = (F(1) + F(sigma) * rng.standard_normal((h, w, 1)).astype(F)) * np.ones((1, 1, 3), F)
        hist = tdr.temporal_history(b, n, p, prev, hist)
        prev = cam
    alpha = tdr.default_params()["alpha_color"]
    ratio = float(np.var(hist[0, ..., 0].astype(np.float64))) / sigma ** 2
    assert abs(ratio / (alpha / (2 - alpha)) - 1) <= 0.1, ratio


def orbit_quality_inputs(orc, w=96, h=96, frames=16, degrees=0.5):
    """Oracle renders of the quality experiment: (per-frame (beauty, albedo, normal, position, camera), 1024-spp truth at the
    last camera)."""
    case = cornell_case()
    otlas, recs = case.oracle(orc)
    fs = tdr.orbit_frames(case.setup, w, h, frames, degrees, first_sample=5000)
    last = dataclasses.replace(case.setup, camera=scenes.orbit(case.setup.camera, (frames - 1) * degrees))
    truth = np.zeros((h, w, 4), F)
    for s in range(1024):
        orc.render_progressive(otlas, recs, case.env, scenes.make_frame(last, w, h, s, s), w, h, truth, threads=8)
    ins = []
    for f in fs:
        b = np.zeros((h, w, 4), F)
        orc.render_progressive(otlas, recs, case.env, f, w, h, b, threads=8)
        aov = aov_reference.render_aovs(orc, otlas, recs, case.meshes, case.env, [f], w, h, names=("albedo", "normal"))
        ins.append((b, aov["albedo"], aov["normal"], tdr.render_positions(orc, otlas, [f], w, h), f.cameraParams))
    return case, fs, ins, truth


def quality_ratios(temporal_out, spatial_out, noisy, truth):
    e = rel_rmse(noisy[..., :3], truth[..., :3])
    return rel_rmse(temporal_out[..., :3], truth[..., :3]) / e, rel_rmse(spatial_out[..., :3], truth[..., :3]) / e


def check_quality(rt_ratio, sp_ratio):
    assert rt_ratio <= TEMPORAL_RATIO_BOUND, rt_ratio
    assert rt_ratio <= TEMPORAL_OVER_SPATIAL_BOUND * sp_ratio, (rt_ratio, sp_ratio)


def test_quality_on_the_oracle(orc):
    _, _, ins, truth = orbit_quality_inputs(orc)
    prev = hist = None
    for b, a, n, p, cam in ins:
        out, hist = tdr.denoise_temporal(b, a, n, p, prev, hist, **tdr.default_params())
        prev = cam
    b, a, n, _, _ = ins[-1]
    t, s = quality_ratios(out, pdr.denoise(b, a, n, *pdr.default_params()), b, truth)
    print(f"temporal / noisy {t:.4f}, spatial / noisy {s:.4f} (rel RMSE against 1024 spp)")
    check_quality(t, s)
