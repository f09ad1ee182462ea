"""CPU: the restatement of the previous-position AOV and of rt_denoise_temporal_motion (tests/motion_reference.py) that the
GPU is held to has the motion variant's exact properties, and on a moving instance it keeps the history that the
position-only pass throws away."""
import numpy as np
import pytest

import aov_reference
import motion_reference as mr
import progressive_denoise_reference as pdr
import temporal_denoise_reference as tdr
from conftest import rel_rmse
from dxrexperiments_b200 import scenes, types as T
from helpers import SceneCase, cornell_case
from test_temporal_denoise_reference import dyadic_camera, dyadic_planes

F = np.float32

# Cornell 96 x 96 with the sliding box (scenes.sliding_box, 0.08 per frame: more than position_tolerance * distance, so
# the position-only pass rejects what moved), static camera, 16 one-sample jitter-free frames, last frame against 1024
# jitter-free samples of the last frame's scene; rel RMSE over the pixels the box covers in the last frame, as a ratio to
# that of the noisy frame.  Measured with this restatement, default parameters:
#   the temporal pass alone (0 a-trous iterations): with motion 0.346, without (rt_denoise_temporal) 0.844;
#   box pixels with history (n > 1): 0.947 with motion, 0.620 without;
#   with the default 5 a-trous iterations: 0.183 with motion, 0.176 without.  The spatial stage already flattens the
#   box's uniformly lit faces, and the history lags the box's changing shading by about 1/alpha frames, so on this small
#   object the motion buys history length, not a lower filtered error.
TEMPORAL_RATIO_MEASURED, TEMPORAL_RATIO_NO_MOTION_MEASURED = 0.346, 0.844
TEMPORAL_RATIO_BOUND = 0.42          # and at most this fraction of the ratio without motion:
TEMPORAL_OVER_NO_MOTION_BOUND = 0.5
HISTORY_SHARE_BOUND = 0.93           # box pixels that keep history with motion
FILTERED_RATIO_BOUND = 0.21          # with the a-trous iterations


def test_identity_and_no_motion_give_the_position_aov(orc):
    case = sliding_case(3)
    w, h = 64, 48
    otlas, _ = case.oracle(orc)
    f = scenes.make_frame(case.setup, w, h, 11, 0, jitter=(0.003, -0.004))
    p = tdr.primary_positions(orc, otlas, f, w, h)
    assert (p[..., 3] == 1).mean() > 0.5
    eye = np.tile(scenes.IDENTITY_3X4, (2, 1))
    for motion in (None, eye, eye[:1], np.zeros((0, 12), F)):  # eye[:1]: the room's index 1 >= n
        q = mr.primary_previous_positions(orc, otlas, f, w, h, motion)
        np.testing.assert_array_equal(q, p)
    # no motion or i >= n is a copy: bit for bit, signed zeros included
    np.testing.assert_array_equal(mr.primary_previous_positions(orc, otlas, f, w, h, None).view(np.uint32), p.view(np.uint32))


@pytest.mark.parametrize("iterations", [0, 3, 5])
def test_motion_reprojection_with_q_equal_p_is_the_temporal_pass(iterations):
    w, h, k = 64, 32, 3
    prev_cam, cam = dyadic_camera(0.0), dyadic_camera(k * 2.0 / w, jitter=(0.25 / w, -0.5 / h))
    n0, p0 = dyadic_planes(w, h, prev_cam, front_x=0.0)  # a pan with a disocclusion: some taps kept, some rejected
    n1, p1 = dyadic_planes(w, h, cam, front_x=0.0)
    b0, a0, _ = pdr.synthetic_inputs(w, h, 5)
    b1, a1, _ = pdr.synthetic_inputs(w, h, 6)
    kw = dict(tdr.default_params(), iterations=iterations)
    _, h0 = tdr.denoise_temporal(b0, a0, n0, p0, **kw)
    want = tdr.denoise_temporal(b1, a1, n1, p1, prev_cam, h0, **kw)
    got = mr.denoise_temporal_motion(b1, a1, n1, p1, p1, prev_cam, h0, **kw)
    assert 0 < (want[1][0, ..., 3] > 1).mean() < 1
    for g, r in zip(got, want):
        np.testing.assert_array_equal(g.view(np.uint32), r.view(np.uint32))


@pytest.mark.parametrize("k", [1, 3])
def test_a_quad_moved_by_k_pixels_reprojects_k_pixels_back(k, orc):
    """A fronto-parallel quad instance translated by k pixel footprints under a static jitter-free camera: its covered
    pixels take their history from exactly k pixels back, where the position-only pass finds another surface."""
    w, h = 64, 32
    cam = dyadic_camera(0.0)
    # closed form: the plane z = 0 seen by the dyadic camera, moved by k footprints (2/w) along +x
    n1, p1 = dyadic_planes(w, h, cam)
    motion = np.array([[1, 0, 0, -k * 2.0 / w, 0, 1, 0, 0, 0, 0, 1, 0]], F)
    q = mr.apply_motion(p1[..., :3], np.zeros((h, w), np.uint32), motion)
    ok, fx, fy, _ = tdr.reproject(n1, np.concatenate([q, p1[..., 3:]], axis=-1), cam)
    px, py = np.meshgrid(np.arange(w), np.arange(h))
    assert ok[:, k:].all()
    np.testing.assert_array_equal(fx[:, k:], (px - k)[:, k:])
    np.testing.assert_array_equal(fy, np.where(ok, py, 0))
    # the oracle's primary hits on a quad instance in front of a wall, moved by k footprints between two frames
    quad = scenes.quad((-0.5, -0.5, 0.0), (0.5, -0.5, 0.0), (0.5, 0.5, 0.0), (-0.5, 0.5, 0.0))
    wall = scenes.quad((-4, -4, -1.0), (4, -4, -1.0), (4, 4, -1.0), (-4, 4, -1.0))
    t0 = np.array(scenes.IDENTITY_3X4)
    t1 = t0.copy()
    t1[3] = k * 2.0 / w
    frame = scenes.make_frame(scenes.FrameSetup(), w, h, 0, 0)
    frame.cameraParams = cam
    case = SceneCase([quad, wall], transforms=[t0, scenes.IDENTITY_3X4])
    otlas0, _ = case.oracle(orc)
    case.transforms = [t1, scenes.IDENTITY_3X4]
    otlas1, _ = case.oracle(orc)
    p0 = tdr.primary_positions(orc, otlas0, frame, w, h)
    p1 = tdr.primary_positions(orc, otlas1, frame, w, h)
    q1 = mr.primary_previous_positions(orc, otlas1, frame, w, h, mr.motion_matrices([t0, scenes.IDENTITY_3X4], [t1, scenes.IDENTITY_3X4]))
    on = (p1[..., 3] == 1) & (np.abs(p1[..., 2]) < 0.5)  # the quad's pixels in this frame
    assert on.sum() >= 100
    n = np.zeros((h, w, 4), F)
    n[..., 2:] = 1
    ok, fx, fy, _ = tdr.reproject(n, q1, cam)
    assert ok[on].all()
    assert np.abs(fx - (px - k))[on].max() <= 1e-3 and np.abs(fy - py)[on].max() <= 1e-3
    # the whole history of the quad comes along: n = 2 on the quad except its newly uncovered column
    b = np.ones((h, w, 4), F)
    _, h0 = tdr.denoise_temporal(b, b, n, p0, iterations=0)
    h1 = mr.temporal_history_motion(b, n, p1, q1, cam, h0)
    src_on = np.abs(p0[..., 2]) < 0.5
    inner = on & np.roll(src_on, k, axis=1)
    assert inner.sum() >= on.sum() - 2 * h
    np.testing.assert_array_equal(h1[0, ..., 3][inner], 2)
    np.testing.assert_array_equal(h1[3], p1)
    # the position-only pass loses the quad's edge columns: what lies k pixels back is the wall
    h1p = tdr.temporal_history(b, n, p1, cam, h0)
    assert (h1p[0, ..., 3][inner] == 1).sum() >= k * 8


# ---------------------------------------------------------------------------------------------------- quality
def sliding_case(frame):
    c = cornell_case()
    meshes, transforms = scenes.sliding_box(frame)
    return SceneCase(meshes, transforms=transforms, setup=c.setup)


def sliding_quality_inputs(orc, w=96, h=96, frames=16):
    """Oracle renders of the quality experiment: (per-frame (beauty, albedo, normal, position, previous position, camera),
    1024-spp truth of the last frame's scene, box pixels of the last frame)."""
    ins = []
    for f in range(frames):
        case = sliding_case(f)
        otlas, recs = case.oracle(orc)
        fr = scenes.make_frame(case.setup, w, h, 5000 + f, 0)
        motion = None if f == 0 else mr.motion_matrices(sliding_case(f - 1).transforms, case.transforms)
        b = np.zeros((h, w, 4), F)
        orc.render_progressive(otlas, recs, case.env, fr, w, h, b, threads=8)
        aov = aov_reference.render_aovs(orc, otlas, recs, case.meshes, case.env, [fr], w, h, names=("albedo", "normal"))
        ins.append((b, aov["albedo"], aov["normal"], tdr.render_positions(orc, otlas, [fr], w, h),
                    mr.render_previous_positions(orc, otlas, [fr], w, h, motion), fr.cameraParams))
    truth = np.zeros((h, w, 4), F)
    for s in range(1024):
        orc.render_progressive(otlas, recs, case.env, scenes.make_frame(case.setup, w, h, s, s), w, h, truth, threads=8)
    hits = otlas.trace(orc.primary_rays(fr, w, h, float(tdr.JITTER_SCALE)), T.RAY_FLAG_CULL_BACK_FACING_TRIANGLES)
    box = ((hits["primitive_index"] != T.NO_HIT) & (hits["instance_index"] == 0)).reshape(h, w)
    return ins, truth, box


def box_ratio(out, noisy, truth, box):
    return rel_rmse(out[box][:, :3], truth[box][:, :3]) / rel_rmse(noisy[box][:, :3], truth[box][:, :3])


def run_sequence(ins, iterations):
    """(out with motion, history with motion, out without, history without) of the last frame."""
    prev = hm = hp = None
    kw = dict(tdr.default_params(), iterations=iterations)
    for b, a, n, p, q, cam in ins:
        om, hm = mr.denoise_temporal_motion(b, a, n, p, q, prev, hm, **kw)
        op, hp = tdr.denoise_temporal(b, a, n, p, prev, hp, **kw)
        prev = cam
    return om, hm, op, hp


def check_quality(motion_ratio, plain_ratio, history_share, filtered_ratio):
    assert motion_ratio <= TEMPORAL_RATIO_BOUND, motion_ratio
    assert motion_ratio <= TEMPORAL_OVER_NO_MOTION_BOUND * plain_ratio, (motion_ratio, plain_ratio)
    assert history_share >= HISTORY_SHARE_BOUND, history_share
    assert filtered_ratio <= FILTERED_RATIO_BOUND, filtered_ratio


def test_quality_on_the_oracle(orc):
    ins, truth, box = sliding_quality_inputs(orc)
    assert box.sum() >= 200
    noisy = ins[-1][0]
    om, hm, op, hp = run_sequence(ins, 0)
    m, pl = box_ratio(om, noisy, truth, box), box_ratio(op, noisy, truth, box)
    share, share_plain = (hm[0, ..., 3][box] > 1).mean(), (hp[0, ..., 3][box] > 1).mean()
    fm = box_ratio(run_sequence(ins, 5)[0], noisy, truth, box)
    print(f"box pixels: temporal pass with motion / noisy {m:.4f}, without {pl:.4f}; with history {share:.4f} / {share_plain:.4f}; "
          f"with the a-trous iterations {fm:.4f}")
    check_quality(m, pl, share, fm)
