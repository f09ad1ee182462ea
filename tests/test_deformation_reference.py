"""CPU: the restatement of the previous-position AOV's deformation term (tests/deformation_reference.py) that the GPU is
held to has the rule's exact properties, and on a deforming mesh it keeps the history that the position test otherwise
throws away."""
import numpy as np
import pytest

import aov_reference
import deformation_reference as dr
import motion_reference as mr
import temporal_denoise_reference as tdr
from dxrexperiments_b200 import scenes, types as T
from helpers import SceneCase, cornell_case
from test_motion_reference import box_ratio, run_sequence
from test_temporal_denoise_reference import dyadic_camera, dyadic_planes

F = np.float32

# Cornell 96 x 96 with scenes.waving_sheet's defaults (a travelling wave moving the sheet by up to 0.075 per frame along
# z), static camera, 16 one-sample jitter-free frames, last frame against 1024 jitter-free samples of the last frame's
# scene; rel RMSE over the sheet's pixels in the last frame, as a ratio to that of the noisy frame.  Measured with this
# restatement, default parameters:
#   sheet pixels with history (n > 1): 1.000 with the deformation, 0.504 without;
#   the temporal pass alone (0 a-trous iterations): 0.268 with the deformation, 0.822 without;
#   with the default 5 a-trous iterations: 0.118 with the deformation, 0.126 without.  As for the sliding box
#   (test_motion_reference.py), the spatial stage already flattens much of the noise, so after it the deformation buys
#   mostly history length.
HISTORY_SHARE_BOUND, HISTORY_SHARE_PLAIN_MAX = 0.98, 0.6
TEMPORAL_RATIO_BOUND = 0.31            # and at most this fraction of the ratio without the deformation:
TEMPORAL_OVER_PLAIN_BOUND = 0.4
FILTERED_RATIO_BOUND = 0.13            # with the a-trous iterations, and no worse than without


def sheet_frame_case(frame):
    c = cornell_case()
    meshes, transforms = scenes.waving_sheet(frame)
    return SceneCase(meshes, transforms=transforms, setup=c.setup)


def test_equal_positions_give_the_motion_only_aov(orc):
    """Previous positions equal to the current ones add nothing: the AOV of the motion alone, for no motion, a motion,
    an unmatched instance (i >= n) and a NULL pointer."""
    case = sheet_frame_case(3)
    w, h = 64, 48
    blas = dr.refitted_blas(orc, scenes.waving_sheet(0)[0][0], case.meshes[0])
    otlas = orc.Tlas([blas, orc.Blas.from_mesh(case.meshes[1])], case.transforms)
    f = scenes.make_frame(case.setup, w, h, 11, 0, jitter=(0.003, -0.004))
    shift = np.array([[1, 0, 0, 0.25, 0, 1, 0, -0.125, 0, 0, 1, 0.5]], F)
    same = [case.meshes[0].vertices["position"], case.meshes[1].vertices["position"]]
    for motion in (None, np.tile(shift, (2, 1))):
        want = mr.primary_previous_positions(orc, otlas, f, w, h, motion)
        assert (want[..., 3] == 1).mean() > 0.5
        for descs in (dr.descriptors(same, case.transforms), dr.descriptors(same[:1], case.transforms[:1]),
                      dr.descriptors([None, None], case.transforms), []):
            got = dr.primary_previous_positions(orc, otlas, f, w, h, motion, case.meshes, descs)
            np.testing.assert_array_equal(got, want)  # values: only a -0 coordinate may come out +0


@pytest.mark.parametrize("k", [1, 3])
def test_a_sheet_translated_by_vertex_edits_reprojects_k_pixels_back(k, orc):
    """A fronto-parallel quad whose vertices move by k pixel footprints under a static jitter-free camera (no instance
    motion): its covered pixels take their history from exactly k pixels back, where the position-only pass finds the
    wall."""
    w, h = 64, 32
    cam = dyadic_camera(0.0)
    quad0 = scenes.quad((-0.5, -0.5, 0.0), (0.5, -0.5, 0.0), (0.5, 0.5, 0.0), (-0.5, 0.5, 0.0))
    quad1 = scenes.Mesh(quad0.vertices.copy(), quad0.indices)
    quad1.vertices["position"][:, 0] += F(k * 2.0 / w)
    wall = scenes.quad((-4, -4, -1.0), (4, -4, -1.0), (4, 4, -1.0), (-4, 4, -1.0))
    frame = scenes.make_frame(scenes.FrameSetup(), w, h, 0, 0)
    frame.cameraParams = cam
    eye = [scenes.IDENTITY_3X4, scenes.IDENTITY_3X4]
    blas = dr.refitted_blas(orc, quad0)
    otlas0 = orc.Tlas([blas, orc.Blas.from_mesh(wall)], eye)
    p0 = tdr.primary_positions(orc, otlas0, frame, w, h)
    blas.update([dict(vertices=quad1.vertices, stride=24, indices=quad1.indices)])
    otlas1 = orc.Tlas([blas, orc.Blas.from_mesh(wall)], eye)
    p1 = tdr.primary_positions(orc, otlas1, frame, w, h)
    descs = dr.descriptors([quad0.vertices["position"], None], eye)
    q1 = dr.primary_previous_positions(orc, otlas1, frame, w, h, None, [quad1, wall], descs)
    on = (p1[..., 3] == 1) & (np.abs(p1[..., 2]) < 0.5)
    assert on.sum() >= 100
    n = np.zeros((h, w, 4), F)
    n[..., 2:] = 1
    px, py = np.meshgrid(np.arange(w), np.arange(h))
    ok, fx, fy, _ = tdr.reproject(n, q1, cam)
    assert ok[on].all()
    assert np.abs(fx - (px - k))[on].max() <= 1e-3 and np.abs(fy - py)[on].max() <= 1e-3
    b = np.ones((h, w, 4), F)
    _, h0 = tdr.denoise_temporal(b, b, n, p0, iterations=0)
    h1 = mr.temporal_history_motion(b, n, p1, q1, cam, h0)
    inner = on & np.roll(np.abs(p0[..., 2]) < 0.5, k, axis=1)
    assert inner.sum() >= on.sum() - 2 * h
    np.testing.assert_array_equal(h1[0, ..., 3][inner], 2)
    h1p = tdr.temporal_history(b, n, p1, cam, h0)
    assert (h1p[0, ..., 3][inner] == 1).sum() >= k * 8


def test_an_out_of_range_index_leaves_the_term_out(orc):
    case = sheet_frame_case(1)
    w, h = 32, 32
    blas = dr.refitted_blas(orc, scenes.waving_sheet(0)[0][0], case.meshes[0])
    otlas = orc.Tlas([blas, orc.Blas.from_mesh(case.meshes[1])], case.transforms)
    f = scenes.make_frame(case.setup, w, h, 0, 0)
    prev = scenes.waving_sheet(0)[0][0].vertices["position"]
    hits = otlas.trace(orc.primary_rays(f, w, h, float(tdr.JITTER_SCALE)), T.RAY_FLAG_CULL_BACK_FACING_TRIANGLES)
    hit = hits[hits["primitive_index"] != T.NO_HIT]
    dw, applied, invalid = dr.displacement(hit, case.meshes, dr.descriptors([prev[:-30], None], case.transforms))
    assert invalid.any() and applied.any() and not (invalid & applied).any()
    assert not dw[~applied].any()


# ---------------------------------------------------------------------------------------------------- quality
def sheet_quality_inputs(orc, w=96, h=96, frames=16):
    """Oracle renders of the quality experiment: (per-frame (beauty, albedo, normal, position, previous position,
    camera), 1024-spp truth of the last frame's scene, sheet pixels of the last frame)."""
    room = orc.Blas.from_mesh(sheet_frame_case(0).meshes[1])
    blas = dr.refitted_blas(orc, sheet_frame_case(0).meshes[0])
    ins, prev = [], None
    for f in range(frames):
        case = sheet_frame_case(f)
        blas.update([dict(vertices=case.meshes[0].vertices, stride=24, indices=case.meshes[0].indices)])
        otlas, recs = orc.Tlas([blas, room], case.transforms), orc.Records(case.meshes, case.materials)
        fr = scenes.make_frame(case.setup, w, h, 5000 + f, 0)
        descs = [] if prev is None else dr.descriptors([prev.vertices["position"], None], case.transforms)
        b = np.zeros((h, w, 4), F)
        orc.render_progressive(otlas, recs, case.env, fr, w, h, b, threads=8)
        aov = aov_reference.render_aovs(orc, otlas, recs, case.meshes, case.env, [fr], w, h, names=("albedo", "normal"))
        ins.append((b, aov["albedo"], aov["normal"], tdr.render_positions(orc, otlas, [fr], w, h),
                    dr.render_previous_positions(orc, otlas, [fr], w, h, None, case.meshes, descs), fr.cameraParams))
        prev = case.meshes[0]
    truth = np.zeros((h, w, 4), F)
    for s in range(1024):
        orc.render_progressive(otlas, recs, case.env, scenes.make_frame(case.setup, w, h, s, s), w, h, truth, threads=8)
    hits = otlas.trace(orc.primary_rays(fr, w, h, float(tdr.JITTER_SCALE)), T.RAY_FLAG_CULL_BACK_FACING_TRIANGLES)
    sheet = ((hits["primitive_index"] != T.NO_HIT) & (hits["instance_index"] == 0)).reshape(h, w)
    return ins, truth, sheet


def quality(ins, truth, sheet):
    """(history share with, without; temporal ratio with, without; filtered ratio with, without) on the sheet's pixels."""
    noisy = ins[-1][0]
    om, hm, op, hp = run_sequence(ins, 0)
    fm, _, fp, _ = run_sequence(ins, 5)
    return ((hm[0, ..., 3][sheet] > 1).mean(), (hp[0, ..., 3][sheet] > 1).mean(), box_ratio(om, noisy, truth, sheet),
            box_ratio(op, noisy, truth, sheet), box_ratio(fm, noisy, truth, sheet), box_ratio(fp, noisy, truth, sheet))


def check_quality(q):
    share, share_plain, m, pl, fm, fp = q
    assert share >= HISTORY_SHARE_BOUND and share_plain <= HISTORY_SHARE_PLAIN_MAX, (share, share_plain)
    assert m <= TEMPORAL_RATIO_BOUND and m <= TEMPORAL_OVER_PLAIN_BOUND * pl, (m, pl)
    assert fm <= FILTERED_RATIO_BOUND and fm <= fp, (fm, fp)


def test_quality_on_the_oracle(orc):
    ins, truth, sheet = sheet_quality_inputs(orc)
    assert sheet.sum() >= 1000
    q = quality(ins, truth, sheet)
    print("sheet pixels: with history %.4f / %.4f; temporal pass with deformation / noisy %.4f, without %.4f; "
          "with the a-trous iterations %.4f / %.4f" % q)
    check_quality(q)
