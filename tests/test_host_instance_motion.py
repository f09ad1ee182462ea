"""dxr_headless --move / --aov previous-position / --denoise-temporal: moving instances through the C++ host (RtScene::update,
ProgressiveRaytracingPipeline::denoiseTemporal with rt_denoise_temporal_motion), held to the Python path replayed from
the frames the run dumped."""
import subprocess

import numpy as np
import pytest

import motion_reference as mr
from conftest import rel_rmse
from dxrexperiments_b200 import scenes, types as T
from test_host_cpp import read_exr, read_pfm
from test_host_temporal_denoise import _replay, _scene, host_built  # noqa: F401

pytestmark = pytest.mark.gpu
MOVE = (0.03, 0.0, -0.02)


def _translation(f):
    t = np.array(scenes.IDENTITY_3X4)
    t[[3, 7, 11]] = [np.float32(f * m) for m in MOVE]
    return t


def test_headless_move_equals_the_python_path(host_built, tmp_path, ctx, rt):  # noqa: F811
    mesh, env, cmd = _scene(tmp_path)
    w, h, n = 96, 64, 8
    clean, prev, frames = tmp_path / "clean.pfm", tmp_path / "prev.exr", tmp_path / "frames.bin"
    r = subprocess.run([host_built] + cmd + ["--width", str(w), "--height", str(h), "--spp", str(n), "--move", *map(str, MOVE),
                                                  "--denoise-temporal", str(clean), "--aov", "previous-position", str(prev),
                                                  "--dump-frames", str(frames)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    ren, fs = _replay(rt, ctx, mesh, env, w, h, frames, n, ("albedo", "normal", T.AOV_POSITION_NAME, T.AOV_PREVIOUS_POSITION_NAME))
    assert len({tuple(f.cameraParams.worldEyePos[:3]) for f in fs}) == 1  # a static camera
    assert all(f.cameraParams.accumCount == 0 for f in fs)
    for k, f in enumerate(fs):
        if k:
            ren.set_transforms([_translation(k)])
            np.testing.assert_array_equal(ren.motion, mr.motion_matrices([_translation(k - 1)], [_translation(k)]))
        ren.dispatch(f)
        out = ren.denoise_temporal()
    ctx.status()
    hist = ren.temporal_history()
    # the moving instance kept its history, except where it uncovers the image edge or the jittered taps leave it
    assert (hist[0, ..., 3][hist[2, ..., 3] == 1] > 1).mean() > 0.85
    assert rel_rmse(read_pfm(clean), out[..., :3]) <= 1e-6
    q = read_exr(prev)
    assert rel_rmse(q, ren.aov(T.AOV_PREVIOUS_POSITION_NAME)) <= 1e-6
    p = ren.aov(T.AOV_POSITION_NAME)
    hit = p[..., 3] == 1
    np.testing.assert_allclose(q[hit][:, :3] - p[hit][:, :3], np.tile(-np.array(MOVE, np.float32), (hit.sum(), 1)), atol=1e-5)
