"""dxr_headless --deform / --aov previous-position / --denoise-temporal: a deforming model through the C++ host
(RtModel::setVertices, RtScene::update's deformation descriptors), held to the Python Renderer replayed from the frames
the run dumped, with and without --move on the same instance."""
import subprocess

import numpy as np
import pytest

from conftest import rel_rmse
from dxrexperiments_b200 import scenes, types as T
from test_host_cpp import read_exr, read_pfm
from test_host_instance_motion import MOVE, _translation
from test_host_temporal_denoise import _scene, host_built  # noqa: F401

pytestmark = pytest.mark.gpu
DEFORM = (0.02, 0.0, -0.015)
GUIDES = ("albedo", "normal", T.AOV_POSITION_NAME, T.AOV_PREVIOUS_POSITION_NAME)


@pytest.mark.parametrize("move", [False, True])
def test_headless_deform_equals_the_python_path(move, host_built, tmp_path, ctx, rt):  # noqa: F811
    mesh, env, cmd = _scene(tmp_path)
    w, h, n = 96, 64, 8
    clean, prev, beauty, frames = tmp_path / "clean.pfm", tmp_path / "prev.exr", tmp_path / "beauty.pfm", tmp_path / "frames.bin"
    args = ["--width", str(w), "--height", str(h), "--spp", str(n), "--deform", *map(str, DEFORM), "--denoise-temporal", str(clean),
            "--aov", "previous-position", str(prev), "--out", str(beauty), "--dump-frames", str(frames)]
    if move:
        args += ["--move", *map(str, MOVE)]
    r = subprocess.run([host_built] + cmd + args, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    raw = np.fromfile(frames, dtype=np.uint8).reshape(n, 188)
    fs = [T.PerFrameConstants.from_buffer_copy(raw[s].tobytes()) for s in range(n)]
    assert all(f.cameraParams.accumCount == 0 for f in fs)
    ren = rt.Renderer(ctx, [mesh], [scenes.IDENTITY_3X4], [scenes.make_material()], env, rt.PROGRESSIVE, w, h, aovs=GUIDES,
                      deforming=(0,))
    rest = mesh.vertices["position"]
    for k, f in enumerate(fs):
        if k:
            ren.set_vertices(0, scenes.sheared_positions(rest, k * np.array(DEFORM, np.float64)), mesh.vertices["normal"])
            if move:
                ren.set_transforms([_translation(k)])
        ren.dispatch(f)
        out = ren.denoise_temporal()
    ctx.status()
    hist = ren.temporal_history()
    assert (hist[0, ..., 3][hist[2, ..., 3] == 1] > 1).mean() > 0.85  # the deforming room kept its history
    assert rel_rmse(read_pfm(beauty), ren.image(0)[..., :3]) <= 1e-6
    assert rel_rmse(read_pfm(clean), out[..., :3]) <= 1e-6
    q, p = read_exr(prev), ren.aov(T.AOV_PREVIOUS_POSITION_NAME)
    assert rel_rmse(q, p) <= 1e-6
    assert np.abs(p - ren.aov(T.AOV_POSITION_NAME)).max() > 0.01
