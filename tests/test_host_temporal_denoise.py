"""dxr_headless --orbit / --denoise-temporal / --aov position: the temporal denoiser and the position AOV through the C++ host
(ProgressiveRaytracingPipeline::denoiseTemporal), held to the Python path replayed from the frames the run dumped."""
import subprocess

import numpy as np
import pytest

from conftest import rel_rmse
from dxrexperiments_b200 import scenes, types as T
from test_host_aov import EXE, HOST
from test_host_cpp import read_exr, read_pfm, write_obj

pytestmark = pytest.mark.gpu
GUIDES = ("albedo", "normal", T.AOV_POSITION_NAME)


@pytest.fixture(scope="module")
def host_built():
    subprocess.run(["make", "-C", HOST, "-s"], check=True)
    return EXE


def _scene(tmp_path):
    mesh = scenes.cornell_box()
    obj = tmp_path / "cornell.obj"
    write_obj(obj, mesh)
    env = scenes.sky_cube(16)
    envf = tmp_path / "env.bin"
    env.astype("<f4").tofile(envf)
    return mesh, env, ["--model", str(obj), "--pipeline", "progressive", "--seed", "7", "--eye", "0", "0", "3.5", "--at", "0", "0", "0",
                       "--light-pos", "0", "0.5", "0", "--env-raw", str(envf), "16"]


def _replay(rt, ctx, mesh, env, w, h, frames_path, n, aovs):
    raw = np.fromfile(frames_path, dtype=np.uint8).reshape(n, 188)
    ren = rt.Renderer(ctx, [mesh], [scenes.IDENTITY_3X4], [scenes.make_material()], env, rt.PROGRESSIVE, w, h, aovs=aovs)
    return ren, [T.PerFrameConstants.from_buffer_copy(raw[s].tobytes()) for s in range(n)]


def test_headless_denoise_temporal_equals_the_python_path(host_built, tmp_path, ctx, rt):
    mesh, env, cmd = _scene(tmp_path)
    w, h, n = 96, 64, 8
    clean, frames = tmp_path / "clean.pfm", tmp_path / "frames.bin"
    r = subprocess.run([EXE] + cmd + ["--width", str(w), "--height", str(h), "--spp", str(n), "--orbit", "0.5",
                                      "--denoise-temporal", str(clean), "--dump-frames", str(frames)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    ren, fs = _replay(rt, ctx, mesh, env, w, h, frames, n, GUIDES)
    eyes = [tuple(f.cameraParams.worldEyePos[:3]) for f in fs]
    assert len(set(eyes)) == n and all(f.cameraParams.accumCount == 0 for f in fs)  # an orbit of one-sample frames
    for f in fs:
        ren.dispatch(f)
        out = ren.denoise_temporal()
    ctx.status()
    assert ren.temporal_history()[0, ..., 3].max() > 1
    got = read_pfm(clean)
    assert rel_rmse(got, out[..., :3]) <= 1e-6
    # EXR by extension
    exr = tmp_path / "clean.exr"
    r = subprocess.run([EXE] + cmd + ["--width", str(w), "--height", str(h), "--spp", str(n), "--orbit", "0.5",
                                      "--denoise-temporal", str(exr)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    np.testing.assert_array_equal(read_exr(exr)[..., :3], got)


def test_headless_position_aov(host_built, tmp_path, ctx, rt):
    mesh, env, cmd = _scene(tmp_path)
    w, h, n = 80, 48, 3
    pos, frames = tmp_path / "position.exr", tmp_path / "frames.bin"
    r = subprocess.run([EXE] + cmd + ["--width", str(w), "--height", str(h), "--spp", str(n), "--aov", "position", str(pos),
                                      "--dump-frames", str(frames)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    ren, fs = _replay(rt, ctx, mesh, env, w, h, frames, n, (T.AOV_POSITION_NAME,))
    for f in fs:
        ren.dispatch(f)
    ctx.status()
    p = read_exr(pos)
    assert rel_rmse(p, ren.aov(T.AOV_POSITION_NAME)) <= 1e-6
    assert 0.0 < p[..., 3].mean() <= 1.0


def test_headless_denoise_temporal_rejections(host_built, tmp_path):
    base = [EXE, "--scene", "cornell", "--width", "32", "--height", "32"]
    for extra in (["--pipeline", "realtime", "--denoise-temporal", str(tmp_path / "c.pfm")],
                  ["--world", "2", "--rank", "0", "--comm-file", str(tmp_path / "id"), "--denoise-temporal", str(tmp_path / "c.pfm")],
                  ["--denoise-temporal"]):
        r = subprocess.run(base + extra, capture_output=True, text=True, timeout=120)
        assert r.returncode != 0 and "denoise-temporal" in r.stderr, (extra, r.stderr)
