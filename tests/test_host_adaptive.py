"""dxr_headless --adaptive / --sample-counts: adaptive sampling through the C++ host
(ProgressiveRaytracingPipeline::setAdaptiveSampling / adaptiveUpdate), held to the Python Renderer replayed from the frames
the run dumped."""
import json
import subprocess

import numpy as np
import pytest

from conftest import rel_rmse
from dxrexperiments_b200 import scenes, types as T
from test_host_aov import EXE
from test_host_cpp import read_exr, read_pfm
from test_host_temporal_denoise import _scene, host_built  # noqa: F401

pytestmark = pytest.mark.gpu


def _run(cmd):
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return json.loads(r.stdout.strip().splitlines()[-1])


def _replay(rt, ctx, mesh, env, w, h, frames_path, aovs):
    raw = np.fromfile(frames_path, dtype=np.uint8).reshape(-1, 188)
    ren = rt.Renderer(ctx, [mesh], [scenes.IDENTITY_3X4], [scenes.make_material()], env, rt.PROGRESSIVE, w, h, aovs=aovs, adaptive=True)
    return ren, [T.PerFrameConstants.from_buffer_copy(raw[s].tobytes()) for s in range(raw.shape[0])]


def test_headless_adaptive_equals_the_python_path(host_built, tmp_path, ctx, rt):  # noqa: F811
    mesh, env, cmd = _scene(tmp_path)
    w, h, spp, every, thr, mn = 64, 48, 64, 4, 0.3, 4
    out, counts, albedo, clean, frames = (tmp_path / n for n in ("out.pfm", "n.pfm", "albedo.exr", "clean.pfm", "frames.bin"))
    res = _run([host_built] + cmd + ["--width", str(w), "--height", str(h), "--spp", str(spp), "--adaptive", str(thr), "--adaptive-min",
                                     str(mn), "--adaptive-every", str(every), "--out", str(out), "--sample-counts", str(counts),
                                     "--aov", "albedo", str(albedo), "--denoise-progressive", str(clean), "--dump-frames", str(frames)])
    ren, fs = _replay(rt, ctx, mesh, env, w, h, frames, ("albedo", "normal"))
    assert len(fs) == res["dispatches"] <= spp
    assert [f.cameraParams.accumCount for f in fs] == list(range(len(fs)))
    params = T.AdaptiveParams(thr, 0.1, mn, spp)
    ctx.ray_counts(reset=True)
    active = []
    for k, f in enumerate(fs):
        ren.dispatch(f)
        if (k + 1) % every == 0:
            active.append(ren.adaptive_update(params))
    ctx.status()
    assert res["primary_rays"] == ctx.ray_counts().primary < len(fs) * w * h, "converged pixels were skipped"
    if len(fs) < spp:
        assert active[-1] == 0, "the run stops when no pixel is active"
    np.testing.assert_array_equal(read_pfm(out), ren.image()[..., :3])
    n, _ = ren.sample_counts()
    np.testing.assert_array_equal(read_pfm(counts), np.repeat(n.astype(np.float32)[..., None], 3, axis=-1))
    assert n.min() >= mn and n.max() <= len(fs) and n.min() < n.max()
    np.testing.assert_array_equal(read_exr(albedo), ren.aov("albedo"))
    assert rel_rmse(read_pfm(clean), ren.denoise()[..., :3]) <= 1e-6
    print(f"dispatches {len(fs)} of {spp}, mean spp {n.mean():.1f}, primary rays {res['primary_rays']}")


def test_camera_move_restarts_the_counts(host_built, tmp_path, ctx, rt):  # noqa: F811
    """Every --orbit frame moves the camera, which restarts accumulation: counts and moments start again from 0, so the
    result is the last one-sample frame and every count is 1."""
    mesh, env, cmd = _scene(tmp_path)
    w, h, spp = 40, 32, 5
    out, counts, frames = tmp_path / "out.pfm", tmp_path / "n.exr", tmp_path / "frames.bin"
    _run([host_built] + cmd + ["--width", str(w), "--height", str(h), "--spp", str(spp), "--orbit", "0.5", "--adaptive", "0.1",
                               "--adaptive-every", "1", "--out", str(out), "--sample-counts", str(counts), "--dump-frames", str(frames)])
    assert np.all(read_exr(counts)[..., :3] == 1.0)
    ren, fs = _replay(rt, ctx, mesh, env, w, h, frames, ())
    assert len(fs) == spp and all(f.cameraParams.accumCount == 0 for f in fs)
    ren.dispatch(fs[-1])
    ctx.status()
    np.testing.assert_array_equal(read_pfm(out), ren.image()[..., :3])


def test_headless_adaptive_rejections(host_built, tmp_path):  # noqa: F811
    base = [EXE, "--scene", "cornell", "--width", "32", "--height", "32"]
    for extra, word in ((["--pipeline", "realtime", "--adaptive", "0.1"], "adaptive"),
                        (["--world", "2", "--rank", "0", "--comm-file", str(tmp_path / "id"), "--adaptive", "0.1"], "adaptive"),
                        (["--adaptive", "0.1", "--denoise-temporal", str(tmp_path / "c.pfm")], "adaptive"),
                        (["--adaptive"], "adaptive"),
                        (["--sample-counts", str(tmp_path / "n.pfm")], "sample-counts"),
                        (["--adaptive", "0.1", "--adaptive-every", "0"], "adaptive-every")):
        r = subprocess.run(base + extra, capture_output=True, text=True, timeout=120)
        assert r.returncode != 0 and word in r.stderr, (extra, r.stderr)
