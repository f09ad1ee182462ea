"""dxr_headless --aov: the progressive pipeline's AOV outputs through the C++ host (RaytracingPipelineBase::enableAov)."""
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import rel_rmse
from dxrexperiments_b200 import scenes, types as T
from test_host_cpp import read_exr, read_pfm, write_obj

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "dxrexperiments_b200", "host")
EXE = os.path.join(HOST, "dxr_headless")


@pytest.fixture(scope="module")
def host_built():
    subprocess.run(["make", "-C", HOST, "-s"], check=True)
    return EXE


def _gpu_count():
    try:
        out = subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True, timeout=30).stdout
        return sum(1 for l in out.splitlines() if l.startswith("GPU "))
    except Exception:
        return 0


def test_headless_aov_files(host_built, tmp_path, ctx, rt):
    mesh = scenes.cornell_box()
    obj = tmp_path / "cornell.obj"
    write_obj(obj, mesh)
    env = scenes.sky_cube(16)
    envf = tmp_path / "env.bin"
    env.astype("<f4").tofile(envf)
    w, h, spp = 96, 64, 3
    cmd = [EXE, "--model", str(obj), "--pipeline", "progressive", "--width", str(w), "--height", str(h), "--spp", str(spp), "--seed", "7",
           "--eye", "0", "0", "3.5", "--at", "0", "0", "0", "--light-pos", "0", "0.5", "0", "--env-raw", str(envf), "16"]
    plain, out, albedo, normal, frames = (tmp_path / n for n in ("plain.pfm", "out.pfm", "albedo.pfm", "normal.exr", "frames.bin"))
    r = subprocess.run(cmd + ["--out", str(plain)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run(cmd + ["--out", str(out), "--aov", "albedo", str(albedo), "--aov", "normal", str(normal), "--dump-frames", str(frames)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert json.loads(r.stdout.strip().splitlines()[-1])["frames"] == spp
    np.testing.assert_array_equal(read_pfm(out), read_pfm(plain))  # the AOVs leave the beauty output alone

    raw = np.fromfile(frames, dtype=np.uint8).reshape(spp, 188)
    ren = rt.Renderer(ctx, [mesh], [scenes.IDENTITY_3X4], [scenes.make_material()], env, rt.PROGRESSIVE, w, h, aovs=("albedo", "normal"))
    for s in range(spp):
        ren.dispatch(T.PerFrameConstants.from_buffer_copy(raw[s].tobytes()))
    ctx.status()
    assert rel_rmse(read_pfm(albedo), ren.aov("albedo")[..., :3]) <= 1e-6
    n = read_exr(normal)
    assert rel_rmse(n, ren.aov("normal")) <= 1e-6
    assert 0.0 < n[..., 3].mean() <= 1.0  # alpha = the fraction of samples that hit


def test_headless_aov_rejects_bad_arguments(host_built, tmp_path):
    base = [EXE, "--scene", "cornell", "--width", "32", "--height", "32"]
    for extra in (["--pipeline", "realtime", "--aov", "albedo", str(tmp_path / "a.pfm")],
                  ["--aov", "depth", str(tmp_path / "d.pfm")], ["--aov", "albedo"]):
        r = subprocess.run(base + extra, capture_output=True, text=True)
        assert r.returncode != 0 and "aov" in r.stderr.lower(), (extra, r.stderr)


@pytest.mark.parametrize("strip_groups", [1, 2])
def test_headless_aovs_world_2_equal_single_process(host_built, tmp_path, strip_groups):
    world = 2
    n = _gpu_count()
    if n < world:
        pytest.skip(f"needs {world} GPUs, this box has {n}")
    common = [EXE, "--scene", "cornell", "--pipeline", "progressive", "--width", "160", "--height", "120", "--spp", "6", "--seed", "11"]
    names = ("direct", "indirect-specular", "normal")
    single = {a: tmp_path / f"single_{a}.pfm" for a in names}
    r = subprocess.run(common + sum((["--aov", a, str(p)] for a, p in single.items()), []), capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    multi, idf = {a: tmp_path / f"multi_{a}.pfm" for a in names}, tmp_path / "id"
    procs = [subprocess.Popen(common + sum((["--aov", a, str(p)] for a, p in multi.items()), []) +
                              ["--world", str(world), "--rank", str(k), "--comm-file", str(idf), "--strip-groups", str(strip_groups), "--strip-rows", "8"],
                              stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for k in range(world)]
    outs = [p.communicate(timeout=300) for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    for a in names:
        assert rel_rmse(read_pfm(multi[a]), read_pfm(single[a])) <= 1e-6, a
