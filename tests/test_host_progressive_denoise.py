"""dxr_headless --denoise-progressive: the beauty output filtered by rt_denoise_progressive through the C++ host
(ProgressiveRaytracingPipeline::denoise), held to the CPU restatement applied to the same run's output files."""
import os
import subprocess

import numpy as np
import pytest

import progressive_denoise_reference as pdr
from conftest import rel_rmse
from test_host_aov import EXE, HOST, _gpu_count
from test_host_cpp import read_exr, read_pfm

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def host_built():
    subprocess.run(["make", "-C", HOST, "-s"], check=True)
    return EXE


def _rgba(rgb):
    return np.concatenate([rgb, np.ones(rgb.shape[:2] + (1,), np.float32)], axis=-1)


def _filtered_files(out, albedo, normal):
    return pdr.denoise(_rgba(read_pfm(out)), _rgba(read_pfm(albedo)), read_exr(normal), *pdr.default_params())


def test_headless_denoise_progressive_equals_the_filter_of_its_outputs(host_built, tmp_path):
    out, albedo, normal, clean = (tmp_path / n for n in ("out.pfm", "albedo.pfm", "normal.exr", "clean.exr"))
    cmd = [EXE, "--scene", "cornell", "--pipeline", "progressive", "--width", "96", "--height", "64", "--spp", "3", "--seed", "7",
           "--out", str(out), "--aov", "albedo", str(albedo), "--aov", "normal", str(normal), "--denoise-progressive", str(clean)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = read_exr(clean)
    assert np.all(got[..., 3] == 1.0)
    assert rel_rmse(got, _filtered_files(out, albedo, normal)) <= 1e-5
    # without --aov files the flag still enables its guides; PFM by extension
    pfm = tmp_path / "clean.pfm"
    r = subprocess.run(cmd[:cmd.index("--out")] + ["--denoise-progressive", str(pfm)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    np.testing.assert_array_equal(read_pfm(pfm), got[..., :3])


def test_headless_denoise_progressive_rejects_realtime(host_built, tmp_path):
    base = [EXE, "--scene", "cornell", "--width", "32", "--height", "32"]
    for extra in (["--pipeline", "realtime", "--denoise-progressive", str(tmp_path / "c.pfm")], ["--denoise-progressive"]):
        r = subprocess.run(base + extra, capture_output=True, text=True)
        assert r.returncode != 0 and "denoise-progressive" in r.stderr, (extra, r.stderr)


@pytest.mark.parametrize("strip_groups", [1, 2])
def test_headless_denoise_progressive_world_2(host_built, tmp_path, strip_groups):
    world = 2
    n = _gpu_count()
    if n < world:
        pytest.skip(f"needs {world} GPUs, this box has {n}")
    common = [EXE, "--scene", "cornell", "--pipeline", "progressive", "--width", "160", "--height", "120", "--spp", "6", "--seed", "11"]
    out, albedo, normal, clean, idf = (tmp_path / n for n in ("out.pfm", "albedo.pfm", "normal.exr", "clean.exr", "id"))
    procs = [subprocess.Popen(common + ["--out", str(out), "--aov", "albedo", str(albedo), "--aov", "normal", str(normal),
                                        "--denoise-progressive", str(clean), "--world", str(world), "--rank", str(k), "--comm-file", str(idf),
                                        "--strip-groups", str(strip_groups), "--strip-rows", "8"],
                              stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for k in range(world)]
    outs = [p.communicate(timeout=300) for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert rel_rmse(read_exr(clean), _filtered_files(out, albedo, normal)) <= 1e-5
