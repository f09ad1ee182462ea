"""The headless C++ host (DXRFramework-style classes + pipelines + dxr_headless).

CPU: the host's own logic (OBJ/PFM/DDS, shader-table packing, program validation) and loud failure without a GPU.
GPU: dxr_headless renders through RtContext / RtModel / RtScene / RtProgram / RtBindings / RaytracingPipeline and the
     DenoiseCompositor; its PFM output must match the oracle fed with the very frame constants the host produced.
"""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import rel_rmse
from dxrexperiments_b200 import scenes, types as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "dxrexperiments_b200", "host")
EXE = os.path.join(HOST, "dxr_headless")


@pytest.fixture(scope="module")
def host_built():
    subprocess.run(["make", "-C", HOST, "-s"], check=True)
    return EXE


def write_obj(path, mesh):
    with open(path, "w") as f:
        for v in mesh.vertices:
            f.write("v %.9g %.9g %.9g\n" % tuple(v["position"]))
        for v in mesh.vertices:
            f.write("vn %.9g %.9g %.9g\n" % tuple(v["normal"]))
        for a, b, c in mesh.indices.reshape(-1, 3) + 1:
            f.write(f"f {a}//{a} {b}//{b} {c}//{c}\n")


def read_pfm(path):
    with open(path, "rb") as f:
        assert f.readline().strip() == b"PF"
        w, h = (int(x) for x in f.readline().split())
        assert float(f.readline()) < 0
        data = np.frombuffer(f.read(), dtype="<f4").reshape(h, w, 3)
    return data[::-1].copy()


def test_host_selftest(host_built, tmp_path):
    r = subprocess.run([os.path.join(HOST, "host_selftest"), str(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "host selftest OK" in r.stdout


def test_headless_fails_loudly_without_gpu(host_built):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = subprocess.run([EXE, "--scene", "cornell", "--width", "32", "--height", "32"], capture_output=True, text=True)
    assert r.returncode != 0 and "no CPU fallback" in r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["progressive", "realtime"])
def test_headless_render_matches_oracle(pipeline, host_built, tmp_path, orc):
    mesh = scenes.cornell_box()
    obj = tmp_path / "cornell.obj"
    write_obj(obj, mesh)
    env = scenes.sky_cube(16)
    envf = tmp_path / "env.bin"
    env.astype("<f4").tofile(envf)
    w, h, spp = 96, 64, 3 if pipeline == "progressive" else 1
    out, out2, den, frames = (tmp_path / n for n in ("out.pfm", "out2.pfm", "den.pfm", "frames.bin"))
    cmd = [EXE, "--model", str(obj), "--pipeline", pipeline, "--width", str(w), "--height", str(h), "--spp", str(spp), "--seed", "7",
           "--eye", "0", "0", "3.5", "--at", "0", "0", "0", "--light-pos", "0", "0.5", "0", "--env-raw", str(envf), "16",
           "--out", str(out), "--dump-frames", str(frames)]
    if pipeline == "realtime":
        cmd += ["--out2", str(out2), "--denoise", str(den)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    info = json.loads(r.stdout.strip().splitlines()[-1])
    assert info["triangles"] == 36 and info["kernel_launches"] > 0 and info["core"].startswith("rt_core")

    raw = np.fromfile(frames, dtype=np.uint8).reshape(spp, 188)
    blas = orc.Blas.from_mesh(mesh)
    tlas = orc.Tlas([blas], [scenes.IDENTITY_3X4])
    recs = orc.Records([mesh], [scenes.make_material()])
    acc = np.zeros((h, w, 4), np.float32)
    for s in range(spp):
        frame = T.PerFrameConstants.from_buffer_copy(raw[s].tobytes())
        assert frame.cameraParams.frameCount == s
        assert abs(frame.cameraParams.jitters[0]) <= 0.5 / w and abs(frame.cameraParams.jitters[1]) <= 0.5 / h
        if pipeline == "progressive":
            assert frame.cameraParams.accumCount == s and frame.options.maxIterations == 1024
            orc.render_progressive(tlas, recs, env, frame, w, h, acc, threads=4)
        else:
            direct, spec = orc.render_realtime(tlas, recs, env, frame, w, h, threads=4)
    if pipeline == "progressive":
        assert rel_rmse(read_pfm(out), acc[..., :3]) <= 1e-3
    else:
        assert rel_rmse(read_pfm(out), direct[..., :3]) <= 1e-3
        assert rel_rmse(read_pfm(out2), spec[..., :3]) <= 1e-3
        ref, _ = orc.denoise(direct, spec, T.DenoiserParams(1.0, 2.2, 1, 0, 12, 0))
        assert rel_rmse(read_pfm(den), ref[..., :3]) <= 1e-3


@pytest.mark.gpu
def test_headless_builtin_scenes(host_built, tmp_path):
    for scene in ("cornell", "triangle"):
        out = tmp_path / f"{scene}.pfm"
        r = subprocess.run([EXE, "--scene", scene, "--width", "64", "--height", "48", "--spp", "2", "--out", str(out)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        img = read_pfm(out)
        assert img.shape == (48, 64, 3) and np.isfinite(img).all() and img.max() > 0


# The part of Assimp's C API (assimp/cimport.h, postprocess.h, scene.h; flag values as Assimp defines them) that
# RtModelAssimp.cpp uses, so that the loader compiles without an Assimp installation.
ASSIMP_HEADERS = {
    "scene.h": r"""
#pragma once
struct aiVector3D { float x, y, z; };
struct aiFace { unsigned int mNumIndices = 0; unsigned int *mIndices = nullptr; };
struct aiMesh {
    unsigned int mNumVertices = 0;
    aiVector3D *mVertices = nullptr;
    aiVector3D *mNormals = nullptr;
    unsigned int mNumFaces = 0;
    aiFace *mFaces = nullptr;
    bool HasNormals() const { return mNormals != nullptr && mNumVertices > 0; }
};
struct aiScene { unsigned int mNumMeshes; aiMesh **mMeshes; };
""",
    "postprocess.h": r"""
#pragma once
enum aiPostProcessSteps {
    aiProcess_JoinIdenticalVertices = 0x2, aiProcess_Triangulate = 0x8, aiProcess_GenSmoothNormals = 0x40,
    aiProcess_PreTransformVertices = 0x100, aiProcess_FlipUVs = 0x800000,
};
""",
    "cimport.h": r"""
#pragma once
#include "scene.h"
extern "C" const aiScene *aiImportFile(const char *pFile, unsigned int pFlags);
extern "C" void aiReleaseImport(const aiScene *pScene);
""",
}
FAKE_ASSIMP = r"""
// A stand-in for libassimp (the reference vendors headers + Windows binaries only): aiImportFile hands out a fixed
// two-mesh scene so that RtModel::loadWithAssimp's merge logic (libs/DXRFramework/RtModel.cpp:35-58) can be exercised.
#include <assimp/cimport.h>
#include <assimp/postprocess.h>
#include <assimp/scene.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "RtModel.h"
static unsigned gFlags = 0, gReleased = 0;
extern "C" const aiScene *aiImportFile(const char *path, unsigned int flags) {
    gFlags = flags;
    if (std::strcmp(path, "missing.fbx") == 0) return nullptr;
    aiScene *s = static_cast<aiScene *>(std::calloc(1, sizeof(aiScene)));  // aiScene's constructor lives in libassimp
    s->mNumMeshes = 2;
    s->mMeshes = new aiMesh *[2];
    aiMesh *a = new aiMesh();  // 3 vertices with normals, 1 triangle
    a->mNumVertices = 3;
    a->mVertices = new aiVector3D[3]{{0, 0, 0}, {1, 0, 0}, {0, 1, 0}};
    a->mNormals = new aiVector3D[3]{{0, 0, 1}, {0, 0, 1}, {0, 0, 1}};
    a->mNumFaces = 1;
    a->mFaces = new aiFace[1];
    a->mFaces[0].mNumIndices = 3;
    a->mFaces[0].mIndices = new unsigned[3]{0, 1, 2};
    aiMesh *b = new aiMesh();  // 4 vertices without normals, 2 triangles and a stray line
    b->mNumVertices = 4;
    b->mVertices = new aiVector3D[4]{{0, 0, 5}, {1, 0, 5}, {1, 1, 5}, {0, 1, 5}};
    b->mNumFaces = 3;
    b->mFaces = new aiFace[3];
    b->mFaces[0].mNumIndices = 3, b->mFaces[0].mIndices = new unsigned[3]{0, 1, 2};
    b->mFaces[1].mNumIndices = 2, b->mFaces[1].mIndices = new unsigned[2]{0, 1};
    b->mFaces[2].mNumIndices = 3, b->mFaces[2].mIndices = new unsigned[3]{0, 2, 3};
    s->mMeshes[0] = a, s->mMeshes[1] = b;
    return s;
}
extern "C" void aiReleaseImport(const aiScene *) { ++gReleased; }
// the inline destructors of aiScene / aiMesh / aiFace are enough; nothing else of libassimp is referenced
#define CHECK(c) do { if (!(c)) { std::fprintf(stderr, "FAILED line %d: %s\n", __LINE__, #c); return 1; } } while (0)
int main() {
    using namespace DXRFramework;
    std::vector<Vertex> v;
    std::vector<uint32_t> idx;
    CHECK(RtModel::loadWithAssimp("two_meshes.fbx", v, idx));
    const unsigned want = aiProcess_Triangulate | aiProcess_GenSmoothNormals | aiProcess_FlipUVs | aiProcess_JoinIdenticalVertices | aiProcess_PreTransformVertices;
    CHECK(gFlags == want && gReleased == 1);
    CHECK(v.size() == 7 && idx.size() == 9);
    CHECK(idx[0] == 0 && idx[1] == 1 && idx[2] == 2);
    CHECK(idx[3] == 3 && idx[4] == 4 && idx[5] == 5 && idx[6] == 3 && idx[7] == 5 && idx[8] == 6);  // per-mesh vertex offset
    CHECK(v[0].normal.z == 1.0f && v[3].normal.x == 0.0f && v[3].normal.y == 0.0f && v[3].normal.z == 0.0f && v[5].position.z == 5.0f);
    CHECK(!RtModel::loadWithAssimp("missing.fbx", v, idx));
    std::puts("assimp path OK");
    return 0;
}
"""


def test_assimp_loader_merges_meshes(tmp_path):
    """The RT_HAVE_ASSIMP branch (RtModelAssimp.cpp) built against ASSIMP_HEADERS, linked with a stand-in aiImportFile:
    flags, per-mesh merge, missing normals, non-triangle faces, failure path."""
    include = tmp_path / "include"
    (include / "assimp").mkdir(parents=True)
    for name, text in ASSIMP_HEADERS.items():
        (include / "assimp" / name).write_text(text)
    src = tmp_path / "fake_assimp_main.cpp"
    src.write_text(FAKE_ASSIMP)
    exe = tmp_path / "assimp_test"
    cmd = ["g++", "-std=c++17", "-O1", "-DRT_HAVE_ASSIMP=1", "-I", str(include), "-I", os.path.join(HOST, "DXRFramework"),
           str(src), os.path.join(HOST, "DXRFramework", "RtModelAssimp.cpp"), "-o", str(exe)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and "assimp path OK" in r.stdout, r.stderr


def read_exr(path):
    """Minimal reader of the uncompressed scan-line RGBA files ImageIO::writeEXR produces (an independent parser)."""
    d = open(path, "rb").read()
    assert int.from_bytes(d[0:4], "little") == 20000630 and d[4] == 2
    p, attrs = 8, {}
    while d[p] != 0:
        e = d.index(b"\0", p); name = d[p:e].decode(); p = e + 1
        e = d.index(b"\0", p); typ = d[p:e].decode(); p = e + 1
        size = int.from_bytes(d[p:p + 4], "little"); p += 4
        attrs[name] = (typ, d[p:p + size]); p += size
    p += 1
    x0, y0, x1, y1 = np.frombuffer(attrs["dataWindow"][1], "<i4")
    w, h = x1 - x0 + 1, y1 - y0 + 1
    assert attrs["compression"][1] == b"\0" and attrs["lineOrder"][1] == b"\0"
    ch, q, names, ptype = attrs["channels"][1], 0, [], None
    while ch[q] != 0:
        e = ch.index(b"\0", q); names.append(ch[q:e].decode()); q = e + 1
        ptype = int.from_bytes(ch[q:q + 4], "little"); q += 16
    assert names == ["A", "B", "G", "R"]
    dt = {1: "<f2", 2: "<f4"}[ptype]
    offs = np.frombuffer(d[p:p + 8 * h], "<u8")
    img = np.zeros((h, w, 4), np.float32)
    for y in range(h):
        o = int(offs[y])
        yy, size = np.frombuffer(d[o:o + 8], "<i4")
        planes = np.frombuffer(d[o + 8:o + 8 + size], dt).reshape(4, w).astype(np.float32)
        img[yy - y0] = planes[::-1].T  # A,B,G,R -> R,G,B,A
    return img


@pytest.mark.gpu
def test_host_hit_groups_with_intersection_shaders(host_built):
    """RtProgram::Desc::addHitGroup(idx, closestHit, anyHit, intersection) + RtModel::createProcedural + RtContext::traceRays."""
    r = subprocess.run([os.path.join(HOST, "host_gputest")], capture_output=True, text=True)
    assert r.returncode == 0 and "host gputest OK" in r.stdout, r.stderr


@pytest.mark.gpu
def test_headless_exr_output_equals_pfm(host_built, tmp_path):
    pfm, exr, hexr = tmp_path / "a.pfm", tmp_path / "a.exr", tmp_path / "h.exr"
    base = [EXE, "--scene", "cornell", "--width", "80", "--height", "56", "--spp", "2"]
    assert subprocess.run(base + ["--out", str(pfm), "--exr", str(exr)], capture_output=True).returncode == 0
    assert subprocess.run(base + ["--exr", str(hexr), "--exr-half"], capture_output=True).returncode == 0
    a, e, hh = read_pfm(pfm), read_exr(exr), read_exr(hexr)
    np.testing.assert_array_equal(e[..., :3], a)                       # fp32 EXR = the accumulation buffer, bit for bit
    assert (e[..., 3] == 1.0).all()
    np.testing.assert_array_equal(hh[..., :3], a.astype(np.float16).astype(np.float32))  # HALF = R16G16B16A16_FLOAT rounding


@pytest.mark.gpu
@pytest.mark.parametrize("world,strip_groups,pipeline", [(2, 1, "progressive"), (2, 2, "progressive"), (2, 2, "realtime")])
def test_headless_multi_gpu_frame_equals_single_gpu_frame(host_built, tmp_path, world, strip_groups, pipeline):
    """One dxr_headless process per GPU (NCCL inside librt_core, id through a file): the reduced frame on rank 0 equals the
    frame one GPU renders, up to fp32 summation order."""
    try:
        n = sum(1 for l in subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True).stdout.splitlines() if l.startswith("GPU "))
    except Exception:
        n = 0
    if n < world:
        pytest.skip(f"needs {world} GPUs, this box has {n}")
    spp = 6 if pipeline == "progressive" else 1
    if pipeline == "realtime" and strip_groups == 1:
        pytest.skip("one sample cannot be split by sample index")
    common = [EXE, "--scene", "cornell", "--pipeline", pipeline, "--width", "160", "--height", "120", "--spp", str(spp), "--seed", "11"]
    single = tmp_path / "single.pfm"
    assert subprocess.run(common + ["--out", str(single)], capture_output=True).returncode == 0
    multi, idf = tmp_path / "multi.pfm", tmp_path / "id"
    procs = [subprocess.Popen(common + ["--out", str(multi), "--world", str(world), "--rank", str(r), "--comm-file", str(idf),
                                        "--strip-groups", str(strip_groups), "--strip-rows", "8"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
             for r in range(world)]
    outs = [p.communicate(timeout=300) for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    a, b = read_pfm(single), read_pfm(multi)
    assert rel_rmse(b, a) <= 1e-6
    info = json.loads(outs[0][0].strip().splitlines()[-1])
    assert info["world"] == world and info["strip_groups"] == strip_groups


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4])
def test_headless_band_sharded_realtime_frame_equals_single_gpu_frame(host_built, tmp_path, world):
    """--band-shard: every dxr_headless process renders AND filters its row band of a realtime frame (plus the filter's reach),
    RtContext::reduceAccumulation composites the filtered bands with weight 1: the frame on rank 0 is the frame one GPU renders
    and filters, bit for bit (SURVEY.md 8e-ii)."""
    try:
        n = sum(1 for l in subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True).stdout.splitlines() if l.startswith("GPU "))
    except Exception:
        n = 0
    if n < world:
        pytest.skip(f"needs {world} GPUs, this box has {n}")
    common = [EXE, "--scene", "cornell", "--pipeline", "realtime", "--width", "200", "--height", "123", "--spp", "1", "--seed", "5"]
    single = tmp_path / "single.pfm"
    r = subprocess.run(common + ["--denoise", str(single)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    multi, idf = tmp_path / "multi.pfm", tmp_path / "id"
    procs = [subprocess.Popen(common + ["--denoise", str(multi), "--world", str(world), "--rank", str(k), "--comm-file", str(idf), "--band-shard"],
                              stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for k in range(world)]
    outs = [p.communicate(timeout=300) for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    np.testing.assert_array_equal(read_pfm(multi), read_pfm(single))


def write_pfm(path, rgb):
    h, w = rgb.shape[:2]
    with open(path, "wb") as f:
        f.write(b"PF\n%d %d\n-1.0\n" % (w, h))
        f.write(np.ascontiguousarray(rgb[::-1, :, :3], "<f4").tobytes())


@pytest.mark.gpu
def test_denoise_compositor_mock_resources_with_the_reference_inputs(host_built, tmp_path, orc):
    """DenoiseCompositor::setMockResources + dispatch with null SRVs (src/DenoiseCompositor.cpp:52-60, 113-116), fed with the
    committed crop of the reference's own mock inputs (DirectLighting.PNG / IndirectSpecular.PNG)."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "denoise_mock_crop.npz"))
    direct = g["direct_u8"].astype(np.float32) / np.float32(255.0)
    spec = g["spec_u8"].astype(np.float32) / np.float32(255.0)
    dp, sp, out = tmp_path / "direct.pfm", tmp_path / "spec.pfm", tmp_path / "out.pfm"
    write_pfm(dp, direct), write_pfm(sp, spec)
    r = subprocess.run([EXE, "--denoise-mock", str(dp), str(sp), "--denoise", str(out)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert json.loads(r.stdout.strip().splitlines()[-1])["denoise_mock"] is True
    d4 = np.ones(direct.shape[:2] + (4,), np.float32); d4[..., :3] = direct[..., :3]
    s4 = np.ones_like(d4); s4[..., :3] = spec[..., :3]
    want, _ = orc.denoise(d4, s4, T.DenoiserParams(1.0, 2.2, 1, 0, 12, 0))
    got = read_pfm(out)
    ok = np.isfinite(want[..., :3]).all(axis=-1)
    np.testing.assert_allclose(got[ok], want[..., :3][ok], rtol=1e-5, atol=1e-6)
