"""CPU-only checks of the boundary and the host logic: the C-ABI library loads and exports every symbol the
header declares, every entry point cites the reference interface it replaces, the product never touches the
oracle, scenes/frames are deterministic, and the multi-GPU sharding logic reduces to the single-GPU frame
(world_size 2, gloo)."""
import ctypes as C
import hashlib
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol(rt):
    names = rt.declared_symbols()
    assert len(names) >= 38
    for n in names:
        assert hasattr(rt.lib, n), n
    assert rt.lib.rt_version().startswith(b"rt_core")
    out = subprocess.run(["nm", "-D", "--defined-only", rt.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (rt_[a-z_0-9]+)", out))
    assert set(names) <= exported


def test_header_is_plain_c_and_cites_the_reference(tmp_path):
    hdr = open(os.path.join(ROOT, "include", "rt_core.h")).read()
    types = open(os.path.join(ROOT, "include", "rt_types.h")).read()
    for text in (hdr, types):
        code = re.sub(r"/\*.*?\*/", "", text, flags=re.S)  # declarations only
        for banned in ("torch", "at::", "std::", "cudaStream_t", "Tensor", "#include <cuda"):
            assert banned not in code, banned
    for anchor in ("RtContext.cpp:12-29", "RtModel.cpp:86-118", "RtScene.cpp:18-52", "FallbackLayer.cpp:317-338",
                   "RtBindings.cpp:100-164", "DenoiseCompositor.cpp:109-148", "UberShaderRayTracingProgram.cpp:213-272"):
        assert anchor in hdr, anchor
    # the header compiles as C99
    src = '#include "rt_core.h"\nint main(void){ rt_per_frame_constants f; (void)f; return sizeof(rt_hit) == 32 ? 0 : 1; }\n'
    exe = str(tmp_path / "rt_core_c99_check")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-x", "c", "-", "-o", exe],
                   input=src, text=True, check=True)
    assert subprocess.run([exe]).returncode == 0


def test_struct_sizes_match_the_reference_layouts():
    from dxrexperiments_b200 import types as T
    assert C.sizeof(T.PerFrameConstants) == 188   # RaytracingHlslCompat.h:79-85
    assert C.sizeof(T.MaterialParams) == 64       # 16 dwords of root constants
    assert C.sizeof(T.InstanceDesc) == 64 and T.InstanceDesc.blas.offset == 56  # RaytracingInstanceDescOffsetToPointer
    assert T.NODE_DTYPE.itemsize == 32 and T.PRIM_DTYPE.itemsize == 40 and T.META_DTYPE.itemsize == 12
    assert T.BVH_METADATA_DTYPE.itemsize == 116


def test_no_gpu_means_loud_failure_not_fallback(rt):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(rt.RtError) as e:
        rt.Context(0)
    assert "no CPU fallback" in str(e.value)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "dxrexperiments_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".hpp", "Makefile")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert not re.search(r"^\s*(import|from)\s+oracle\b", text, flags=re.M), f
                assert "liboracle" not in text and "oracle/" not in text.replace("the oracle/", ""), f


def test_scenes_are_deterministic_and_wound_outward():
    from dxrexperiments_b200 import scenes
    m = scenes.bunny_scale(3)
    h1 = hashlib.sha256(m.vertices.tobytes() + m.indices.tobytes()).hexdigest()
    m2 = scenes.bunny_scale(3)
    assert h1 == hashlib.sha256(m2.vertices.tobytes() + m2.indices.tobytes()).hexdigest()
    assert scenes.bunny_scale(6).num_triangles == 81922
    assert scenes.cornell_box().num_triangles == 36
    ico = scenes.icosphere(2)
    tri = ico.triangles().astype(np.float64)
    n = np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0])
    assert (np.einsum("ij,ij->i", n, tri.mean(1)) > 0).all()  # geometric normals point away from the solid
    soup = scenes.triangle_soup(1000, seed=1)
    assert soup.num_triangles == 1000 and np.abs(soup.vertices["position"]).max() <= 500.5
    xf = scenes.random_rigid_transforms(10, seed=10)
    R = xf.reshape(10, 3, 4)[:, :, :3]
    s = np.cbrt(np.linalg.det(R))
    np.testing.assert_allclose(np.einsum("nij,nkj->nik", R, R), (s ** 2)[:, None, None] * np.eye(3), atol=1e-4)


def test_frame_constants_follow_update():
    """calculateCameraVariables + update() (src/ProgressiveRaytracingPipeline.cpp:151-213)."""
    from dxrexperiments_b200 import scenes
    setup = scenes.FrameSetup()
    f = scenes.make_frame(setup, 1920, 1080, 5, 3, jitter=(0.25 / 1920, -0.5 / 1080))
    U, V, W = (np.array(list(x)[:3]) for x in (f.cameraParams.U, f.cameraParams.V, f.cameraParams.W))
    assert abs(np.linalg.norm(W) - 1) < 1e-6 and abs(U @ V) < 1e-6 and abs(U @ W) < 1e-6 and abs(V @ W) < 1e-6
    np.testing.assert_allclose(np.linalg.norm(V), np.tan(np.pi / 8), rtol=1e-6)          # vertical FOV pi/4
    np.testing.assert_allclose(np.linalg.norm(U) / np.linalg.norm(V), 1920 / 1080, rtol=1e-6)
    assert f.cameraParams.frameCount == 5 and f.cameraParams.accumCount == 3
    d = np.array(list(f.directionalLight.forwardDir)[:3])
    np.testing.assert_allclose(np.linalg.norm(d), np.linalg.norm([0.3, -0.2, -1.0]), rtol=1e-6)  # a rotation about Y
    assert abs(d[1] + 0.2) < 1e-7
    assert list(f.pointLight.color) == pytest.approx([0.2, 0.8, 0.6, 2.0])
    assert f.options.maxIterations == 1024 and f.options.cosineHemisphereSampling == 1
    j = scenes.jitter_sequence(1234, 16, 1920, 1080)
    assert j.shape == (16, 2) and np.abs(j[:, 0]).max() <= 0.5 / 1920 and np.abs(j[:, 1]).max() <= 0.5 / 1080


def test_sharding_plans():
    from dxrexperiments_b200 import sharding
    assert sharding.samples_for_rank(1, 4, 10) == [1, 5, 9]
    assert sum(sharding.combine_scale(r, 4, 10) for r in range(4)) == pytest.approx(1.0)
    w, h = 200, 130
    cover = np.zeros((h, w), int)
    for r in range(3):
        for x0, y0, x1, y1 in sharding.tiles_for_rank(r, 3, w, h, tile=64):
            cover[y0:y1, x0:x1] += 1
    assert (cover == 1).all()
    with pytest.raises(ValueError):
        sharding.samples_for_rank(4, 4, 10)
    # strip x sample plans: every (row, sample) is rendered exactly once, the weights of a row's owners add up to 1
    for world, spp, groups in [(1, 5, None), (2, 8, 1), (2, 8, 2), (4, 6, 2), (8, 64, None), (8, 64, 2), (8, 2, None), (6, 3, 3)]:
        h = 77
        hits = np.zeros((h, spp), int)
        wsum = np.zeros(h)
        for r in range(world):
            pl = sharding.plan(r, world, spp, strip_groups=groups, strip_rows=8)
            assert pl.strip_groups * pl.sample_groups == world
            rows = pl.rows(h)
            for smp in pl.samples:
                hits[rows, smp] += 1
            wsum[rows] += pl.weight
        assert (hits == 1).all(), (world, spp, groups)
        np.testing.assert_allclose(wsum, 1.0, rtol=1e-12)
    # realtime row bands: the cores partition the frame, the rendered rows add the filter's reach, clipped at the border
    for world, h, halo in ((1, 37, 12), (2, 1080, 12), (3, 203, 20), (8, 2160, 12), (5, 7, 3)):
        bands = [sharding.band_plan(r, world, h, halo) for r in range(world)]
        assert bands[0].y0 == 0 and bands[-1].y1 == h and all(a.y1 == b.y0 for a, b in zip(bands, bands[1:]))
        for b in bands:
            assert b.r0 == max(0, b.y0 - halo) and b.r1 == min(h, b.y1 + halo) and b.r0 <= b.y0 <= b.y1 <= b.r1
    with pytest.raises(ValueError):
        sharding.band_plan(2, 2, 100, 12)
    assert sharding.default_strip_groups(8, 64) == 1 and sharding.default_strip_groups(8, 2) == 4 and sharding.default_strip_groups(8, 1) == 8
    with pytest.raises(ValueError):
        sharding.plan(0, 4, 8, strip_groups=3)
    with pytest.raises(ValueError):
        sharding.plan(0, 4, 8, strip_groups=2, strip_rows=12)


WORKER = r'''
import os, sys
import numpy as np
import torch, torch.distributed as dist
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
import oracle
from dxrexperiments_b200 import scenes, sharding
from helpers import cornell_case
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
case = cornell_case(); tlas, recs = case.oracle(oracle)
w = h = 24; total = 6
jit = scenes.jitter_sequence(9, total, w, h)
acc = np.zeros((h, w, 4), np.float32)
plan = sharding.plan(rank, world, total, strip_groups=int(os.environ["STRIP_GROUPS"]), strip_rows=4)
for local, s in enumerate(plan.samples):
    oracle.render_progressive(tlas, recs, case.env, scenes.make_frame(case.setup, w, h, s, local, jitter=jit[s]), w, h, acc)
mine = np.zeros(h, bool); mine[plan.rows(h)] = True
acc[~mine] = 0  # a strip-interleaved dispatch leaves the other groups' rows untouched (zero)
t = torch.from_numpy(acc * np.float32(plan.weight))
dist.reduce(t, dst=0, op=dist.ReduceOp.SUM)
if rank == 0:
    ref = np.zeros((h, w, 4), np.float32)
    for s in range(total):
        oracle.render_progressive(tlas, recs, case.env, scenes.make_frame(case.setup, w, h, s, s, jitter=jit[s]), w, h, ref)
    err = float(np.abs(t.numpy() - ref).max() / ref.max())
    print("MAXREL", err)
    assert err < 1e-5, err
dist.destroy_process_group()
'''


@pytest.mark.parametrize("strip_groups", [1, 2])
def test_sample_sharded_accumulation_world2_gloo(tmp_path, strip_groups):
    """N > 1 host logic on CPU: two gloo ranks render their shard of the samples / strips (the oracle stands in for the
    renderer), weight by their share and sum-reduce; rank 0 must hold the single-process 6-spp frame."""
    script = tmp_path / "worker.py"
    script.write_text(WORKER.format(root=ROOT))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29731", OMP_NUM_THREADS="1", STRIP_GROUPS=str(strip_groups))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29731", str(script)], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "MAXREL" in r.stdout


BAND_WORKER = r'''
import os, sys
import numpy as np
import torch, torch.distributed as dist
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
import oracle
from dxrexperiments_b200 import sharding, types as T
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
w, h, k = 61, 53, 12
rng = np.random.Generator(np.random.PCG64(5))           # the same AOVs on every rank (a rank renders only its rows of them)
direct = rng.random((h, w, 4), dtype=np.float32); direct[:, : w // 3, :3] *= 0.05
spec = (rng.random((h, w, 4), dtype=np.float32) ** 3).astype(np.float32)
prm = T.DenoiserParams(1.0, 2.2, 1, 0, k, 0)
band = sharding.band_plan(rank, world, h, halo=k)
out = oracle.denoise(direct[band.r0:band.r1], spec[band.r0:band.r1], prm)
out = out[0] if isinstance(out, tuple) else out
final = np.zeros((h, w, 4), np.float32)
final[band.y0:band.y1] = out[band.y0 - band.r0: band.y1 - band.r0]  # the core rows only: halo rows are cleared
t = torch.from_numpy(final)
dist.reduce(t, dst=0, op=dist.ReduceOp.SUM)                         # rt_accum_reduce with weight 1
if rank == 0:
    ref = oracle.denoise(direct, spec, prm)
    ref = ref[0] if isinstance(ref, tuple) else ref
    assert np.array_equal(t.numpy(), ref), float(np.abs(t.numpy() - ref).max())
    print("BANDS_OK")
dist.destroy_process_group()
'''


def test_realtime_row_bands_world2_gloo(tmp_path):
    """N > 1 host logic of the band-sharded realtime frame on CPU: two gloo ranks filter their band plus the filter's reach (the
    oracle's DenoiseCompositor stands in for rt_denoise), keep their core rows and sum-reduce; rank 0 must hold the full-frame
    filter output bit for bit."""
    script = tmp_path / "band_worker.py"
    script.write_text(BAND_WORKER.format(root=ROOT))
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29733", OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29733", str(script)], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "BANDS_OK" in r.stdout


def test_python_constants_match_the_c_header():
    """The ctypes mirror (dxrexperiments_b200/types.py) and include/rt_types.h must not drift apart: every enum value the
    Python side names is parsed out of the header and compared."""
    text = open(os.path.join(ROOT, "include", "rt_types.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    header = {}
    for name, val in re.findall(r"\b(RT_[A-Z0-9_]+)\s*=\s*(0x[0-9A-Fa-f]+|\d+)", text):
        header[name] = int(val, 0)
    for name, val in re.findall(r"#define\s+(RT_[A-Z0-9_]+)\s+(0x[0-9A-Fa-f]+|\d+)[uU]?\b", text):
        header[name] = int(val, 0)
    from dxrexperiments_b200 import types as T
    checked = 0
    for py_name in dir(T):
        c_name = "RT_" + py_name
        if c_name in header and isinstance(getattr(T, py_name), int):
            assert getattr(T, py_name) == header[c_name], (py_name, getattr(T, py_name), header[c_name])
            checked += 1
    assert checked >= 30, checked
    assert T.PROCEDURAL_FLAG == header["RT_NODE_PROCEDURAL_FLAG"] and T.LEAF_FLAG == header["RT_NODE_LEAF_FLAG"]
    assert T.PRIMITIVE_TYPE_PROCEDURAL == header["RT_PRIMITIVE_TYPE_PROCEDURAL"]
    import ctypes as C
    assert C.sizeof(T.GeometryDesc) == 48  # the `type` field took the place of padding: the ABI size did not move
