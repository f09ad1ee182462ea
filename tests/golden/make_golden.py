"""Regenerates tests/golden/*.npz from the CPU oracle.

    python tests/golden/make_golden.py [REFERENCE_CHECKOUT]

The reference cannot be executed here (Windows/D3D12), so these vectors are NOT reference outputs: they freeze the
oracle's answers (which tests/test_oracle_reference_kats.py pins against the reference's own test logic) so that
(a) a later change to the oracle cannot silently move the goalposts and (b) the GPU box — which has no
/root/reference and may have a different libm — checks the CUDA path against bytes committed to the repo.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

import oracle  # noqa: E402
from dxrexperiments_b200 import scenes, types as T  # noqa: E402
from helpers import cornell_case  # noqa: E402


def rng_kats():
    rows = []
    for v0, v1 in [(0, 0), (12345, 7), (1920 * 1080 - 1, 15), (0xFFFFFFFF, 0xFFFFFFFF)]:
        s = oracle.init_rand(v0, v1)
        vals = []
        st = s
        for _ in range(4):
            v, st = oracle.next_rand(st)
            vals.append(v)
        rows.append((v0, v1, s, vals))
    return (np.array([[r[0], r[1], r[2]] for r in rows], np.uint64), np.array([r[3] for r in rows], np.float32))


def hit_group_scene():
    """Mixed BLAS (non-opaque triangles + opaque spheres) used by the hit-group golden vectors: (mesh, aabbs, rays)."""
    from helpers import random_rays
    mesh = scenes.icosphere(2)
    rng = np.random.Generator(np.random.PCG64(321))
    c = rng.uniform(-2.5, 2.5, size=(300, 3))
    hh = rng.uniform(0.1, 0.45, size=(300, 3))
    aabbs = np.concatenate([c - hh, c + hh], axis=1).astype(np.float32)
    rays = random_rays(4096, seed=77, lo=(-4, -4, -4), hi=(4, 4, 4), tmin=1e-4)
    return mesh, aabbs, rays


HIT_GROUP_CASES = [  # (name, programs per record [geometry 0, geometry 1], ray flags)
    ("sphere", [[T.ANYHIT_NONE, T.INTERSECTION_NONE], [T.ANYHIT_NONE, T.INTERSECTION_SPHERE]], 0),
    ("cutout_box", [[T.ANYHIT_CUTOUT, T.INTERSECTION_NONE], [T.ANYHIT_ACCEPT, T.INTERSECTION_BOX]], 0),
    ("ignore_forced", [[T.ANYHIT_IGNORE, T.INTERSECTION_NONE], [T.ANYHIT_IGNORE, T.INTERSECTION_SPHERE]], T.RAY_FLAG_FORCE_NON_OPAQUE),
    ("first_hit", [[T.ANYHIT_ACCEPT, T.INTERSECTION_NONE], [T.ANYHIT_END_SEARCH, T.INTERSECTION_SPHERE]],
     T.RAY_FLAG_ACCEPT_FIRST_HIT_AND_END_SEARCH | T.RAY_FLAG_FORCE_NON_OPAQUE),
]


def hit_group_vectors(orc):
    mesh, aabbs, rays = hit_group_scene()
    blas = orc.Blas([dict(vertices=mesh.vertices, stride=24, indices=mesh.indices, flags=T.GEOMETRY_FLAG_NONE), dict(aabbs=aabbs)])
    tlas = orc.Tlas([blas], [scenes.IDENTITY_3X4], hit_groups=[0])
    out = {"blob": np.asarray(blas.blob()).copy()}
    for name, progs, flags in HIT_GROUP_CASES:
        h = tlas.trace_hit_groups(rays, progs, ray_flags=flags, geometry_multiplier=1)
        out[name + "_prim"], out[name + "_t"], out[name + "_geom"] = h["primitive_index"], h["t"], h["geometry_index"]
        out[name + "_kind"] = (h["leaf_slot"] >> 24).astype(np.uint8)
    return out


def main():
    seeds, rands = rng_kats()
    # build: a seeded soup with duplicate codes
    soup = scenes.triangle_soup(2000, seed=99, extent=50.0, edge=2.0)
    blas = oracle.Blas.from_mesh(soup)
    build = dict(aabb=blas.scene_aabb(), morton=blas.morton(), perm=blas.perm())
    # hierarchy + fitted nodes per treelet-pass count: default flags (1 pass), PREFER_FAST_BUILD (0: the plain Karras
    # tree), PREFER_FAST_TRACE (3) — FL/TreeletReorder.cpp:66-80
    for suffix, flags in (("", 0), ("_fast_build", T.BUILD_FLAG_PREFER_FAST_BUILD), ("_fast_trace", T.BUILD_FLAG_PREFER_FAST_TRACE)):
        b = oracle.Blas.from_mesh(soup, build_flags=flags)
        build["hier" + suffix] = b.hierarchy().view(np.uint32).reshape(-1, 3)
        build["nodes" + suffix] = T.parse_blas_blob(b.blob())["nodes"].view(np.uint32).reshape(-1, 8)
    np.savez_compressed(os.path.join(HERE, "build_soup2000.npz"), **build)
    # trace + render: Cornell 48x48
    case = cornell_case()
    tlas, recs = case.oracle(oracle)
    w = h = 48
    frame = scenes.make_frame(case.setup, w, h, 0, 0)
    rays = oracle.primary_rays(frame, w, h)
    hits = tlas.trace(rays, T.RAY_FLAG_CULL_BACK_FACING_TRIANGLES)
    acc = np.zeros((h, w, 4), np.float32)
    jit = scenes.jitter_sequence(5, 4, w, h)
    for s in range(4):
        oracle.render_progressive(tlas, recs, case.env, scenes.make_frame(case.setup, w, h, s, s, jitter=jit[s]), w, h, acc)
    direct, spec = oracle.render_realtime(tlas, recs, case.env, scenes.make_frame(case.setup, w, h, 3, 0, jitter=jit[0]), w, h)
    prm = T.DenoiserParams(1.0, 2.2, 1, 0, 12, 0)
    den, _ = oracle.denoise(direct, spec, prm)
    np.savez_compressed(os.path.join(HERE, "cornell48.npz"), prim=hits["primitive_index"], t=hits["t"], bary=hits["bary"],
                        progressive4=acc, direct=direct, spec=spec, denoised=den)
    np.savez_compressed(os.path.join(HERE, "rng.npz"), seeds=seeds, rands=rands)
    np.savez_compressed(os.path.join(HERE, "hitgroups_mixed.npz"), **hit_group_vectors(oracle))
    # a 192 x 128 crop of the reference's own mock denoiser inputs (src/DenoiseCompositor.cpp:52-60 loads
    # assets/textures/{DirectLighting,IndirectSpecular}.PNG, 1922 x 1126, 8-bit) around the busiest region: the repository
    # does not carry the full files, so it is rewritten only when the path of a reference checkout is given.
    tex = os.path.join(sys.argv[1], "assets", "textures") if len(sys.argv) > 1 else ""
    if tex and os.path.exists(os.path.join(tex, "DirectLighting.PNG")):
        from PIL import Image
        y0, x0, hh, ww = 128, 832, 128, 192
        d = np.asarray(Image.open(os.path.join(tex, "DirectLighting.PNG")).convert("RGBA"))[y0:y0 + hh, x0:x0 + ww]
        sp = np.asarray(Image.open(os.path.join(tex, "IndirectSpecular.PNG")).convert("RGBA"))[y0:y0 + hh, x0:x0 + ww]
        np.savez_compressed(os.path.join(HERE, "denoise_mock_crop.npz"), direct_u8=d, spec_u8=sp, origin=np.array([y0, x0]))
    print("wrote", sorted(f for f in os.listdir(HERE) if f.endswith(".npz")))


if __name__ == "__main__":
    main()
