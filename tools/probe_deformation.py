#!/usr/bin/env python
"""probe_deformation.py — cost of the previous-position AOV's deformation term and of Renderer.set_vertices on C2.

C2's scene (the bunny-scale mesh of 81 920 triangles plus its 2-triangle ground, 1920x1080, the scene bench.py renders)
as one-sample frames under a static camera, instance 0 translated by 0.05 along x (Renderer.set_transforms) and its
mesh sheared by (0.5, 0, 0.25) at the top (scenes.sheared_positions, Renderer.set_vertices), accumulation off, the albedo,
normal, position and previous-position AOVs bound.  Times a 1-spp dispatch with the deformation descriptors bound against
the same renderer with only the motion bound, the two alternating.  Then times one set_vertices (vertex upload, BLAS refit,
TLAS rebuild, descriptor upload; it ends in a device synchronise) with a host clock.  CUDA events for the dispatches:
warmed up, each rep a batch of calls, the median of the reps.  Prints the GPU name and power limit beside the numbers.

  python tools/probe_deformation.py [--reps 20] [--calls 3] [--out result.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from dxrexperiments_b200 import scenes, types as T  # noqa: E402
from probe_aov import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20, help="timed batches per measurement, at least 5")
    ap.add_argument("--calls", type=int, default=3, help="dispatches per timed batch")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if args.reps < 5:
        raise SystemExit("--reps must be at least 5")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("probe_deformation.py: no CUDA device")

    from dxrexperiments_b200 import rtcore as rt
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = rt.Context(0, stream=stream.cuda_stream)
    wl = scenes.workload("C2")
    W, H = wl.width, wl.height
    env = scenes.sky_cube(64)
    frame = scenes.make_frame(wl.setup, W, H, 0, 0, jitter=scenes.jitter_sequence(wl.setup.seed, 1, W, H)[0])
    mesh = wl.meshes[0]
    rest, normals = mesh.vertices["position"], mesh.vertices["normal"]

    def sheared(s):
        return scenes.sheared_positions(rest, s * np.array([0.5, 0.0, 0.25]))
    moved = np.array(wl.transforms, np.float32).reshape(len(wl.transforms), 12).copy()
    moved[0, 3] += np.float32(0.05)
    aovs = ("albedo", "normal", T.AOV_POSITION_NAME, T.AOV_PREVIOUS_POSITION_NAME)
    rs = []
    for _ in range(2):
        r = rt.Renderer(ctx, wl.meshes, wl.transforms, wl.materials, env, rt.PROGRESSIVE, W, H, aovs=aovs,
                        instance_mesh=wl.instance_mesh, deforming=(0,))
        r.set_transforms(moved)
        r.set_vertices(0, sheared(1.0), normals)
        rs.append(r)
    deformed, motion_only = rs
    motion_only._deform_buf = None  # the same geometry and motion, the deformation descriptors unbound

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(n):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    res = {"probe": "deformation", "workload": wl.description + "; one sample per frame, instance 0 moving and its mesh deforming, "
           "static camera", "gpu": None, "power_limit": None, "width": W, "height": H, "triangles": int(mesh.num_triangles)}
    with_d, without = [], []
    for r in rs:
        for _ in range(3):
            r.dispatch(frame)
    for _ in range(args.reps):
        with_d.append(timed(lambda: deformed.dispatch(frame), args.calls))
        without.append(timed(lambda: motion_only.dispatch(frame), args.calls))
    ctx.status()
    a, b = deformed.aov(T.AOV_PREVIOUS_POSITION_NAME), motion_only.aov(T.AOV_PREVIOUS_POSITION_NAME)
    res["dispatch_1spp"] = {"median_ms_motion_only": float(np.median(without)), "median_ms_with_deformation": float(np.median(with_d)),
                            "deformation_cost_ms": float(np.median(with_d) - np.median(without)),
                            "min_ms_motion_only": float(np.min(without)), "min_ms_with_deformation": float(np.min(with_d)),
                            "pixels_moved_by_the_deformation": int((np.abs(a - b).max(axis=-1) > 0).sum())}
    # ---- one set_vertices: it synchronises (uploads, refit, TLAS build), so a host clock around it times the device work
    ms = []
    for k in range(args.reps + 2):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        deformed.set_vertices(0, sheared(1.0 + 0.01 * k), normals)
        ms.append((time.perf_counter() - t0) * 1e3)
    ms = ms[2:]
    res["set_vertices"] = {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms))}
    ctx.status()
    res["gpu"], res["power_limit"] = gpu_info()
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
