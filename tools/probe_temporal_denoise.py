#!/usr/bin/env python
"""probe_temporal_denoise.py — cost of rt_denoise_temporal and of the position AOV on the C2 workload.

C2's scene (bunny-scale mesh, 1920x1080, the scene bench.py renders) as one-sample frames of a camera orbiting its `at`
point by 0.5 degrees per frame, accumulation off, with the albedo, normal and position AOVs bound.  After two filtered
frames (so that the history is real), times rt_denoise_temporal at 0 ... 5 iterations next to rt_denoise_progressive on the
same frame, with CUDA events: warmed up, each rep a batch of calls, the median of the reps.  Also times a 1-spp dispatch
with and without the position AOV bound (albedo and normal bound in both), the two alternating.  Prints the GPU name and
power limit beside the numbers.

  python tools/probe_temporal_denoise.py [--reps 20] [--calls 10] [--out result.json]
"""
import argparse
import ctypes as C
import dataclasses
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from dxrexperiments_b200 import scenes, types as T  # noqa: E402
from probe_aov import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20, help="timed batches per measurement, at least 5")
    ap.add_argument("--calls", type=int, default=10, help="calls per timed batch")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if args.reps < 5:
        raise SystemExit("--reps must be at least 5")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("probe_temporal_denoise.py: no CUDA device")

    from dxrexperiments_b200 import rtcore as rt
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = rt.Context(0, stream=stream.cuda_stream)
    wl = scenes.workload("C2")
    W, H = wl.width, wl.height
    env = scenes.sky_cube(64)
    jit = scenes.jitter_sequence(wl.setup.seed, 3, W, H)
    frames = [scenes.make_frame(dataclasses.replace(wl.setup, camera=scenes.orbit(wl.setup.camera, 0.5 * f)), W, H, f, 0, jitter=jit[f])
              for f in range(3)]
    guides = ("albedo", "normal", T.AOV_POSITION_NAME)
    r = rt.Renderer(ctx, wl.meshes, wl.transforms, wl.materials, env, rt.PROGRESSIVE, W, H, aovs=guides)
    r2 = rt.Renderer(ctx, wl.meshes, wl.transforms, wl.materials, env, rt.PROGRESSIVE, W, H, aovs=("albedo", "normal"))

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(n):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    res = {"probe": "temporal_denoise", "workload": wl.description + "; one sample per frame, 0.5-degree orbit", "gpu": None,
           "power_limit": None, "width": W, "height": H, "dispatch_1spp": {}, "temporal": {}, "progressive": {}}
    # ---- the position AOV's cost on a 1-spp dispatch (accumCount 0), alternating with and without it
    with_pos, without = [], []
    for rr in (r, r2):
        rr.dispatch(frames[0])
    for _ in range(args.reps):
        with_pos.append(timed(lambda: r.dispatch(frames[0]), 3))
        without.append(timed(lambda: r2.dispatch(frames[0]), 3))
    res["dispatch_1spp"] = {"median_ms_albedo_normal": float(np.median(without)),
                            "median_ms_albedo_normal_position": float(np.median(with_pos)),
                            "position_cost_ms": float(np.median(with_pos) - np.median(without))}
    # ---- two filtered frames, then the third frame is the one every call filters, with the second's history
    for f in frames[:2]:
        r.dispatch(f)
        r.denoise_temporal()
    r.dispatch(frames[2])
    prev_cam = r._prev_camera
    prev, hist, tmp, out = r._temporal
    ctx.status()
    for it in range(6):
        tp = T.TemporalDenoiseParams(T.ProgressiveDenoiseParams(it, 7, 4.0, 0.1), 0.2, 0.2, 0.9, 0.02)
        sp = tp.spatial

        def temporal():
            rt.check(rt.lib.rt_denoise_temporal(ctx.handle, r.out[0].ptr, r.aovs["albedo"].ptr, r.aovs["normal"].ptr,
                                                r.aovs[T.AOV_POSITION_NAME].ptr, C.byref(prev_cam), prev.ptr, hist.ptr, tmp.ptr,
                                                out.ptr, W, H, C.byref(tp)))

        def progressive():
            rt.check(rt.lib.rt_denoise_progressive(ctx.handle, r.out[0].ptr, r.aovs["albedo"].ptr, r.aovs["normal"].ptr, tmp.ptr,
                                                   out.ptr, W, H, C.byref(sp)))
        for name, fn in (("temporal", temporal), ("progressive", progressive)):
            for _ in range(3):
                fn()
            ms = [timed(fn, args.calls) for _ in range(args.reps)]
            res[name][it] = {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms))}
    ctx.status()
    n = hist.download(np.float32, count=W * H * 4).reshape(H, W, 4)[..., 3]
    res["history_kept_share"] = float((n > 1).mean())
    res["gpu"], res["power_limit"] = gpu_info()
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
