#!/usr/bin/env python
"""probe_instance_motion.py — cost of the previous-position AOV and of rt_denoise_temporal_motion on the C2 workload.

C2's scene (bunny-scale mesh, 1920x1080, the scene bench.py renders) as one-sample frames under a static camera, with
instance 0 translated by 0.05 along x per frame (Renderer.set_transforms), accumulation off, the albedo, normal and
position AOVs bound.  Times a 1-spp dispatch with and without the previous-position AOV (and its instance motion) bound,
the two alternating.  After two filtered frames (so that the history is real), times rt_denoise_temporal_motion and
rt_denoise_temporal at 0 ... 5 iterations on the same frame, alternating.  CUDA events: warmed up, each rep a batch of
calls, the median of the reps.  Prints the GPU name and power limit beside the numbers.

  python tools/probe_instance_motion.py [--reps 20] [--calls 10] [--out result.json]
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
        raise SystemExit("probe_instance_motion.py: no CUDA device")

    from dxrexperiments_b200 import rtcore as rt
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = rt.Context(0, stream=stream.cuda_stream)
    wl = scenes.workload("C2")
    W, H = wl.width, wl.height
    env = scenes.sky_cube(64)
    jit = scenes.jitter_sequence(wl.setup.seed, 3, W, H)
    frames = [scenes.make_frame(wl.setup, W, H, f, 0, jitter=jit[f]) for f in range(3)]

    def moved(f):
        t = np.array(wl.transforms, np.float32).reshape(len(wl.transforms), 12).copy()
        t[0, 3] += np.float32(0.05 * f)
        return t
    guides = ("albedo", "normal", T.AOV_POSITION_NAME)
    PREV = T.AOV_PREVIOUS_POSITION_NAME
    kw = dict(instance_mesh=wl.instance_mesh)
    r = rt.Renderer(ctx, wl.meshes, wl.transforms, wl.materials, env, rt.PROGRESSIVE, W, H, aovs=guides + (PREV,), **kw)
    r2 = rt.Renderer(ctx, wl.meshes, wl.transforms, wl.materials, env, rt.PROGRESSIVE, W, H, aovs=guides, **kw)
    r.set_transforms(moved(1))
    r2.set_transforms(moved(1))

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(n):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    res = {"probe": "instance_motion", "workload": wl.description + "; one sample per frame, instance 0 moving, static camera",
           "gpu": None, "power_limit": None, "width": W, "height": H, "instances": len(wl.transforms), "dispatch_1spp": {},
           "temporal_motion": {}, "temporal": {}}
    # ---- the previous-position AOV's cost on a 1-spp dispatch (accumCount 0), alternating with and without it
    with_prev, without = [], []
    for rr in (r, r2):
        rr.dispatch(frames[0])
    for _ in range(args.reps):
        with_prev.append(timed(lambda: r.dispatch(frames[0]), 3))
        without.append(timed(lambda: r2.dispatch(frames[0]), 3))
    res["dispatch_1spp"] = {"median_ms_albedo_normal_position": float(np.median(without)),
                            "median_ms_with_previous_position": float(np.median(with_prev)),
                            "previous_position_cost_ms": float(np.median(with_prev) - np.median(without))}
    # ---- two filtered frames, then the third frame is the one every call filters, with the second's history
    for k, f in enumerate(frames):
        r.set_transforms(moved(k + 2))
        r.dispatch(f)
        if k < 2:
            r.denoise_temporal()
    prev_cam = r._prev_camera
    prev, hist, tmp, out = r._temporal
    ctx.status()
    ins = (r.out[0].ptr, r.aovs["albedo"].ptr, r.aovs["normal"].ptr, r.aovs[T.AOV_POSITION_NAME].ptr)
    for it in range(6):
        tp = T.TemporalDenoiseParams(T.ProgressiveDenoiseParams(it, 7, 4.0, 0.1), 0.2, 0.2, 0.9, 0.02)

        def motion():
            rt.check(rt.lib.rt_denoise_temporal_motion(ctx.handle, *ins, r.aovs[PREV].ptr, C.byref(prev_cam), prev.ptr, hist.ptr,
                                                       tmp.ptr, out.ptr, W, H, C.byref(tp)))

        def temporal():
            rt.check(rt.lib.rt_denoise_temporal(ctx.handle, *ins, C.byref(prev_cam), prev.ptr, hist.ptr, tmp.ptr, out.ptr, W, H,
                                                C.byref(tp)))
        for fn in (motion, temporal):
            for _ in range(3):
                fn()
        ms = {"temporal_motion": [], "temporal": []}
        for _ in range(args.reps):
            ms["temporal_motion"].append(timed(motion, args.calls))
            ms["temporal"].append(timed(temporal, args.calls))
        for name, v in ms.items():
            res[name][it] = {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v))}
    ctx.status()
    motion()
    ctx.status()
    n = hist.download(np.float32, count=W * H * 4).reshape(H, W, 4)[..., 3]
    res["history_kept_share_with_motion"] = float((n > 1).mean())
    temporal()
    ctx.status()
    n = hist.download(np.float32, count=W * H * 4).reshape(H, W, 4)[..., 3]
    res["history_kept_share_without_motion"] = float((n > 1).mean())
    res["gpu"], res["power_limit"] = gpu_info()
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
