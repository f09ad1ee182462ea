#!/usr/bin/env python
"""probe_progressive_denoise.py — cost of rt_denoise_progressive on the C2 workload.

Renders one 16-spp step of C2 (bunny-scale mesh, 1920x1080, the scene bench.py renders) with the albedo and normal AOVs
bound, then times the filter on those buffers with CUDA events at 1 ... 5 iterations: warmed up, each rep a batch of calls,
the median of the reps.  For scale it also times the 16-spp step itself.  Reports algorithmic bytes (48 B/pixel for the
variance pass, 64 B/pixel per iteration) over time, and prints the GPU name and power limit beside the numbers.

  python tools/probe_progressive_denoise.py [--reps 30] [--calls 10] [--out result.json]
"""
import argparse
import ctypes as C
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
    ap.add_argument("--reps", type=int, default=30, help="timed batches per iteration count, at least 5")
    ap.add_argument("--calls", type=int, default=10, help="filter calls per timed batch")
    ap.add_argument("--step-reps", type=int, default=5, help="timed 16-spp steps")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if args.reps < 5:
        raise SystemExit("--reps must be at least 5")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("probe_progressive_denoise.py: no CUDA device")

    from dxrexperiments_b200 import rtcore as rt
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = rt.Context(0, stream=stream.cuda_stream)
    wl = scenes.workload("C2")
    W, H, SPP = wl.width, wl.height, wl.spp
    env = scenes.sky_cube(64)
    jit = scenes.jitter_sequence(wl.setup.seed, SPP, W, H)
    frames = [scenes.make_frame(wl.setup, W, H, frame_count=s, accum_count=s, jitter=jit[s]) for s in range(SPP)]
    r = rt.Renderer(ctx, wl.meshes, wl.transforms, wl.materials, env, rt.PROGRESSIVE, W, H, aovs=("albedo", "normal"))

    def timed(fn, n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(n):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    def step():
        for f in frames:
            r.dispatch(f)

    step()  # warm-up, and the frame the filter is timed on
    step_ms = [timed(step, 1) for _ in range(args.step_reps)]
    # the 16-spp accumulation of the first step is the filter's input: render it again so every rep filters the same frame
    for f in frames:
        r.dispatch(f)
    clean = r.denoise()  # allocates tmp / out
    ctx.status()
    tmp, out = r._denoise_bufs
    res = {"probe": "progressive_denoise", "workload": wl.description, "gpu": None, "power_limit": None, "width": W, "height": H,
           "median_ms_16spp_step": float(np.median(step_ms)), "ms_16spp_step": step_ms, "filter": {}}
    for it in range(1, 6):
        p = T.ProgressiveDenoiseParams(it, 7, 4.0, 0.1)

        def call():
            rt.check(rt.lib.rt_denoise_progressive(ctx.handle, r.out[0].ptr, r.aovs["albedo"].ptr, r.aovs["normal"].ptr, tmp.ptr, out.ptr,
                                                   W, H, C.byref(p)))
        for _ in range(3):
            call()
        ms = [timed(call, args.calls) for _ in range(args.reps)]
        med = float(np.median(ms))
        nbytes = (48 + 64 * it) * W * H
        res["filter"][it] = {"median_ms": med, "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms)),
                             "algorithmic_bytes": nbytes, "algorithmic_GBps": nbytes / med / 1e6,
                             "share_of_16spp_step": med / res["median_ms_16spp_step"]}
    ctx.status()
    assert np.isfinite(clean).all()
    res["gpu"], res["power_limit"] = gpu_info()
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
