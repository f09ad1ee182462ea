#!/usr/bin/env python
"""probe_adaptive.py — cost and gain of adaptive sampling (rt_set_adaptive_sampling, rt_adaptive_update).

1. C2 (bunny-scale mesh, 1920x1080, the scene bench.py renders): a 1-spp dispatch with adaptive sampling bound and every
   pixel active against the plain dispatch, the two alternating.
2. rt_adaptive_update at 1920x1080, ms per call.
3. Cornell and C2 at 1920x1080, jitter-free: the rays traced and the GPU time (dispatches plus updates) to bring the rel
   RMSE against a 1024-spp reference down to that of a uniform 64-spp frame, adaptive (threshold --threshold, floor 0.1,
   min 8, an update every 4 dispatches) against uniform.  The error is checked every 4 dispatches, outside the timing.
CUDA events, warmed up; medians of the reps.  Prints the GPU name and power limit beside the numbers.

  python tools/probe_adaptive.py [--reps 20] [--threshold 0.03] [--out result.json]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from dxrexperiments_b200 import scenes, types as T  # noqa: E402
from probe_aov import gpu_info  # noqa: E402


def rel_rmse(a, b):
    a, b = a[..., :3].astype(np.float64), b[..., :3].astype(np.float64)
    return float(np.sqrt(np.mean((a - b) ** 2)) / np.sqrt(np.mean(b ** 2)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20, help="timed batches per measurement, at least 5")
    ap.add_argument("--threshold", type=float, default=0.03)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.reps < 5:
        raise SystemExit("--reps must be at least 5")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("probe_adaptive.py: no CUDA device")
    from dxrexperiments_b200 import rtcore as rt
    from helpers import cornell_case
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = rt.Context(0, stream=stream.cuda_stream)

    def timed(fn, n=1):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(n):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    wl = scenes.workload("C2")
    W, H = wl.width, wl.height
    env = scenes.sky_cube(64)
    res = {"probe": "adaptive", "workload": wl.description, "gpu": None, "power_limit": None, "width": W, "height": H}

    def renderer(scene, adaptive):
        if scene == "C2":
            return rt.Renderer(ctx, wl.meshes, wl.transforms, wl.materials, env, rt.PROGRESSIVE, W, H, instance_mesh=wl.instance_mesh,
                               adaptive=adaptive), wl.setup
        c = cornell_case()
        return rt.Renderer(ctx, c.meshes, c.transforms, c.materials, c.env, rt.PROGRESSIVE, W, H, adaptive=adaptive), c.setup

    # ---- 1. all-active adaptive 1-spp dispatch against the plain one
    plain, setup = renderer("C2", False)
    adapt, _ = renderer("C2", True)
    f0 = scenes.make_frame(setup, W, H, 0, 0)
    for r in (plain, adapt, plain, adapt):
        r.dispatch(f0)
    a_ms, p_ms = [], []
    for _ in range(args.reps):
        adapt.reset_adaptive()  # outside the timing: every pixel stays active with n_p = 0
        a_ms.append(timed(lambda: adapt.dispatch(f0)))
        p_ms.append(timed(lambda: plain.dispatch(f0)))
    res["dispatch_1spp_C2"] = {"plain_median_ms": float(np.median(p_ms)), "adaptive_all_active_median_ms": float(np.median(a_ms)),
                               "adaptive_cost_ms": float(np.median(a_ms) - np.median(p_ms))}
    # ---- 2. the update
    counts, moments, active = adapt.adaptive
    prm = T.adaptive_defaults()
    u_ms = [timed(lambda: ctx.adaptive_update(moments, counts, W, H, prm, active), 10) for _ in range(args.reps)]
    res["adaptive_update_ms"] = {"median": float(np.median(u_ms)), "min": float(np.min(u_ms)), "max": float(np.max(u_ms))}
    del plain, adapt
    ctx.status()
    # ---- 3. rays and time to a fixed error
    for scene in ("cornell", "C2"):
        ref_r, setup = renderer(scene, False)
        for k in range(1024):
            ref_r.dispatch(scenes.make_frame(setup, W, H, k, k, jitter=(0.0, 0.0)))
        ref = ref_r.image()
        del ref_r
        uni, _ = renderer(scene, False)
        for k in range(64):
            uni.dispatch(scenes.make_frame(setup, W, H, 5000 + k, k, jitter=(0.0, 0.0)))
        target = rel_rmse(uni.image(), ref)
        out = {"target_rel_rmse": target}
        for mode in ("uniform", "adaptive"):
            r, _ = renderer(scene, mode == "adaptive")
            prm = T.AdaptiveParams(args.threshold, 0.1, 8, 1024)
            ms, k, err, left = 0.0, 0, None, W * H
            ctx.ray_counts(reset=True)
            while k < 1024:
                def step():
                    for j in range(4):
                        r.dispatch(scenes.make_frame(setup, W, H, 5000 + k + j, k + j, jitter=(0.0, 0.0)))
                    if mode == "adaptive":
                        ctx.adaptive_update(r.adaptive[1], r.adaptive[0], W, H, prm, r.adaptive[2])
                ms += timed(step)
                k += 4
                err = rel_rmse(r.image(), ref)
                if mode == "adaptive":
                    left = int(r.adaptive[2].download(np.uint32, 1)[0])
                if err <= target or left == 0:
                    break
            c = ctx.ray_counts()
            out[mode] = {"dispatches": k, "rel_rmse": err, "reached": err <= target, "gpu_ms": ms,
                         "rays": int(c.primary + c.secondary + c.shadow), "primary_rays": int(c.primary), "active_left": left}
            del r
        out["ray_ratio_adaptive_over_uniform"] = out["adaptive"]["rays"] / out["uniform"]["rays"]
        out["time_ratio_adaptive_over_uniform"] = out["adaptive"]["gpu_ms"] / out["uniform"]["gpu_ms"]
        res["fixed_error_" + scene] = out
        ctx.status()
    res["gpu"], res["power_limit"] = gpu_info()
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
