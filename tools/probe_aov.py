#!/usr/bin/env python
"""probe_aov.py — cost of the progressive pipeline's AOV outputs (rt_set_aov_output) on the C2 workload.

Renders C2 (bunny-scale mesh, 1920x1080, 16 spp per step) with no AOV bound and with all six bound, alternating the two
arms, and reports device-timed ms per step for each arm and the overhead.  Both arms render the same frames into their own
beauty buffer, which must come out bit-identical.  Prints the GPU name and power limit beside the numbers.

  python tools/probe_aov.py [--reps 5] [--warmup 2] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from dxrexperiments_b200 import scenes, types as T  # noqa: E402


def gpu_info():
    """Read-only query of the card the numbers come from."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        name, power = (s.strip() for s in out[0].split(","))
        return name, power
    except Exception as e:  # the timing does not depend on it; say what is missing
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5, help="timed steps per arm (alternating), at least 5")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if args.reps < 5:
        raise SystemExit("--reps must be at least 5")
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("probe_aov.py: no CUDA device")

    from dxrexperiments_b200 import rtcore as rt
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = rt.Context(0, stream=stream.cuda_stream)
    wl = scenes.workload("C2")
    W, H, SPP = wl.width, wl.height, wl.spp
    env = scenes.sky_cube(64)
    jit = scenes.jitter_sequence(wl.setup.seed, SPP, W, H)
    frames = [scenes.make_frame(wl.setup, W, H, frame_count=s, accum_count=s, jitter=jit[s]) for s in range(SPP)]
    arms = {"no_aov": rt.Renderer(ctx, wl.meshes, wl.transforms, wl.materials, env, rt.PROGRESSIVE, W, H),
            "all_aovs": rt.Renderer(ctx, wl.meshes, wl.transforms, wl.materials, env, rt.PROGRESSIVE, W, H, aovs=T.AOV_NAMES)}

    def step(r):
        for f in frames:
            r.dispatch(f)

    for _ in range(args.warmup):
        for r in arms.values():
            step(r)
    ctx.status()
    times = {k: [] for k in arms}
    for _ in range(args.reps):
        for name, r in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record(stream)
            step(r)
            e1.record(stream)
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1))
    ctx.status()
    identical = bool(np.array_equal(arms["no_aov"].image(0), arms["all_aovs"].image(0)))
    gpu, power = gpu_info()
    base, aov = float(np.median(times["no_aov"])), float(np.median(times["all_aovs"]))
    res = {"probe": "aov_overhead", "workload": wl.description, "gpu": gpu, "power_limit": power, "spp_per_step": SPP,
           "reps": args.reps, "ms_per_step": times, "median_ms_no_aov": base, "median_ms_all_aovs": aov,
           "overhead_pct": 100.0 * (aov - base) / base, "beauty_bit_identical": identical,
           "aov_bytes_per_step_estimate": 6 * 32 * W * H * SPP}
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()
    if not identical:
        raise SystemExit("beauty buffers of the two arms differ")


if __name__ == "__main__":
    main()
