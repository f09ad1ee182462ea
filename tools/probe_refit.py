#!/usr/bin/env python
"""probe_refit.py — time of the fit paths the build benchmark does not cover: PERFORM_UPDATE refits of a bottom-level
structure and top-level builds and updates (CUDA events around each call, median over --reps after two warm-up calls).
For A/B runs, select the library with RT_CORE_LIB=path/to/librt_core.so.

  python tools/probe_refit.py --refit 1000000,10000000 --tlas 512,50000
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from dxrexperiments_b200 import scenes, types as T  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--refit", default="1000000,10000000", help="comma list of triangle counts")
    ap.add_argument("--tlas", default="512,50000", help="comma list of instance counts")
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    import torch

    from dxrexperiments_b200 import rtcore as rt
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = rt.Context(0, stream=stream.cuda_stream)
    lib = os.environ.get("RT_CORE_LIB", "default")
    smi = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    card = {"gpu": torch.cuda.get_device_name(0), "power_limit": smi.stdout.strip() or "unknown"}

    def timed(call):
        times = []
        for r in range(args.reps + 2):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            call()
            e1.record(stream)
            torch.cuda.synchronize()
            if r >= 2:
                times.append(e0.elapsed_time(e1))
        return float(np.median(times)), float(np.min(times))

    upd = T.BUILD_FLAG_ALLOW_UPDATE
    for n in [int(x) for x in args.refit.split(",") if x]:
        mesh = scenes.triangle_soup(n)
        vb, ib = ctx.upload(mesh.vertices), ctx.upload(mesh.indices)
        desc = (T.GeometryDesc * 1)()
        desc[0].vertex_buffer, desc[0].vertex_count, desc[0].vertex_stride_bytes = vb.ptr, mesh.vertices.shape[0], 24
        desc[0].index_buffer, desc[0].index_count, desc[0].index_format = ib.ptr, mesh.indices.size, 32
        desc[0].flags = T.GEOMETRY_FLAG_OPAQUE
        info = T.PrebuildInfo()
        rt.check(rt.lib.rt_blas_prebuild(ctx.handle, desc, 1, upd, C.byref(info)))
        scr, res = ctx.alloc(info.scratch_bytes), ctx.alloc(info.result_bytes)
        rt.check(rt.lib.rt_blas_build(ctx.handle, desc, 1, upd, scr.ptr, scr.nbytes, res.ptr, res.nbytes))
        ms, lo = timed(lambda: rt.check(rt.lib.rt_blas_build(ctx.handle, desc, 1, upd | T.BUILD_FLAG_PERFORM_UPDATE, scr.ptr, scr.nbytes,
                                                              res.ptr, res.nbytes)))
        ctx.status()
        print(json.dumps({"probe": "blas_refit", "triangles": n, "ms": ms, "min_ms": lo, "lib": lib, **card}), flush=True)
        del vb, ib, scr, res

    blas = ctx.build_blas_from_mesh(scenes.icosphere(2))
    for n in [int(x) for x in args.tlas.split(",") if x]:
        descs = ctx.upload(rt._instance_descs_bytes([blas] * n, scenes.random_rigid_transforms(n, seed=n)))
        info = T.PrebuildInfo()
        rt.check(rt.lib.rt_tlas_prebuild(ctx.handle, n, upd, C.byref(info)))
        scr, res = ctx.alloc(info.scratch_bytes), ctx.alloc(info.result_bytes)
        for kind, flags in (("tlas_build", upd), ("tlas_update", upd | T.BUILD_FLAG_PERFORM_UPDATE)):
            ms, lo = timed(lambda: rt.check(rt.lib.rt_tlas_build(ctx.handle, descs.ptr, n, flags, scr.ptr, scr.nbytes, res.ptr, res.nbytes)))
            ctx.status()
            print(json.dumps({"probe": kind, "instances": n, "ms": ms, "min_ms": lo, "lib": lib, **card}), flush=True)


if __name__ == "__main__":
    main()
