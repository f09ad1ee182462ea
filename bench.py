#!/usr/bin/env python
"""bench.py — the driver's measurement contract for the B200 ray-tracing core.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one process per GPU under torchrun)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's algorithm on the host CPU (oracle port)

Workload (BASELINE.json configs[1], "C2"): the bunny-scale synthetic mesh (displaced icosphere, 81 922 triangles)
at 1920x1080, 16 spp of the progressive pipeline.  One STEP = one 16-spp progressive frame = 16 DispatchRays.
Metric: Mrays/s = all rays actually traced (primary + incoherent secondary + shadow, counted on the device) per
second of device time, whole job over all ranks.  The same line carries `build` (LBVH build Mtri/s on a 10 M-triangle
soup, the second half of BASELINE.json's metric).  `--config C3|C4|C5` measures the other BASELINE configs the same
way (C5: realtime pipeline + denoise, reported as per-frame latency); they are extra lines, not the driver's.

N > 1: the frame shards by SAMPLE INDEX (SURVEY.md 8e): rank r renders samples r, r+N, ... with frameCount = the global
sample index, every rank holds a replicated BVH, and one NCCL reduce (rt_accum_reduce, inside librt_core; each rank's
weight applied in the reduction) sums the accumulation buffers onto rank 0.  Per-GPU work of the headline is fixed (16 spp
each), so its scaling is "weak"; the reduce is inside the timed region.

Every run ALSO emits `strong`: ONE fixed C3 frame (3840x2160, 64 spp total) sharded over the N ranks by sample index and by
interleaved screen strips, timed from "scene in pinned host memory" to "frame in rank 0's pinned host memory" (H2D,
replicated BLAS+TLAS build, the rank's dispatches, the NCCL reduce, ONE D2H on the root).  time_to_frame_ms at N = 1, 2, 4, 8
is the north star's strong-scaling number; `target_scene` is the >= 1 Grays/s incoherent-ray target on the 1.31 M-triangle
scene; `incoherent_mrays_per_s` pulls BASELINE.json's "Mrays/s (incoherent, 1080p)" to the top level.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from dxrexperiments_b200 import scenes, types as T  # noqa: E402

METRIC = "Mrays/s"
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md, used only if MEASURED_PEAKS.json is absent


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2", choices=["C2", "C3", "C4", "C5", "C1M"])
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--spp", type=int, default=None)
    ap.add_argument("--build-tris", type=int, default=10_000_000, help="triangle soup size of the `build` measurement (0 = skip)")
    ap.add_argument("--subdiv", type=int, default=6, help="icosphere subdivisions of the bunny-scale mesh (6 -> 81 920 tris)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-denoise", action="store_true", help="skip the DenoiseCompositor kernel measurement")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling block (fixed C3 4K 64-spp frame over N ranks)")
    ap.add_argument("--strong-spp", type=int, default=64)
    ap.add_argument("--strong-config", default="C3", choices=["C2", "C3", "C4", "C1M"])
    ap.add_argument("--strong-strip-groups", type=int, default=None,
                    help="strip groups of the strong-scaling shard plan (default: sample sharding first, strips when samples run out)")
    ap.add_argument("--strong-reps", type=int, default=2)
    ap.add_argument("--strong-depth", type=int, default=2, choices=[1, 2],
                    help="MAX_RADIANCE_RAY_DEPTH of the strong-scaling frame (BASELINE config 3 is '2-bounce'; the reference's shaders are 1)")
    ap.add_argument("--radiance-depth", type=int, default=1, choices=[1, 2], help="MAX_RADIANCE_RAY_DEPTH of the headline workload (1 = reference)")
    ap.add_argument("--no-target-scene", action="store_true", help="skip the 1.31 M-triangle incoherent-ray target measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame buffers of the last timed step to DIR/<name>.npy (float32; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA path computed (--impl ours)")
    return args


def load_workload(args):
    wl = scenes.workload(args.config, args.subdiv)
    wl.width, wl.height, wl.spp = args.width or wl.width, args.height or wl.height, args.spp or wl.spp
    args.width, args.height, args.spp = wl.width, wl.height, wl.spp
    return wl


def workload_config(args, wl):
    return {
        "workload": wl.description, "width": wl.width, "height": wl.height, "spp_per_step": wl.spp,
        "triangles": wl.num_triangles, "instances": len(wl.transforms), "max_radiance_ray_depth": getattr(args, "radiance_depth", 1),
        "l2": "per-frame ray queues (~0.45 KB/pixel, ~0.9 GB per 1080p frame) exceed the 126 MB L2 and are rewritten "
              "every frame; the traversal structure of C2/C3 stays L1/L2-resident by design",
    }


def frame_for(setup, args, jitters, sample_global, sample_local):
    return scenes.make_frame(setup, args.width, args.height, frame_count=sample_global, accum_count=sample_local,
                             jitter=jitters[sample_global % len(jitters)])


# ---------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- oracle scene (CPU arm)
def oracle_scene(wl):
    """The workload's scene in the CPU oracle (the reference's algorithm restated; test infrastructure)."""
    import oracle
    blases = [oracle.Blas.from_mesh(m) for m in wl.meshes]
    tlas = oracle.Tlas([blases[k] for k in wl.instance_mesh], wl.transforms)
    recs = oracle.Records([wl.meshes[k] for k in wl.instance_mesh], [wl.materials[k] for k in wl.instance_mesh])
    return oracle, tlas, recs, blases


def oracle_frame(orc, tlas, recs, env, wl, frame, acc, cores, counts):
    if wl.realtime:
        d, s = orc.render_realtime(tlas, recs, env, frame, wl.width, wl.height, threads=cores, counts=counts)
        orc.denoise(d, s, denoiser_params(), threads=cores)
    else:
        orc.render_progressive(tlas, recs, env, frame, wl.width, wl.height, acc, threads=cores, counts=counts)


def denoiser_params():
    p = T.DenoiserParams()  # src/DenoiseCompositor.cpp:45-50
    p.exposure, p.gamma, p.tonemap, p.gammaCorrect, p.maxKernelSize, p.debugVisualize = 1.0, 2.2, 1, 0, 12, 0
    return p


# ---------------------------------------------------------------------------------------------- reference arm
def run_reference(args):
    """The reference's algorithm on the host CPU: the oracle port (there is no oracle/_ref — the reference is
    Windows/D3D12-only), all host threads, each step = 1 spp of the same frame (a bounded sample)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    wl = load_workload(args)
    cores = os.cpu_count() or 1
    env = scenes.sky_cube(64)
    import oracle
    cflags = oracle.use_native()
    orc, tlas, recs, _keep = oracle_scene(wl)
    jit = scenes.jitter_sequence(wl.setup.seed, 1024, wl.width, wl.height)
    acc = np.zeros((wl.height, wl.width, 4), np.float32)

    def step(i, counts):
        oracle_frame(orc, tlas, recs, env, wl, frame_for(wl.setup, args, jit, i, 0), acc, cores, counts)

    for i in range(args.warmup):
        step(i, None)
    counts = T.RayCounts()
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(args.warmup + i, counts)
    dt = time.perf_counter() - t0
    rays = counts.primary + counts.secondary + counts.shadow
    mrays = rays / dt / 1e6
    sample = (f"{args.steps} x 1 spp of the {wl.width}x{wl.height} frame ({rays} rays), {cores} threads, row-parallel, "
              f"oracle port compiled {cflags}")
    metric, value, hib = metric_of(wl, mrays, dt / args.steps * 1e3)
    out = {"impl": "reference", "metric": metric, "value": value, "unit": metric, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": hib, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, wl),
           "cpu_baseline": {"value": value, "unit": metric, "cores": cores, "kind": "port", "sample": sample},
           "e2e": {"value": value, "unit": metric, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))
    return 0


def metric_of(wl, mrays, ms_per_step):
    """C2-C4: Mrays/s (higher is better).  C5: per-frame latency of realtime dispatch + denoise (lower is better)."""
    if wl.realtime:
        return "ms/frame (realtime 1 spp + denoise)", ms_per_step, False
    return METRIC, mrays, True


# ---------------------------------------------------------------------------------------------- our arm
class TorchBuffer:
    """A torch CUDA tensor exposed to the C ABI as a raw device pointer (torch = device memory plumbing)."""

    def __init__(self, tensor):
        self.tensor = tensor
        self.ptr = tensor.data_ptr()
        self.nbytes = tensor.numel() * tensor.element_size()


def run_ours(args):
    import torch
    import torch.distributed as dist

    from dxrexperiments_b200 import rtcore as rt

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — rt_core has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = rt.Context(local_rank, stream=stream.cuda_stream)

    wl = load_workload(args)
    W, H, SPP = wl.width, wl.height, wl.spp
    setup = wl.setup
    env = scenes.sky_cube(64)
    jit = scenes.jitter_sequence(setup.seed, 1024, W, H)
    ctx.set_render_options(args.radiance_depth, False)
    n_out = 2 if wl.realtime else 1
    outs = [torch.zeros(H * W * 4, dtype=torch.float32, device="cuda") for _ in range(n_out)]
    out_t = outs[0]
    renderer = rt.Renderer(ctx, wl.meshes, wl.transforms, wl.materials, env, rt.REALTIME if wl.realtime else rt.PROGRESSIVE, W, H,
                           outputs=[TorchBuffer(t) for t in outs], instance_mesh=wl.instance_mesh)
    dn = None
    if wl.realtime:
        dn = {"tmp": torch.empty_like(out_t), "out": torch.empty_like(out_t), "params": denoiser_params()}

    def barrier():
        if world > 1:
            dist.barrier()

    comm = make_comm(rt, ctx, torch, dist, world, rank) if world > 1 else None
    reduced_t = torch.zeros_like(out_t) if (world > 1 and rank == 0) else None

    def step(step_index):
        # rank r renders global samples r, r + world, ...; RNG is a pure function of (pixel, frameCount)
        for s in range(SPP):
            renderer.dispatch(frame_for(setup, args, jit, s * world + rank, s))
            if dn:  # DenoiseCompositor::dispatch on the two AOVs of this frame
                rt.check(rt.lib.rt_denoise(ctx.handle, outs[0].data_ptr(), outs[1].data_ptr(), dn["tmp"].data_ptr(), dn["out"].data_ptr(),
                                           W, H, C.byref(dn["params"])))
        if world > 1:  # the path's one collective, inside the product: weight 1/world applied in the NCCL reduction
            comm.reduce(out_t.data_ptr(), reduced_t.data_ptr() if rank == 0 else None, out_t.numel(), 1.0 / world, root=0)

    for i in range(args.warmup):
        step(i)
    ctx.status()

    # ---- headline: K steps, device timed, barrier + synchronize on both sides, max over ranks
    ctx.ray_counts(reset=True)
    launches0 = ctx.launches()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    torch.cuda.synchronize()
    e0.record(stream)
    for i in range(args.steps):
        step(i)
    e1.record(stream)
    torch.cuda.synchronize()
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:  # before the measurements below dispatch into the same buffers again
        frame = reduced_t if world > 1 else out_t
        named = {"direct": frame, "indirect_specular": outs[1], "denoised": dn["out"]} if wl.realtime else {"accumulation": frame}
        dump_outputs(args.dump_outputs, {k: v.cpu().numpy() for k, v in named.items()}, W, H)
    clock_info = clocks.stop() if rank == 0 else None
    launches = ctx.launches() - launches0  # this rank's own kernels; NCCL's reduce kernels are not counted
    rc = ctx.ray_counts(reset=True)
    rays = np.array([rc.primary, rc.secondary, rc.shadow], dtype=np.float64)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    r = torch.tensor(rays, dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(r, op=dist.ReduceOp.SUM)
    ms = float(t.item())
    rays = r.cpu().numpy()
    mrays = rays.sum() / (ms * 1e-3) / 1e6
    metric, value, hib = metric_of(wl, mrays, ms / args.steps)

    # ---- e2e: the same step through the C ABI with HOST buffers (pinned), copies inside the timed region
    e2e = None
    if not args.no_e2e:
        e2e = measure_e2e(args, wl, ctx, rt, torch, dist, stream, env, jit, world, rank, comm)

    # ---- strong scaling: ONE fixed 4K 64-spp C3 frame over the N ranks, host scene -> host frame on the root
    strong = None
    if not args.no_strong:
        strong = measure_strong(args, ctx, rt, torch, dist, stream, world, rank, comm)

    # ---- roofline of the dominant kernel (rank 0: a single-GPU kernel property)
    roofline, stages = None, None
    if rank == 0:
        roofline, stages = measure_roofline(args, ctx, renderer, setup, jit, world, rank)

    build = None
    if rank == 0 and world == 1 and args.build_tris > 0:
        build = measure_build(args, ctx, rt, torch, stream)

    denoise = None
    if rank == 0 and world == 1 and not args.no_denoise:
        denoise = measure_denoise(args, ctx, rt, torch, stream)

    target = None
    if rank == 0 and world == 1 and not args.no_target_scene and args.config == "C2":
        target = measure_target_scene(args, ctx, rt, torch)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = measure_cpu_baseline(args, wl, env, jit)

    ctx.status()
    if rank == 0:
        out = {"metric": metric, "value": value, "unit": metric, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": ms / args.steps, "higher_is_better": hib, "scaling": "weak", "vs_baseline": None,
               "dtype": "f32", "data": "synthetic", "config": workload_config(args, wl), "mrays_per_s": mrays,
               "rays_per_step": {"primary": rays[0] / args.steps, "secondary_incoherent": rays[1] / args.steps,
                                 "shadow": rays[2] / args.steps},
               "e2e": e2e, "gpu_launches": int(launches), "clocks": clock_info, "roofline": roofline, "stages": stages,
               "incoherent_mrays_per_s": incoherent_summary(wl, stages, target), "strong": strong, "target_scene": target,
               "build": build, "denoise": denoise, "cpu_baseline": cpu_baseline,
               "parallelism": f"sample-index sharding x{world}, replicated BVH, 1 NCCL reduce/frame (rt_accum_reduce)" if world > 1 else "single GPU"}
        print(json.dumps(out))
    if comm:
        comm.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


DUMP_LIMIT_BYTES = 64 * 2**20


def dump_outputs(path, arrays, W, H):
    """Writes each RGBA float32 frame of `arrays` to path/<name>.npy: the whole (H, W, 4) frame when all of them fit in
    DUMP_LIMIT_BYTES, else the same fixed sample of pixels from each, an (n, 4) array whose rows are the pixels
    np.sort(np.random.Generator(np.random.PCG64(0)).choice(H * W, n, replace=False)) in row-major order."""
    os.makedirs(path, exist_ok=True)
    frames = {k: np.ascontiguousarray(v, np.float32).reshape(H * W, 4) for k, v in arrays.items()}
    pix = None
    if sum(v.nbytes for v in frames.values()) > DUMP_LIMIT_BYTES:
        n = (DUMP_LIMIT_BYTES - 1024 * len(frames)) // (16 * len(frames))  # room for the .npy headers
        pix = np.sort(np.random.Generator(np.random.PCG64(0)).choice(H * W, n, replace=False))
    for k, v in frames.items():
        np.save(os.path.join(path, k + ".npy"), v.reshape(H, W, 4) if pix is None else v[pix])


def make_comm(rt, ctx, torch, dist, world, rank):
    """rt_comm over NCCL inside librt_core; torch.distributed only carries rank 0's 128-byte unique id."""
    def exchange(uid):
        box = [uid]
        dist.broadcast_object_list(box, src=0)
        return box[0]
    return rt.Comm(ctx, world, rank, exchange)


def incoherent_summary(wl, stages, target):
    """BASELINE.json's metric is "Mrays/s (incoherent, 1080p)": the incoherent secondary rays alone (cosine-hemisphere and
    Phong-lobe bounces, k_trace_persistent<0>), CUDA-event timed around their kernel, for the headline workload and for the
    north star's 1 M-triangle target scene."""
    out = {"definition": "incoherent secondary rays traced / CUDA-event time of their traversal kernel (stage-timed dispatches)"}
    if stages:
        for k, v in stages.items():
            if k.startswith("secondary_incoherent"):
                out[wl.name] = v["mrays_per_s"]
    if target:
        out["C1M"] = target["incoherent_mrays_per_s"]
        out["target_ge_1000_on_1M_triangles"] = bool(target["incoherent_mrays_per_s"] >= 1000.0)
    return out


def measure_e2e(args, wl, ctx, rt, torch, dist, stream, env, jit, world, rank, comm=None):
    """Step through the reference-facing C ABI starting from HOST memory: pinned VB/IB/instance descs -> device,
    BLAS + TLAS builds, the step's dispatches (+ denoise for C5), accumulated frame -> pinned host."""
    W, H, SPP = wl.width, wl.height, wl.spp
    n_inst = len(wl.transforms)
    host, dev, descs, binfo, bscr, bres = [], [], [], [], [], []
    for m in wl.meshes:
        vb_h = torch.from_numpy(m.vertices.view(np.uint8).reshape(-1).copy()).pin_memory()
        ib_h = torch.from_numpy(m.indices.view(np.uint8).reshape(-1).copy()).pin_memory()
        vb_d, ib_d = torch.empty_like(vb_h, device="cuda"), torch.empty_like(ib_h, device="cuda")
        host.append((vb_h, ib_h))
        dev.append((vb_d, ib_d))
        d = (T.GeometryDesc * 1)()
        d[0].vertex_buffer, d[0].vertex_count, d[0].vertex_stride_bytes = vb_d.data_ptr(), m.vertices.shape[0], 24
        d[0].index_buffer, d[0].index_count, d[0].index_format = ib_d.data_ptr(), m.indices.size, 32
        d[0].flags = T.GEOMETRY_FLAG_OPAQUE
        info = T.PrebuildInfo()
        rt.check(rt.lib.rt_blas_prebuild(ctx.handle, d, 1, 0, C.byref(info)))
        descs.append(d)
        bscr.append(torch.empty(info.scratch_bytes, dtype=torch.uint8, device="cuda"))
        bres.append(torch.empty(info.result_bytes, dtype=torch.uint8, device="cuda"))
    tinfo = T.PrebuildInfo()
    rt.check(rt.lib.rt_tlas_prebuild(ctx.handle, n_inst, 0, C.byref(tinfo)))
    tscr = torch.empty(tinfo.scratch_bytes, dtype=torch.uint8, device="cuda")
    tres = torch.empty(tinfo.result_bytes, dtype=torch.uint8, device="cuda")
    inst = (T.InstanceDesc * n_inst)()
    for i, (k, xf) in enumerate(zip(wl.instance_mesh, wl.transforms)):
        inst[i].transform[:] = np.asarray(xf, np.float32).reshape(12).tolist()
        inst[i].instance_id_and_mask = (i & 0xFFFFFF) | (0xFF << 24)
        inst[i].hit_group_and_flags = 2 * i  # InstanceContributionToHitGroupIndex = i * hitGroupCount (RtScene.cpp:29)
        inst[i].blas = bres[k].data_ptr()
    inst_h = torch.from_numpy(np.frombuffer(bytes(inst), dtype=np.uint8).copy()).pin_memory()
    inst_d = torch.empty_like(inst_h, device="cuda")
    env_d = torch.from_numpy(np.ascontiguousarray(env, np.float32).reshape(-1)).cuda()
    prog = rt.Program(ctx, rt.REALTIME if wl.realtime else rt.PROGRESSIVE)
    for i, k in enumerate(wl.instance_mesh):
        for ray_type in range(2):
            rt.check(rt.lib.rt_bindings_set_hit_record(prog.handle, ray_type, i, dev[k][0].data_ptr(), dev[k][1].data_ptr(),
                                                       C.byref(wl.materials[k])))
    rt.check(rt.lib.rt_bindings_set_miss_record(prog.handle, 0, env_d.data_ptr(), env.shape[1]))
    n_out = 2 if wl.realtime else 1
    outs = [torch.zeros(H * W * 4, dtype=torch.float32, device="cuda") for _ in range(n_out)]
    result_t = outs[0]
    dn_tmp = dn_out = None
    if wl.realtime:
        dn_tmp, dn_out = torch.empty_like(outs[0]), torch.empty_like(outs[0])
        result_t = dn_out
    dparams = denoiser_params()
    img_h = torch.empty(H * W * 4, dtype=torch.float32).pin_memory() if rank == 0 else None  # only the root holds the frame
    reduced_t = torch.zeros_like(result_t) if (world > 1 and rank == 0) else None

    def step(i):
        for (vb_h, ib_h), (vb_d, ib_d) in zip(host, dev):
            vb_d.copy_(vb_h, non_blocking=True)
            ib_d.copy_(ib_h, non_blocking=True)
        inst_d.copy_(inst_h, non_blocking=True)
        for d, sc, rs in zip(descs, bscr, bres):
            rt.check(rt.lib.rt_blas_build(ctx.handle, d, 1, 0, sc.data_ptr(), sc.numel(), rs.data_ptr(), rs.numel()))
        rt.check(rt.lib.rt_tlas_build(ctx.handle, inst_d.data_ptr(), n_inst, 0, tscr.data_ptr(), tscr.numel(), tres.data_ptr(), tres.numel()))
        rt.check(rt.lib.rt_set_tlas(ctx.handle, tres.data_ptr()))
        for slot, o in enumerate(outs):
            rt.check(rt.lib.rt_set_output(ctx.handle, slot, o.data_ptr(), 16 * W))
        for s in range(SPP):
            f = frame_for(wl.setup, args, jit, s * world + rank, s)
            rt.check(rt.lib.rt_set_frame_constants(ctx.handle, C.byref(f)))
            rt.check(rt.lib.rt_dispatch_rays(ctx.handle, prog.handle, W, H, 3))
            if wl.realtime:
                rt.check(rt.lib.rt_denoise(ctx.handle, outs[0].data_ptr(), outs[1].data_ptr(), dn_tmp.data_ptr(), dn_out.data_ptr(), W, H,
                                           C.byref(dparams)))
        if world > 1:
            comm.reduce(result_t.data_ptr(), reduced_t.data_ptr() if rank == 0 else None, result_t.numel(), 1.0 / world, root=0)
        if rank == 0:
            img_h.copy_(reduced_t if world > 1 else result_t, non_blocking=True)

    for i in range(max(1, min(args.warmup, 2))):
        step(i)
    ctx.ray_counts(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0.record(stream)
    for i in range(args.steps):
        step(i)
    e1.record(stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    rc = ctx.ray_counts(reset=True)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    r = torch.tensor([float(rc.primary + rc.secondary + rc.shadow)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(r, op=dist.ReduceOp.SUM)
    if rank == 0:
        assert float(img_h.sum()) > 0.0 and bool(torch.isfinite(img_h).all())
    ms = float(t.item())
    metric, value, _ = metric_of(wl, float(r.item()) / (ms * 1e-3) / 1e6, ms / args.steps)
    h2d = sum(int(a.numel() + b.numel()) for a, b in host) + int(inst_h.numel())
    return {"value": value, "unit": metric, "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": int(H * W * 16),
            "ms_per_step": ms / args.steps,
            "includes": "pinned H2D of VB/IB/instance descs, BLAS+TLAS build, the step's dispatches"
                        + (" + denoise" if wl.realtime else "") + (", rt_accum_reduce onto rank 0" if world > 1 else "")
                        + ", D2H of the frame (root only)"}


def measure_strong(args, ctx, rt, torch, dist, stream, world, rank, comm):
    """The north star's strong-scaling number: ONE fixed progressive frame (default C3: 3840x2160, 64 spp in total) split
    across the N ranks by sample index and by interleaved screen strips (sharding.plan), replicated BVH.  Timed region, per
    rank, on the device: pinned-host scene -> device, BLAS + TLAS build, this rank's dispatches, rt_accum_reduce, and on
    the root the D2H of the finished frame into pinned memory.  time_to_frame = max over ranks."""
    from dxrexperiments_b200 import sharding
    wl = scenes.workload(args.strong_config)
    W, H, SPP = wl.width, wl.height, args.strong_spp
    plan = sharding.plan(rank, world, SPP, strip_groups=args.strong_strip_groups, strip_rows=32)
    env = scenes.sky_cube(64)
    jit = scenes.jitter_sequence(wl.setup.seed, max(SPP, 1), W, H)
    n_inst = len(wl.transforms)
    host, dev, descs, bscr, bres = [], [], [], [], []
    for m in wl.meshes:
        vb_h = torch.from_numpy(m.vertices.view(np.uint8).reshape(-1).copy()).pin_memory()
        ib_h = torch.from_numpy(m.indices.view(np.uint8).reshape(-1).copy()).pin_memory()
        vb_d, ib_d = torch.empty_like(vb_h, device="cuda"), torch.empty_like(ib_h, device="cuda")
        host.append((vb_h, ib_h))
        dev.append((vb_d, ib_d))
        d = (T.GeometryDesc * 1)()
        d[0].vertex_buffer, d[0].vertex_count, d[0].vertex_stride_bytes = vb_d.data_ptr(), m.vertices.shape[0], 24
        d[0].index_buffer, d[0].index_count, d[0].index_format = ib_d.data_ptr(), m.indices.size, 32
        d[0].flags = T.GEOMETRY_FLAG_OPAQUE
        info = T.PrebuildInfo()
        rt.check(rt.lib.rt_blas_prebuild(ctx.handle, d, 1, 0, C.byref(info)))
        descs.append(d)
        bscr.append(torch.empty(info.scratch_bytes, dtype=torch.uint8, device="cuda"))
        bres.append(torch.empty(info.result_bytes, dtype=torch.uint8, device="cuda"))
    tinfo = T.PrebuildInfo()
    rt.check(rt.lib.rt_tlas_prebuild(ctx.handle, n_inst, 0, C.byref(tinfo)))
    tscr = torch.empty(tinfo.scratch_bytes, dtype=torch.uint8, device="cuda")
    tres = torch.empty(tinfo.result_bytes, dtype=torch.uint8, device="cuda")
    inst = (T.InstanceDesc * n_inst)()
    for i, (k, xf) in enumerate(zip(wl.instance_mesh, wl.transforms)):
        inst[i].transform[:] = np.asarray(xf, np.float32).reshape(12).tolist()
        inst[i].instance_id_and_mask = (i & 0xFFFFFF) | (0xFF << 24)
        inst[i].hit_group_and_flags = 2 * i
        inst[i].blas = bres[k].data_ptr()
    inst_h = torch.from_numpy(np.frombuffer(bytes(inst), dtype=np.uint8).copy()).pin_memory()
    inst_d = torch.empty_like(inst_h, device="cuda")
    env_d = torch.from_numpy(np.ascontiguousarray(env, np.float32).reshape(-1)).cuda()
    prog = rt.Program(ctx, rt.PROGRESSIVE)
    for i, k in enumerate(wl.instance_mesh):
        for ray_type in range(2):
            rt.check(rt.lib.rt_bindings_set_hit_record(prog.handle, ray_type, i, dev[k][0].data_ptr(), dev[k][1].data_ptr(),
                                                       C.byref(wl.materials[k])))
    rt.check(rt.lib.rt_bindings_set_miss_record(prog.handle, 0, env_d.data_ptr(), env.shape[1]))
    acc = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")  # zero outside this rank's strips, for ever
    frame_d = torch.zeros_like(acc) if (world > 1 and rank == 0) else None
    img_h = torch.empty(H * W * 4, dtype=torch.float32).pin_memory() if rank == 0 else None
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]

    def frame_once():
        ev[0].record(stream)
        for (vb_h, ib_h), (vb_d, ib_d) in zip(host, dev):
            vb_d.copy_(vb_h, non_blocking=True)
            ib_d.copy_(ib_h, non_blocking=True)
        inst_d.copy_(inst_h, non_blocking=True)
        for d, sc, rs in zip(descs, bscr, bres):
            rt.check(rt.lib.rt_blas_build(ctx.handle, d, 1, 0, sc.data_ptr(), sc.numel(), rs.data_ptr(), rs.numel()))
        rt.check(rt.lib.rt_tlas_build(ctx.handle, inst_d.data_ptr(), n_inst, 0, tscr.data_ptr(), tscr.numel(), tres.data_ptr(), tres.numel()))
        ev[1].record(stream)
        rt.check(rt.lib.rt_set_tlas(ctx.handle, tres.data_ptr()))
        rt.check(rt.lib.rt_set_output(ctx.handle, 0, acc.data_ptr(), 16 * W))
        for local, smp in enumerate(plan.samples):
            f = scenes.make_frame(wl.setup, W, H, frame_count=smp, accum_count=local, jitter=jit[smp % len(jit)])
            rt.check(rt.lib.rt_set_frame_constants(ctx.handle, C.byref(f)))
            if plan.strip_groups > 1:
                rt.check(rt.lib.rt_dispatch_rays_interleaved(ctx.handle, prog.handle, W, H, plan.strip_rows, plan.strip_groups, plan.strip_group))
            else:
                rt.check(rt.lib.rt_dispatch_rays(ctx.handle, prog.handle, W, H, 3))
        ev[2].record(stream)
        if world > 1:
            comm.reduce(acc.data_ptr(), frame_d.data_ptr() if rank == 0 else None, acc.numel(), plan.weight, root=0)
        ev[3].record(stream)
        if rank == 0:
            img_h.copy_(frame_d if world > 1 else acc, non_blocking=True)
        ev[4].record(stream)

    ctx.set_render_options(args.strong_depth, False)
    frame_once()  # warm-up (also grows the wavefront workspace)
    torch.cuda.synchronize()
    ctx.status()
    ctx.ray_counts(reset=True)
    times, parts = [], []
    for _ in range(max(1, args.strong_reps)):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        frame_once()
        torch.cuda.synchronize()
        t = torch.tensor([ev[0].elapsed_time(ev[4])], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        times.append(float(t.item()))
        parts.append([ev[i].elapsed_time(ev[i + 1]) for i in range(4)])
    rc = ctx.ray_counts(reset=True)
    ctx.set_render_options(args.radiance_depth, False)
    r = torch.tensor([float(rc.primary + rc.secondary + rc.shadow)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(r, op=dist.ReduceOp.SUM)
    if rank != 0:
        return None
    assert bool(torch.isfinite(img_h).all()) and float(img_h.sum()) > 0.0
    best = int(np.argmin(times))
    ms = float(np.median(times))
    rays_per_frame = float(r.item()) / len(times)
    h2d = sum(int(a.numel() + b.numel()) for a, b in host) + int(inst_h.numel())
    return {"metric": "time to frame, ms (fixed frame, strong scaling; lower is better)", "time_to_frame_ms": ms, "all_ms": times,
            "n_gpus": world, "workload": f"{wl.description.split(' progressive')[0]}: ONE frame of {SPP} spp in total, split over {world} rank(s)",
            "width": W, "height": H, "spp_total": SPP, "triangles": wl.num_triangles,
            "max_radiance_ray_depth": args.strong_depth,
            "shard_plan": {"strip_groups": plan.strip_groups, "sample_groups": plan.sample_groups, "strip_rows": plan.strip_rows,
                           "samples_on_rank0": len(plan.samples)},
            "root_breakdown_ms": dict(zip(["h2d_and_build", "dispatches", "nccl_reduce", "d2h_root"], parts[best])),
            "mrays_per_s": rays_per_frame / (ms * 1e-3) / 1e6, "rays_per_frame": rays_per_frame,
            "h2d_bytes_per_rank": h2d, "reduce_bytes_per_rank": int(H * W * 16) if world > 1 else 0, "d2h_bytes_root": int(H * W * 16),
            "includes": "pinned H2D of VB/IB/instance descs + BLAS/TLAS build on every rank, the rank's dispatches, "
                        "rt_accum_reduce (NCCL, weighted) onto rank 0, one D2H of the frame on rank 0"}


def measure_target_scene(args, ctx, rt, torch):
    """North-star target: >= 1 Grays/s of incoherent secondary rays on a ~1 M-triangle scene at 1080p.  C1M = displaced
    icosphere, 1 310 722 triangles in one flat BLAS (traversal section ~440 MB, several times the L2).  Reported: the
    incoherent stage alone (CUDA events around k_trace_persistent<0>), its algorithmic bytes per launch from the
    instrumented pass, the whole-frame rate, and the measured DRAM traffic of the same kernel (ncu, profiles/traffic.json)."""
    wl = scenes.workload("C1M")
    W, H, SPP = wl.width, wl.height, 2
    env = scenes.sky_cube(64)
    jit = scenes.jitter_sequence(wl.setup.seed, 16, W, H)
    out = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    r = rt.Renderer(ctx, wl.meshes, wl.transforms, wl.materials, env, rt.PROGRESSIVE, W, H, outputs=[TorchBuffer(out)],
                    instance_mesh=wl.instance_mesh)

    def frames(n0, n):
        for s in range(n0, n0 + n):
            r.dispatch(scenes.make_frame(wl.setup, W, H, frame_count=s, accum_count=s, jitter=jit[s % len(jit)]))

    frames(0, 2)  # warm-up
    ctx.enable_trace_stats(True)
    ctx.trace_stats(reset=True)
    frames(0, SPP)
    st = ctx.trace_stats(reset=True)
    ctx.enable_trace_stats(False)
    ctx.enable_stage_timing(True)
    ctx.stage_timing(reset=True)
    reps = 3
    for _ in range(reps):
        frames(0, SPP)
    tp, ts, tsh = ctx.stage_timing(reset=True)
    ctx.enable_stage_timing(False)
    # whole frames, overlapped dispatch
    ctx.ray_counts(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        frames(0, SPP)
    e1.record()
    torch.cuda.synchronize()
    rc = ctx.ray_counts(reset=True)
    ms = e0.elapsed_time(e1)
    sec = st[1]
    n_launch = reps * SPP
    ms_launch = ts / n_launch
    bytes_launch = (48.0 * sec.rays + 64.0 * sec.internal_visits + 48.0 * sec.leaf_visits) / SPP
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = float(json.load(open(peaks_path))["hbm_gbs"]) if os.path.exists(peaks_path) else FALLBACK_HBM_GBS
    gbs = bytes_launch / (ms_launch * 1e-3) / 1e9
    traffic = load_ncu_traffic("C1M secondary_incoherent (k_trace_persistent<0>)")
    roof = {"bound": "hbm", "kernel": "k_trace_persistent<0> (closest hit, incoherent secondary rays)", "achieved": gbs, "peak": peak,
            "unit": "GB/s", "frac": gbs / peak, "traffic": traffic,
            "dram_frac": (traffic / (ms_launch * 1e-3) / 1e9 / peak) if traffic else None,
            "note": "achieved = algorithmic bytes (48 + 64 n_int + 48 n_leaf per ray over the BVH2 visit counts of the same rays) / "
                    "CUDA-event launch time; traffic = dram bytes per launch of the same kernel from the committed ncu capture; "
                    "dram_frac = traffic / time / peak is the share of the HBM roof the kernel really uses"}
    # the reference's own traversal lever: build flags -> 0 / 1 / 3 treelet passes (FL/TreeletReorder.cpp:66-80).  Same scene,
    # same rays; build time (device, CUDA events) next to the traversal speed each tree yields.
    tradeoff = {}
    import ctypes as C2_
    for name, flags in (("PREFER_FAST_BUILD (0 treelet passes)", T.BUILD_FLAG_PREFER_FAST_BUILD), ("NONE (1 pass: the application's build)", 0),
                        ("PREFER_FAST_TRACE (3 passes)", T.BUILD_FLAG_PREFER_FAST_TRACE)):
        m = wl.meshes[0]
        vb, ib = ctx.upload(m.vertices), ctx.upload(m.indices)
        desc = (T.GeometryDesc * 1)()
        desc[0].vertex_buffer, desc[0].vertex_count, desc[0].vertex_stride_bytes = vb.ptr, m.vertices.shape[0], 24
        desc[0].index_buffer, desc[0].index_count, desc[0].index_format = ib.ptr, m.indices.size, 32
        desc[0].flags = T.GEOMETRY_FLAG_OPAQUE
        info = T.PrebuildInfo()
        rt.check(rt.lib.rt_blas_prebuild(ctx.handle, desc, 1, flags, C2_.byref(info)))
        scr, res = ctx.alloc(info.scratch_bytes), ctx.alloc(info.result_bytes)
        bt = []
        for rep in range(4):
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record()
            rt.check(rt.lib.rt_blas_build(ctx.handle, desc, 1, flags, scr.ptr, scr.nbytes, res.ptr, res.nbytes))
            b1.record()
            torch.cuda.synchronize()
            if rep:
                bt.append(b0.elapsed_time(b1))
        del scr, res, vb, ib
        rr = rt.Renderer(ctx, wl.meshes, wl.transforms, wl.materials, env, rt.PROGRESSIVE, W, H, outputs=[TorchBuffer(out)],
                         instance_mesh=wl.instance_mesh, build_flags=flags)
        for s in range(2):
            rr.dispatch(scenes.make_frame(wl.setup, W, H, frame_count=s, accum_count=s, jitter=jit[s]))
        ctx.enable_stage_timing(True)
        ctx.stage_timing(reset=True)
        ctx.ray_counts(reset=True)
        for _ in range(2):
            for s in range(SPP):
                rr.dispatch(scenes.make_frame(wl.setup, W, H, frame_count=s, accum_count=s, jitter=jit[s]))
        _tp, ts2, _tsh = ctx.stage_timing(reset=True)
        ctx.enable_stage_timing(False)
        rc2 = ctx.ray_counts(reset=True)
        tradeoff[name] = {"build_ms": float(np.median(bt)), "build_mtri_per_s": wl.num_triangles / float(np.median(bt)) / 1e3,
                          "incoherent_mrays_per_s": rc2.secondary / (ts2 * 1e-3) / 1e6}
        del rr
    return {"workload": wl.description, "triangles": wl.num_triangles, "width": W, "height": H,
            "build_flags_tradeoff": tradeoff,
            "incoherent_mrays_per_s": sec.rays / SPP / (ms_launch * 1e-3) / 1e6,
            "incoherent_rays_per_launch": sec.rays / SPP, "ms_per_launch": ms_launch,
            "n_int_per_ray": sec.internal_visits / max(sec.rays, 1), "n_leaf_per_ray": sec.leaf_visits / max(sec.rays, 1),
            "primary_mrays_per_s": st[0].rays / SPP / (tp / n_launch * 1e-3) / 1e6,
            "shadow_mrays_per_s": st[2].rays / SPP / (tsh / n_launch * 1e-3) / 1e6,
            "all_rays_mrays_per_s": (rc.primary + rc.secondary + rc.shadow) / (ms * 1e-3) / 1e6, "ms_per_frame": ms / n_launch,
            "roofline": roof}


def measure_roofline(args, ctx, renderer, setup, jit, world, rank):
    """Algorithmic bytes (SURVEY 8d: 48 + 64*n_int + 48*n_leaf per ray) / CUDA-event time of each trace stage."""
    SPP = args.spp
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    else:
        peak, peak_src = FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"
    # 1) instrumented pass (untimed): node visits / triangle tests of the very same rays in the reference's visit order
    ctx.enable_trace_stats(True)
    ctx.trace_stats(reset=True)
    for s in range(SPP):
        renderer.dispatch(frame_for(setup, args, jit, s * world + rank, s))
    st = ctx.trace_stats(reset=True)
    ctx.enable_trace_stats(False)
    # 2) timed pass with CUDA events around each trace kernel, on the launching stream
    ctx.enable_stage_timing(True)
    ctx.stage_timing(reset=True)
    reps = max(1, args.steps)
    for _ in range(reps):
        for s in range(SPP):
            renderer.dispatch(frame_for(setup, args, jit, s * world + rank, s))
    tp, ts, tsh = ctx.stage_timing(reset=True)
    ctx.enable_stage_timing(False)
    names = ["primary (k_primary)", "secondary_incoherent (k_trace_persistent<0>)", "shadow (k_trace_persistent<1>, 2 launches/frame)"]
    keys = ["primary", "secondary", "shadow"]
    times = [tp, ts, tsh]
    launches_per_frame = [1, 1, 2]
    stages = {}
    for name, s, t, lpf in zip(names, st, times, launches_per_frame):
        n_launch = reps * SPP * lpf
        bytes_total = 48.0 * s.rays + 64.0 * s.internal_visits + 48.0 * s.leaf_visits  # over SPP instrumented frames
        bytes_per_launch = bytes_total / (SPP * lpf)
        ms_per_launch = t / n_launch
        stages[name] = {"rays_per_launch": s.rays / (SPP * lpf), "n_int_per_ray": s.internal_visits / max(s.rays, 1),
                        "n_leaf_per_ray": s.leaf_visits / max(s.rays, 1), "max_stack": int(s.max_stack),
                        "ms_per_launch": ms_per_launch, "algorithmic_bytes_per_launch": bytes_per_launch,
                        "achieved_gbs": bytes_per_launch / (ms_per_launch * 1e-3) / 1e9 if ms_per_launch > 0 else None,
                        "mrays_per_s": s.rays / (SPP * lpf) / (ms_per_launch * 1e-3) / 1e6 if ms_per_launch > 0 else None,
                        "share_of_trace_time": t / max(sum(times), 1e-12)}
    dom_i = max(range(3), key=lambda i: times[i])
    d = stages[names[dom_i]]
    traffic = load_ncu_traffic(names[dom_i]) if args.config == "C2" else None
    dram_frac = (traffic / (d["ms_per_launch"] * 1e-3) / 1e9 / peak) if traffic and d["ms_per_launch"] else None
    # The bound that binds on an L2-resident scene is instruction issue, not HBM: thread-instructions per second against
    # SMs x 4 schedulers x 32 lanes x SM clock.  Instruction counts come from the committed ncu capture of the same kernel
    # (they are a property of the rays and the tree, not of the run); the time is measured live.
    issue = None
    ncu = load_ncu_counters(names[dom_i]) if args.config == "C2" else None
    if ncu and d["ms_per_launch"]:
        sm_hz = 1.965e9
        peak_tinst = 148 * 4 * 32 * sm_hz / 1e12
        ach = ncu["warp_instructions"] * ncu["lanes_per_instruction"] / (d["ms_per_launch"] * 1e-3) / 1e12
        issue = {"bound": "issue", "kernel": names[dom_i], "achieved": ach, "peak": peak_tinst, "unit": "T thread-instructions/s",
                 "frac": ach / peak_tinst, "warp_instructions_per_launch": ncu["warp_instructions"],
                 "lanes_per_instruction": ncu["lanes_per_instruction"], "source": ncu.get("source"),
                 "note": "frac = (issue-slot utilisation) x (lanes active / 32): what separates the kernel from a perfectly "
                         "converged, always-issuing SIMT machine"}
    roofline = {"bound": "hbm", "kernel": names[dom_i], "achieved": d["achieved_gbs"], "peak": peak, "unit": "GB/s",
                "frac": d["achieved_gbs"] / peak if d["achieved_gbs"] else None, "traffic": traffic, "dram_frac": dram_frac,
                "binds": False, "issue": issue,
                "peak_source": peak_src,
                "note": "achieved = algorithmic bytes/ray (48 + 64*n_int + 48*n_leaf over the BVH2 visit counts of the same rays, "
                        "SURVEY 8d) x rays per launch / CUDA-event launch time, as the contract defines it.  On this workload the "
                        "HBM roof does NOT bind (`binds`: false): the traversal structure is L1/L2-resident, measured DRAM traffic "
                        "(`traffic`, ncu) is a few per cent of the algorithmic bytes (`dram_frac` of the HBM peak), which is also why "
                        "frac can exceed 1.  The binding roof is instruction issue (`issue`); the HBM-relevant measurement is "
                        "`target_scene.roofline` (1.31 M triangles, structure several times the L2).  Stage times are measured with the "
                        "dispatch in its sequential, stage-timed mode; `value` with the stages of two pixel bands overlapped (DESIGN 4.2)"}
    return roofline, stages


def load_ncu_traffic(stage_key):
    """dram bytes per launch of a trace stage from the committed ncu summary (profiles/traffic.json), if present."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get("dram_bytes_per_launch", {}).get(stage_key)
        except Exception:
            return None
    return None


def load_ncu_counters(stage_key):
    """warp instructions / lanes per instruction of a trace stage from the committed ncu capture (profiles/traffic.json)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            c = j.get("issue_counters", {}).get(stage_key)
            if c:
                c = dict(c, source=j.get("source"))
            return c
        except Exception:
            return None
    return None


def measure_build(args, ctx, rt, torch, stream):
    """LBVH build Mtri/s: device-resident VB/IB of a triangle soup -> traversable BVH (SURVEY 8d: 432 B/triangle)."""
    n = args.build_tris
    g = torch.Generator(device="cuda")
    g.manual_seed(1234)
    c = (torch.rand((n, 1, 3), device="cuda", generator=g) * 2 - 1) * 500.0   # centroids uniform in [-500, 500]^3
    off = torch.rand((n, 3, 3), device="cuda", generator=g) - 0.5             # edge <= 1
    vb = torch.zeros((3 * n, 6), dtype=torch.float32, device="cuda")          # {position, normal} stride 24
    vb[:, :3] = (c + off).reshape(-1, 3)
    ib = torch.arange(3 * n, dtype=torch.int32, device="cuda")
    del c, off
    desc = (T.GeometryDesc * 1)()
    desc[0].vertex_buffer, desc[0].vertex_count, desc[0].vertex_stride_bytes = vb.data_ptr(), 3 * n, 24
    desc[0].index_buffer, desc[0].index_count, desc[0].index_format = ib.data_ptr(), 3 * n, 32
    desc[0].flags = T.GEOMETRY_FLAG_OPAQUE
    info = T.PrebuildInfo()
    rt.check(rt.lib.rt_blas_prebuild(ctx.handle, desc, 1, 0, C.byref(info)))
    scr = torch.empty(info.scratch_bytes, dtype=torch.uint8, device="cuda")
    res = torch.empty(info.result_bytes, dtype=torch.uint8, device="cuda")
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = float(json.load(open(peaks_path))["hbm_gbs"]) if os.path.exists(peaks_path) else FALLBACK_HBM_GBS

    def timed(flags):
        times = []
        l0 = ctx.launches()
        reps = 3 + max(3, args.steps)
        for r in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            rt.check(rt.lib.rt_blas_build(ctx.handle, desc, 1, flags, scr.data_ptr(), scr.numel(), res.data_ptr(), res.numel()))
            e1.record(stream)
            torch.cuda.synchronize()
            if r >= 3:
                times.append(e0.elapsed_time(e1))
        return float(np.median(times)), int((ctx.launches() - l0) // reps)

    # Headline: the LBVH of the north star (Morton codes, radix sort, Karras hierarchy, bottom-up fit) = PREFER_FAST_BUILD,
    # which skips the Fallback Layer's treelet optimisation (FL/TreeletReorder.cpp:66-69).  `with_treelet_pass` = default
    # flags, what the reference application builds (one optimisation pass), `fast_trace` = three passes.
    ms, launches = timed(T.BUILD_FLAG_PREFER_FAST_BUILD)
    ms_default, launches_default = timed(0)
    ms_trace, _ = timed(T.BUILD_FLAG_PREFER_FAST_TRACE)
    gbs = n * 432.0 / (ms * 1e-3) / 1e9
    return {"metric": "LBVH build Mtri/s", "value": n / ms / 1e3, "triangles": n, "ms": ms, "launches_per_build": launches,
            "build_flags": "PREFER_FAST_BUILD (plain LBVH)",
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                         "algorithmic_bytes_per_triangle": 432},
            "with_treelet_pass": {"value": n / ms_default / 1e3, "ms": ms_default, "launches_per_build": launches_default,
                                  "build_flags": "NONE (1 treelet pass, the reference application's build)"},
            "fast_trace": {"value": n / ms_trace / 1e3, "ms": ms_trace, "build_flags": "PREFER_FAST_TRACE (3 treelet passes)"},
            "workload": f"{n}-triangle soup, uniform centroids in [-500,500]^3, edge <= 1, device-resident VB/IB -> traversable BVH "
                        "(working set >> L2)", "result_mb": info.result_bytes / 2**20, "scratch_mb": info.scratch_bytes / 2**20}


def measure_denoise(args, ctx, rt, torch, stream):
    """DenoiseCompositor::dispatch alone at 1920x1080, maxKernelSize 12 (SURVEY 8d: 96 B/pixel algorithmic = 2 passes x
    (2 float4 reads + 1 float4 write)).  Between timed launches a 256 MB buffer is rewritten so the 132 MB of images do
    not stay in the 126 MB L2."""
    W, H = 1920, 1080
    g = torch.Generator(device="cuda")
    g.manual_seed(7)
    direct = torch.rand((H * W * 4,), device="cuda", generator=g)
    spec = torch.rand((H * W * 4,), device="cuda", generator=g)
    tmp, out = torch.empty_like(direct), torch.empty_like(direct)
    flush = torch.empty(64 * 2**20, dtype=torch.float32, device="cuda")
    prm = denoiser_params()
    times = []
    for r in range(3 + 10):
        flush.fill_(float(r))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        rt.check(rt.lib.rt_denoise(ctx.handle, direct.data_ptr(), spec.data_ptr(), tmp.data_ptr(), out.data_ptr(), W, H, C.byref(prm)))
        e1.record(stream)
        torch.cuda.synchronize()
        if r >= 3:
            times.append(e0.elapsed_time(e1))
    ms = float(np.median(times))
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = float(json.load(open(peaks_path))["hbm_gbs"]) if os.path.exists(peaks_path) else FALLBACK_HBM_GBS
    gbs = W * H * 96.0 / (ms * 1e-3) / 1e9
    return {"metric": "DenoiseCompositor ms/frame (1920x1080, maxKernelSize 12, 2 launches)", "ms": ms, "mpixels_per_s": W * H / ms / 1e3,
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                         "algorithmic_bytes_per_pixel": 96}, "l2": "256 MB flush between launches"}


def measure_cpu_baseline(args, wl, env, jit):
    """BASELINE.md section 2: the oracle port compiled -O3 -march=native on this host, all cores, median of >= 3
    repetitions, build and trace timed separately (Mtri/s and Mrays/s defined as for the GPU)."""
    import oracle
    cflags = oracle.use_native()
    cores = os.cpu_count() or 1
    # build: BLAS (+ TLAS) of the workload's meshes, single-threaded (the restated builder is sequential)
    build_times = []
    for _ in range(3):
        t0 = time.perf_counter()
        orc, tlas, recs, _keep = oracle_scene(wl)
        build_times.append(time.perf_counter() - t0)
    build_s = float(np.median(build_times))
    acc = np.zeros((wl.height, wl.width, 4), np.float32)
    vals, rays_total, t_start = [], 0, time.perf_counter()
    for n in range(5):
        counts = T.RayCounts()
        t0 = time.perf_counter()
        oracle_frame(orc, tlas, recs, env, wl, frame_for(wl.setup, args, jit, n, 0), acc, cores, counts)
        dt = time.perf_counter() - t0
        rays = counts.primary + counts.secondary + counts.shadow
        rays_total += rays
        vals.append(metric_of(wl, rays / dt / 1e6, dt * 1e3)[1])
        if len(vals) >= 3 and time.perf_counter() - t_start > 20.0:
            break
    metric = metric_of(wl, 0.0, 0.0)[0]
    return {"value": float(np.median(vals)), "unit": metric, "cores": cores, "kind": "port",
            "sample": f"median of {len(vals)} x 1 spp of the {wl.width}x{wl.height} frame ({rays_total // len(vals)} rays each) in "
                      f"{time.perf_counter() - t_start:.1f} s, row-parallel over {cores} threads, compiled {cflags}",
            "all_values": vals,
            "build": {"metric": "LBVH build Mtri/s (CPU, 1 thread, default flags = 1 treelet pass)", "value": wl.num_triangles / build_s / 1e6,
                      "triangles": wl.num_triangles, "ms": build_s * 1e3, "cores": 1, "repetitions": 3}}


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
