"""ctypes binding of the C ABI in ``include/rt_core.h`` (``librt_core.so``).

This is the only way Python reaches the CUDA kernels.  There is no fallback of any kind: if the shared
library is missing, or was built without every symbol the header declares, importing fails; if no CUDA
device is present, :class:`Context` raises :class:`RtError`.
"""
import ctypes as C
import os
import re

import numpy as np

from . import types as T

_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RT_CORE_LIB") or os.path.join(_DIR, "librt_core.so")  # RT_CORE_LIB: development builds with other tuning macros
HEADER_PATH = os.path.join(_DIR, "..", "include", "rt_core.h")


class RtError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"rt_core error {code}: {message}")
        self.code = code


def declared_symbols(header_path: str = HEADER_PATH):
    """Every function name declared in rt_core.h (used by the symbol-coverage test)."""
    text = open(header_path).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rt_[a-z_0-9]+)\s*\(", text)))


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C dxrexperiments_b200/csrc).  rt_core has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    missing = [s for s in declared_symbols() if not hasattr(lib, s)]
    if missing:
        raise ImportError(f"{LIB_PATH} lacks symbols declared in rt_core.h: {missing}")
    vp, u32, u64, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int
    pp = C.POINTER(vp)
    sig = {
        "rt_last_error": (C.c_char_p, []),
        "rt_version": (C.c_char_p, []),
        "rt_context_create": (i32, [i32, pp]),
        "rt_context_destroy": (i32, [vp]),
        "rt_context_set_stream": (i32, [vp, vp]),
        "rt_sync": (i32, [vp]),
        "rt_get_status": (i32, [vp]),
        "rt_launch_count": (u64, [vp]),
        "rt_malloc": (i32, [vp, u64, pp]),
        "rt_free": (i32, [vp, vp]),
        "rt_memset": (i32, [vp, vp, i32, u64]),
        "rt_upload": (i32, [vp, vp, vp, u64]),
        "rt_download": (i32, [vp, vp, vp, u64]),
        "rt_host_alloc_pinned": (i32, [u64, pp]),
        "rt_host_free_pinned": (i32, [vp]),
        "rt_blas_prebuild": (i32, [vp, vp, u32, u32, vp]),
        "rt_blas_build": (i32, [vp, vp, u32, u32, vp, u64, vp, u64]),
        "rt_tlas_prebuild": (i32, [vp, u32, u32, vp]),
        "rt_tlas_build": (i32, [vp, vp, u32, u32, vp, u64, vp, u64]),
        "rt_tlas_build_ptrs": (i32, [vp, vp, u32, u32, vp, u64, vp, u64]),
        "rt_blas_prebuild_ptrs": (i32, [vp, vp, u32, u32, vp]),
        "rt_blas_build_ptrs": (i32, [vp, vp, u32, u32, vp, u64, vp, u64]),
        "rt_build_scratch_layout": (i32, [u32, i32, vp]),
        "rt_update_cache_layout": (i32, [u32, i32, C.POINTER(u64), C.POINTER(u64)]),
        "rt_as_copy": (i32, [vp, vp, u64, vp, i32]),
        "rt_as_emit_postbuild_info": (i32, [vp, vp, u32, vp]),
        "rt_as_get_info": (i32, [vp, vp, vp]),
        "rt_blob_bytes": (u64, [u32, i32]),
        "rt_program_create": (i32, [vp, i32, u32, u32, pp]),
        "rt_program_destroy": (i32, [vp]),
        "rt_bindings_set_hit_record": (i32, [vp, u32, u32, vp, vp, vp]),
        "rt_bindings_set_miss_record": (i32, [vp, u32, vp, u32]),
        "rt_set_frame_constants": (i32, [vp, vp]),
        "rt_set_output": (i32, [vp, u32, vp, u64]),
        "rt_set_aov_output": (i32, [vp, u32, vp, u64]),
        "rt_set_tlas": (i32, [vp, vp]),
        "rt_set_instance_motion": (i32, [vp, vp, u32]),
        "rt_set_instance_deformation": (i32, [vp, vp, u32]),
        "rt_set_render_options": (i32, [vp, vp]),
        "rt_set_adaptive_sampling": (i32, [vp, vp, vp]),
        "rt_adaptive_update": (i32, [vp, vp, vp, u32, u32, vp, vp]),
        "rt_dispatch_rays": (i32, [vp, vp, u32, u32, u32]),
        "rt_dispatch_rays_region": (i32, [vp, vp, u32, u32, u32, u32, u32, u32]),
        "rt_get_ray_counts": (i32, [vp, vp, i32]),
        "rt_enable_trace_stats": (i32, [vp, i32]),
        "rt_get_trace_stats": (i32, [vp, vp, vp, vp, i32]),
        "rt_enable_stage_timing": (i32, [vp, i32]),
        "rt_get_stage_timing": (i32, [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double), i32]),
        "rt_denoise": (i32, [vp, vp, vp, vp, vp, u32, u32, vp]),
        "rt_denoise_progressive": (i32, [vp, vp, vp, vp, vp, vp, u32, u32, vp]),
        "rt_denoise_temporal": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, u32, u32, vp]),
        "rt_denoise_temporal_motion": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, u32, u32, vp]),
        "rt_trace_rays": (i32, [vp, vp, vp, u64, u32, u32, vp]),
        "rt_trace_rays_stats": (i32, [vp, vp, vp, u64, u32, u32, vp, vp]),
        "rt_trace_rays_hit_groups": (i32, [vp, vp, vp, u64, u32, u32, u32, u32, vp, u32, vp]),
        "rt_generate_primary_rays": (i32, [vp, vp, u32, u32, C.c_float, vp]),
        "rt_scale_buffer": (i32, [vp, vp, u64, C.c_float]),
        "rt_dispatch_rays_interleaved": (i32, [vp, vp, u32, u32, u32, u32, u32]),
        "rt_enable_debug_capture": (i32, [vp, i32]),
        "rt_debug_counts": (i32, [vp, C.POINTER(u32), C.POINTER(u32), C.POINTER(u32)]),
        "rt_debug_download": (i32, [vp, i32, u32, vp, u64]),
        "rt_comm_get_unique_id": (i32, [vp]),
        "rt_comm_create": (i32, [vp, vp, i32, i32, pp]),
        "rt_comm_destroy": (i32, [vp]),
        "rt_comm_info": (i32, [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]),
        "rt_accum_reduce": (i32, [vp, vp, vp, vp, u64, C.c_float, i32]),
    }
    for name, (res, args) in sig.items():
        f = getattr(lib, name)
        f.restype = res
        f.argtypes = args
    return lib


lib = _load()


class ScratchLayout(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("scene_aabb", "morton_codes", "sorted_codes", "sorted_indices", "hierarchy",
                                          "primitives", "metadata", "total")]


def check(code):
    if code != 0:
        raise RtError(code, lib.rt_last_error().decode())


class Buffer:
    """A device allocation owned by a context."""

    def __init__(self, ctx, nbytes: int):
        self.ctx = ctx
        self.nbytes = int(nbytes)
        p = C.c_void_p()
        check(lib.rt_malloc(ctx.handle, self.nbytes, C.byref(p)))
        self.ptr = p.value

    def upload(self, host: np.ndarray, offset: int = 0):
        host = np.ascontiguousarray(host)
        assert offset + host.nbytes <= self.nbytes
        check(lib.rt_upload(self.ctx.handle, self.ptr + offset, host.ctypes.data, host.nbytes))
        self.ctx.sync()  # host is pageable here; keep it alive until the copy is done
        return self

    def download(self, dtype=np.uint8, count=None, offset: int = 0) -> np.ndarray:
        dtype = np.dtype(dtype)
        if count is None:
            count = (self.nbytes - offset) // dtype.itemsize
        out = np.empty(count, dtype=dtype)
        check(lib.rt_download(self.ctx.handle, out.ctypes.data, self.ptr + offset, out.nbytes))
        return out

    def zero(self):
        check(lib.rt_memset(self.ctx.handle, self.ptr, 0, self.nbytes))
        return self

    def free(self):
        if self.ptr:
            lib.rt_free(self.ctx.handle, self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            if self.ptr and self.ctx.handle:
                self.free()
        except Exception:
            pass


class Context:
    def __init__(self, device: int = 0, stream: int = None):
        h = C.c_void_p()
        check(lib.rt_context_create(device, C.byref(h)))
        self.handle = h.value
        self.device = device
        if stream is not None:
            check(lib.rt_context_set_stream(self.handle, stream))

    def close(self):
        if self.handle:
            lib.rt_context_destroy(self.handle)
            self.handle = None

    def sync(self):
        check(lib.rt_sync(self.handle))

    def status(self):
        check(lib.rt_get_status(self.handle))

    def set_render_options(self, max_radiance_ray_depth: int = 1, half_render_targets: bool = False):
        """MAX_RADIANCE_RAY_DEPTH (1 = the reference's shaders, 2 = one more Phong-lobe bounce) and R16G16B16A16_FLOAT emulation."""
        o = (C.c_uint32 * 2)(max_radiance_ray_depth, 1 if half_render_targets else 0)
        check(lib.rt_set_render_options(self.handle, o))

    def launches(self) -> int:
        return int(lib.rt_launch_count(self.handle))

    def alloc(self, nbytes) -> Buffer:
        return Buffer(self, nbytes)

    def upload(self, host: np.ndarray) -> Buffer:
        host = np.ascontiguousarray(host)
        return Buffer(self, max(host.nbytes, 16)).upload(host)

    # ---------------------------------------------------------------- acceleration structures
    def build_blas(self, geoms, build_flags: int = 0, keep_scratch: bool = False, array_of_pointers: bool = False):
        """geoms: list of dicts {vertices: Buffer|ptr, vertex_count, stride, indices: Buffer|ptr|None, index_count,
        index_format, transform: Buffer|ptr|None, flags}."""
        descs = _geometry_descs(geoms)
        info = T.PrebuildInfo()
        if array_of_pointers:  # D3D12_ELEMENTS_LAYOUT_ARRAY_OF_POINTERS: a host array of pointers to the descriptors
            pp = (C.c_void_p * len(geoms))(*[C.addressof(descs[i]) for i in range(len(geoms))])
            check(lib.rt_blas_prebuild_ptrs(self.handle, pp, len(geoms), build_flags, C.byref(info)))
        else:
            check(lib.rt_blas_prebuild(self.handle, descs, len(geoms), build_flags, C.byref(info)))
        scratch = self.alloc(info.scratch_bytes)
        result = self.alloc(info.result_bytes)
        if array_of_pointers:
            check(lib.rt_blas_build_ptrs(self.handle, pp, len(geoms), build_flags, scratch.ptr, scratch.nbytes, result.ptr,
                                         result.nbytes))
        else:
            check(lib.rt_blas_build(self.handle, descs, len(geoms), build_flags, scratch.ptr, scratch.nbytes, result.ptr,
                                    result.nbytes))
        n = sum(g["aabb_count"] if "aabbs" in g else
                (g.get("index_count", 0) if g.get("index_format", 32 if g.get("indices") is not None else 0) else
                 g["vertex_count"]) // 3 for g in geoms)
        acc = Accel(self, result, n, top=False, scratch=scratch if keep_scratch else None, keep=list(geoms),
                    build_flags=build_flags)
        if not keep_scratch:
            self.sync()
            scratch.free()
        return acc

    def build_blas_from_mesh(self, mesh, flags=T.GEOMETRY_FLAG_OPAQUE, keep_scratch=False, build_flags: int = 0):
        vb = self.upload(mesh.vertices)
        ib = self.upload(mesh.indices)
        acc = self.build_blas([dict(vertices=vb, vertex_count=mesh.vertices.shape[0], stride=24, indices=ib,
                                    index_count=mesh.indices.size, index_format=32, flags=flags)],
                              build_flags=build_flags, keep_scratch=keep_scratch)
        acc.vb, acc.ib = vb, ib
        return acc

    def update_blas(self, acc, geoms):
        """PERFORM_UPDATE of an ALLOW_UPDATE bottom-level build with new geometry data (same counts and order)."""
        descs = _geometry_descs(geoms)
        flags = acc.build_flags | T.BUILD_FLAG_PERFORM_UPDATE
        info = T.PrebuildInfo()
        check(lib.rt_blas_prebuild(self.handle, descs, len(geoms), acc.build_flags, C.byref(info)))
        scratch = self.alloc(info.update_scratch_bytes or info.scratch_bytes)
        check(lib.rt_blas_build(self.handle, descs, len(geoms), flags, scratch.ptr, scratch.nbytes, acc.result.ptr,
                                acc.result.nbytes))
        self.sync()
        scratch.free()
        acc._keep = list(geoms)
        return acc

    def update_tlas(self, acc, transforms, ids=None, masks=None, hit_groups=None, flags=None):
        """PERFORM_UPDATE of an ALLOW_UPDATE top-level build: same instances in the same order, new descs."""
        blases = acc._keep[1]
        dev_descs = self.upload(_instance_descs_bytes(blases, transforms, ids, masks, hit_groups, flags))
        info = T.PrebuildInfo()
        check(lib.rt_tlas_prebuild(self.handle, acc.n, acc.build_flags, C.byref(info)))
        scratch = self.alloc(info.update_scratch_bytes or info.scratch_bytes)
        check(lib.rt_tlas_build(self.handle, dev_descs.ptr, acc.n, acc.build_flags | T.BUILD_FLAG_PERFORM_UPDATE, scratch.ptr,
                                scratch.nbytes, acc.result.ptr, acc.result.nbytes))
        self.sync()
        scratch.free()
        acc._keep = [dev_descs, blases]
        return acc

    def compacted_sizes(self, accels):
        """EmitRaytracingAccelerationStructurePostbuildInfo: compacted byte size of each structure."""
        n = len(accels)
        out = self.alloc(max(8 * n, 8))
        arr = (C.c_void_p * max(n, 1))(*[a.result.ptr for a in accels])
        check(lib.rt_as_emit_postbuild_info(self.handle, out.ptr, n, arr))
        return out.download(np.uint64, n)

    def build_tlas(self, blases, transforms, ids=None, masks=None, hit_groups=None, flags=None, build_flags: int = 0,
                   keep_scratch: bool = False, array_of_pointers: bool = False):
        """array_of_pointers: D3D12_ELEMENTS_LAYOUT_ARRAY_OF_POINTERS — the descriptors are stored in reverse order with a gap
        between them and handed over as a device array of device addresses (rt_tlas_build_ptrs)."""
        n = len(blases)
        descs = _instance_descs_bytes(blases, transforms, ids, masks, hit_groups, flags)
        info = T.PrebuildInfo()
        check(lib.rt_tlas_prebuild(self.handle, n, build_flags, C.byref(info)))
        scratch = self.alloc(info.scratch_bytes)
        result = self.alloc(info.result_bytes)
        if array_of_pointers and n:
            stride = 64 + 64  # descriptors scattered: reversed, one 64-byte gap after each
            scattered = np.zeros(n * stride, np.uint8)
            for i in range(n):
                scattered[(n - 1 - i) * stride:(n - 1 - i) * stride + 64] = descs[64 * i:64 * i + 64]
            dev_descs = self.upload(scattered)
            ptrs = np.array([dev_descs.ptr + (n - 1 - i) * stride for i in range(n)], np.uint64)
            dev_ptrs = self.upload(ptrs.view(np.uint8))
            check(lib.rt_tlas_build_ptrs(self.handle, dev_ptrs.ptr, n, build_flags, scratch.ptr, scratch.nbytes, result.ptr,
                                         result.nbytes))
            dev_descs = [dev_descs, dev_ptrs]
        else:
            dev_descs = self.upload(descs) if n else None
            check(lib.rt_tlas_build(self.handle, dev_descs.ptr if n else None, n, build_flags, scratch.ptr, scratch.nbytes,
                                    result.ptr, result.nbytes))
        acc = Accel(self, result, n, top=True, scratch=scratch if keep_scratch else None, keep=[dev_descs, list(blases)],
                    build_flags=build_flags)
        if not keep_scratch:
            self.sync()
            scratch.free()
        return acc

    # ---------------------------------------------------------------- wavefront primitives
    def trace(self, tlas, rays: np.ndarray, ray_flags: int = 0, mask: int = 0xFF, stats: bool = False):
        rays = np.ascontiguousarray(rays, dtype=T.RAY_DTYPE)
        n = rays.shape[0]
        d_rays = self.upload(rays.view(np.uint8).reshape(-1))
        d_hits = self.alloc(max(32 * n, 32))
        if stats:
            d_stats = self.alloc(64).zero()
            check(lib.rt_trace_rays_stats(self.handle, tlas.result.ptr, d_rays.ptr, n, ray_flags, mask, d_hits.ptr,
                                          d_stats.ptr))
            st = d_stats.download(np.uint64, 5)
        else:
            check(lib.rt_trace_rays(self.handle, tlas.result.ptr, d_rays.ptr, n, ray_flags, mask, d_hits.ptr))
            st = None
        hits = d_hits.download(T.HIT_DTYPE, n)
        self.status()
        return (hits, st) if stats else hits

    def trace_hit_groups(self, tlas, rays: np.ndarray, programs, ray_flags: int = 0, mask: int = 0xFF,
                         ray_contribution: int = 0, geometry_multiplier: int = 0):
        """Traversal with any-hit / intersection programs; programs: (R, 2) uint32 {any_hit, intersection}."""
        rays = np.ascontiguousarray(rays, dtype=T.RAY_DTYPE)
        n = rays.shape[0]
        progs = np.ascontiguousarray(programs, np.uint32).reshape(-1, 2)
        d_rays = self.upload(rays.view(np.uint8).reshape(-1))
        d_hits = self.alloc(max(32 * n, 32))
        check(lib.rt_trace_rays_hit_groups(self.handle, tlas.result.ptr, d_rays.ptr, n, ray_flags, mask, ray_contribution,
                                           geometry_multiplier, progs.ctypes.data, progs.shape[0], d_hits.ptr))
        hits = d_hits.download(T.HIT_DTYPE, n)
        self.status()
        return hits

    def primary_rays(self, frame, width, height, jitter_scale=30.0) -> np.ndarray:
        d = self.alloc(32 * width * height)
        check(lib.rt_generate_primary_rays(self.handle, C.byref(frame), width, height, jitter_scale, d.ptr))
        return d.download(T.RAY_DTYPE, width * height)

    def denoise(self, direct: np.ndarray, spec: np.ndarray, params: T.DenoiserParams):
        h, w = direct.shape[:2]
        d_dir = self.upload(np.ascontiguousarray(direct, np.float32).reshape(-1))
        d_spec = self.upload(np.ascontiguousarray(spec, np.float32).reshape(-1))
        d_tmp = self.alloc(16 * w * h)
        d_out = self.alloc(16 * w * h)
        check(lib.rt_denoise(self.handle, d_dir.ptr, d_spec.ptr, d_tmp.ptr, d_out.ptr, w, h, C.byref(params)))
        out = d_out.download(np.float32).reshape(h, w, 4)
        tmp = d_tmp.download(np.float32).reshape(h, w, 4)
        return out, tmp

    def denoise_progressive(self, beauty: np.ndarray, albedo: np.ndarray, normal: np.ndarray,
                            params: T.ProgressiveDenoiseParams = None) -> np.ndarray:
        """rt_denoise_progressive on host images: (h, w, 4) float32 beauty, albedo and normal AOVs -> (h, w, 4) float32."""
        h, w = beauty.shape[:2]
        d_in = [self.upload(np.ascontiguousarray(a, np.float32).reshape(-1)) for a in (beauty, albedo, normal)]
        d_tmp = self.alloc(32 * w * h)
        d_out = self.alloc(16 * w * h)
        params = T.progressive_denoise_defaults() if params is None else params
        check(lib.rt_denoise_progressive(self.handle, *(d.ptr for d in d_in), d_tmp.ptr, d_out.ptr, w, h, C.byref(params)))
        return d_out.download(np.float32).reshape(h, w, 4)

    def denoise_temporal(self, beauty: np.ndarray, albedo: np.ndarray, normal: np.ndarray, position: np.ndarray,
                         prev_camera: T.CameraParams = None, prev_history: np.ndarray = None,
                         params: T.TemporalDenoiseParams = None):
        """rt_denoise_temporal on host images: (h, w, 4) float32 beauty and albedo, normal and position AOVs, the previous
        frame's camera and the history it returned (both None for a first frame) -> (out (h, w, 4), history (4, h, w, 4)),
        both float32.  The history planes are (C, n), (m1, m2, 0, 0), normal, position (include/rt_core.h)."""
        h, w = beauty.shape[:2]
        d_in = [self.upload(np.ascontiguousarray(a, np.float32).reshape(-1)) for a in (beauty, albedo, normal, position)]
        d_prev = None if prev_history is None else self.upload(np.ascontiguousarray(prev_history, np.float32).reshape(-1))
        d_hist, d_tmp, d_out = self.alloc(64 * w * h), self.alloc(32 * w * h), self.alloc(16 * w * h)
        params = T.temporal_denoise_defaults() if params is None else params
        check(lib.rt_denoise_temporal(self.handle, *(d.ptr for d in d_in), C.byref(prev_camera) if prev_camera is not None else None,
                                      d_prev.ptr if d_prev is not None else None, d_hist.ptr, d_tmp.ptr, d_out.ptr, w, h,
                                      C.byref(params)))
        return d_out.download(np.float32).reshape(h, w, 4), d_hist.download(np.float32).reshape(4, h, w, 4)

    def denoise_temporal_motion(self, beauty: np.ndarray, albedo: np.ndarray, normal: np.ndarray, position: np.ndarray,
                                previous_position: np.ndarray, prev_camera: T.CameraParams = None, prev_history: np.ndarray = None,
                                params: T.TemporalDenoiseParams = None):
        """rt_denoise_temporal_motion on host images: denoise_temporal with the previous-position AOV, which the
        reprojection and the position test use in place of the position AOV."""
        h, w = beauty.shape[:2]
        d_in = [self.upload(np.ascontiguousarray(a, np.float32).reshape(-1)) for a in (beauty, albedo, normal, position, previous_position)]
        d_prev = None if prev_history is None else self.upload(np.ascontiguousarray(prev_history, np.float32).reshape(-1))
        d_hist, d_tmp, d_out = self.alloc(64 * w * h), self.alloc(32 * w * h), self.alloc(16 * w * h)
        params = T.temporal_denoise_defaults() if params is None else params
        check(lib.rt_denoise_temporal_motion(self.handle, *(d.ptr for d in d_in),
                                             C.byref(prev_camera) if prev_camera is not None else None,
                                             d_prev.ptr if d_prev is not None else None, d_hist.ptr, d_tmp.ptr, d_out.ptr, w, h,
                                             C.byref(params)))
        return d_out.download(np.float32).reshape(h, w, 4), d_hist.download(np.float32).reshape(4, h, w, 4)

    def set_instance_motion(self, matrices=None, n: int = 0):
        """rt_set_instance_motion: `matrices` is a device Buffer (or address) of n row-major 3x4 float32 world ->
        previous-world matrices, one per InstanceIndex(); None with n = 0 unbinds."""
        check(lib.rt_set_instance_motion(self.handle, _ptr(matrices), n))

    def set_instance_deformation(self, descs=None, n: int = 0):
        """rt_set_instance_deformation: `descs` is a device Buffer (or address) of n types.DeformationDesc, one per
        InstanceIndex(); None with n = 0 unbinds."""
        check(lib.rt_set_instance_deformation(self.handle, _ptr(descs), n))

    def set_adaptive_sampling(self, counts=None, moments=None):
        """rt_set_adaptive_sampling: `counts` (width*height uint32) and `moments` (width*height*2 float32) are device Buffers
        (or addresses) that the following progressive dispatches sample adaptively with; None, None unbinds."""
        check(lib.rt_set_adaptive_sampling(self.handle, _ptr(counts), _ptr(moments)))

    def adaptive_update(self, moments, counts, width: int, height: int, params: T.AdaptiveParams = None, active_count=None):
        """rt_adaptive_update on device buffers: marks converged pixels in `counts`; `active_count` (a device Buffer or
        address of one uint32, or None) receives the number of pixels still active.  Stream-ordered, no synchronisation."""
        params = T.adaptive_defaults() if params is None else params
        check(lib.rt_adaptive_update(self.handle, _ptr(moments), _ptr(counts), width, height, C.byref(params), _ptr(active_count)))

    def ray_counts(self, reset=False) -> T.RayCounts:
        c = T.RayCounts()
        check(lib.rt_get_ray_counts(self.handle, C.byref(c), 1 if reset else 0))
        return c

    # ---------------------------------------------------------------- parity instrumentation
    DEBUG_ARRAYS = {"primary_hits": (0, "pixels", np.dtype([("t", "<f4"), ("u", "<f4"), ("v", "<f4"), ("prim", "<u4")])),
                    "primary_records": (1, "pixels", np.dtype("<u4")),
                    "slot_info": (2, "slots", np.dtype([("pixel", "<u4"), ("record", "<u4"), ("flags", "<u4"), ("pad", "<u4")])),
                    "secondary_rays": (3, "slots", T.RAY_DTYPE),
                    "secondary_hits": (4, "slots", np.dtype([("t", "<f4"), ("u", "<f4"), ("v", "<f4"), ("prim", "<u4")])),
                    "secondary_records": (5, "slots", np.dtype("<u4")),
                    "shadow0_rays": (6, "slots", T.RAY_DTYPE), "shadow0_visibility": (7, "slots", np.dtype("u1")),
                    "shadow1_rays": (8, "pairs", T.RAY_DTYPE), "shadow1_visibility": (9, "pairs", np.dtype("u1"))}

    def enable_debug_capture(self, on=True):
        check(lib.rt_enable_debug_capture(self.handle, 1 if on else 0))

    def debug_counts(self):
        p, s, q = C.c_uint32(), C.c_uint32(), C.c_uint32()
        check(lib.rt_debug_counts(self.handle, C.byref(p), C.byref(s), C.byref(q)))
        return {"pixels": p.value, "slots": s.value, "pairs": q.value}

    def debug_array(self, name: str, plane: int = 0) -> np.ndarray:
        """A stage product of the last captured dispatch (rt_debug_download)."""
        code, which, dtype = self.DEBUG_ARRAYS[name]
        n = self.debug_counts()[which]
        out = np.zeros(max(n, 1), dtype=dtype)
        check(lib.rt_debug_download(self.handle, code, plane, out.ctypes.data, out.nbytes))
        return out[:n]

    def enable_trace_stats(self, on=True):
        check(lib.rt_enable_trace_stats(self.handle, 1 if on else 0))

    def trace_stats(self, reset=False):
        """(primary, secondary, shadow) TraceStats of the instrumented dispatches so far."""
        out = [T.TraceStats() for _ in range(3)]
        check(lib.rt_get_trace_stats(self.handle, C.byref(out[0]), C.byref(out[1]), C.byref(out[2]), 1 if reset else 0))
        return out

    def enable_stage_timing(self, on=True):
        check(lib.rt_enable_stage_timing(self.handle, 1 if on else 0))

    def stage_timing(self, reset=False):
        """Accumulated device milliseconds of the (primary, secondary, shadow) trace kernels."""
        p, s, sh = C.c_double(), C.c_double(), C.c_double()
        check(lib.rt_get_stage_timing(self.handle, C.byref(p), C.byref(s), C.byref(sh), 1 if reset else 0))
        return p.value, s.value, sh.value


def _geometry_descs(geoms):
    descs = (T.GeometryDesc * len(geoms))()
    for d, g in zip(descs, geoms):
        if "aabbs" in g:  # procedural-primitive geometry: {aabbs: Buffer|ptr, aabb_count, stride, flags}
            d.type = T.GEOMETRY_TYPE_PROCEDURAL_AABBS
            d.vertex_buffer = _ptr(g["aabbs"])
            d.vertex_count = g["aabb_count"]
            d.vertex_stride_bytes = g.get("stride", 24)
            d.flags = g.get("flags", T.GEOMETRY_FLAG_OPAQUE)
            continue
        d.vertex_buffer = _ptr(g["vertices"])
        d.vertex_count = g["vertex_count"]
        d.vertex_stride_bytes = g.get("stride", 24)
        d.index_buffer = _ptr(g.get("indices"))
        d.index_count = g.get("index_count", 0)
        d.index_format = g.get("index_format", 32 if g.get("indices") is not None else 0)
        d.transform3x4 = _ptr(g.get("transform"))
        d.flags = g.get("flags", T.GEOMETRY_FLAG_OPAQUE)
    return descs


def _instance_descs_bytes(blases, transforms, ids=None, masks=None, hit_groups=None, flags=None) -> np.ndarray:
    n = len(blases)
    descs = (T.InstanceDesc * max(n, 1))()
    for i in range(n):
        tr = np.asarray(transforms[i], np.float32).reshape(12)
        descs[i].transform[:] = tr.tolist()
        iid = i if ids is None else ids[i]
        mask = 0xFF if masks is None else masks[i]
        hg = 2 * i if hit_groups is None else hit_groups[i]
        fl = 0 if flags is None else flags[i]
        descs[i].instance_id_and_mask = (iid & 0xFFFFFF) | ((mask & 0xFF) << 24)
        descs[i].hit_group_and_flags = (hg & 0xFFFFFF) | ((fl & 0xFF) << 24)
        descs[i].blas = blases[i].result.ptr
    return np.frombuffer(bytes(descs), dtype=np.uint8)[: 64 * n].copy() if n else np.zeros(0, np.uint8)


def _ptr(x):
    if x is None:
        return None
    if isinstance(x, Buffer):
        return x.ptr
    return int(x)


class Accel:
    """A built acceleration structure: the result buffer plus (optionally) the scratch of its build."""

    def __init__(self, ctx, result: Buffer, n: int, top: bool, scratch=None, keep=None, build_flags: int = 0):
        self.ctx, self.result, self.n, self.top, self.scratch, self._keep = ctx, result, n, top, scratch, keep
        self.build_flags = build_flags

    def info(self) -> T.AsInfo:
        i = T.AsInfo()
        check(lib.rt_as_get_info(self.ctx.handle, self.result.ptr, C.byref(i)))
        return i

    def clone(self, compact: bool = False, nbytes: int = None):
        """CopyRaytracingAccelerationStructure into a new buffer (CLONE, or COMPACT which drops the update caches)."""
        i = self.info()
        need = int(i.compacted_bytes if compact else i.total_bytes)
        dst = self.ctx.alloc(need if nbytes is None else nbytes)
        check(lib.rt_as_copy(self.ctx.handle, dst.ptr, dst.nbytes, self.result.ptr, T.COPY_MODE_COMPACT if compact else T.COPY_MODE_CLONE))
        flags = self.build_flags & ~T.BUILD_FLAG_ALLOW_UPDATE if compact else self.build_flags
        out = Accel(self.ctx, dst, self.n, self.top, keep=self._keep, build_flags=flags)
        for a in ("vb", "ib"):
            if hasattr(self, a):
                setattr(out, a, getattr(self, a))
        return out

    def update_caches(self):
        """(sort cache, parents) of an ALLOW_UPDATE build: load-order element -> sorted slot; parent of every node."""
        so, po = C.c_uint64(), C.c_uint64()
        check(lib.rt_update_cache_layout(self.n, 1 if self.top else 0, C.byref(so), C.byref(po)))
        return (self.result.download(np.uint32, self.n, offset=so.value),
                self.result.download(np.uint32, max(2 * self.n - 1, 0), offset=po.value))

    def blob(self) -> np.ndarray:
        nbytes = int(lib.rt_blob_bytes(self.n, 1 if self.top else 0))
        return self.result.download(np.uint8, nbytes)

    def ext_header(self) -> np.ndarray:
        """The 128-byte rt_ext_header behind the blob (csrc/common.cuh) as 32 little-endian 32-bit words."""
        ext = (int(lib.rt_blob_bytes(self.n, 1 if self.top else 0)) + 63) // 64 * 64
        return self.result.download(np.uint32, 32, offset=ext)

    def traversal_section(self) -> dict:
        """The arrays the trace kernels read — BVH2 wide nodes (64 B), packed leaves (48 B triangles / 96 B instances),
        4-wide nodes (128 B) — located through the rt_ext_header behind the blob."""
        hdr = self.ext_header().view(np.uint64)
        off_wide, off_leaf, off_wide4 = int(hdr[2]), int(hdr[3]), int(hdr[8])
        n_int = max(self.n - 1, 0)
        return {"wide": self.result.download(np.uint32, 16 * n_int, offset=off_wide).reshape(-1, 16),
                "leaf": self.result.download(np.uint32, (24 if self.top else 12) * self.n, offset=off_leaf),
                "wide4": self.result.download(np.uint32, 32 * n_int, offset=off_wide4).reshape(-1, 32)}

    def scratch_layout(self) -> ScratchLayout:
        L = ScratchLayout()
        check(lib.rt_build_scratch_layout(self.n, 1 if self.top else 0, C.byref(L)))
        return L

    def stage(self, name: str) -> np.ndarray:
        """Download an intermediate build product (needs keep_scratch=True)."""
        assert self.scratch is not None, "build with keep_scratch=True"
        L = self.scratch_layout()
        n = self.n
        if name in ("primitives", "metadata"):
            # load-order scratch records are 48-byte packed triangles {v[9], primitiveIndex, geometryIndex, flags}
            rec = self.scratch.download(T.PACKED_TRI_DTYPE, n, offset=L.primitives)
            if name == "primitives":
                out = np.zeros(n, T.PRIM_DTYPE)
                out["type"] = 1
                out["v"] = rec["v"]
                return out
            out = np.zeros(n, T.META_DTYPE)
            out["geom"], out["prim"], out["flags"] = rec["geom"], rec["prim"], rec["flags"]
            return out
        spec = {"scene_aabb": (np.float32, 6), "morton_codes": (np.uint32, n), "sorted_codes": (np.uint32, n),
                "sorted_indices": (np.uint32, n), "hierarchy": (T.HIER_DTYPE, max(2 * n - 1, 0))}[name]
        return self.scratch.download(spec[0], spec[1], offset=getattr(L, name))


class Program:
    """rt_program + its bindings: the compiled-in counterpart of RtProgram / RtBindings / RtState."""

    def __init__(self, ctx: Context, kind: int, hit_group_count: int = 2, miss_count: int = 2):
        self.ctx = ctx
        h = C.c_void_p()
        check(lib.rt_program_create(ctx.handle, kind, hit_group_count, miss_count, C.byref(h)))
        self.handle = h.value
        self.hit_group_count = hit_group_count
        self._keep = []

    def set_hit_record(self, ray_type, instance, vb: Buffer, ib: Buffer, material: T.MaterialParams):
        check(lib.rt_bindings_set_hit_record(self.handle, ray_type, instance, vb.ptr, ib.ptr, C.byref(material)))
        self._keep += [vb, ib]

    def set_env(self, texels: np.ndarray):
        if texels is None:
            check(lib.rt_bindings_set_miss_record(self.handle, 0, None, 0))
            return
        tex = np.ascontiguousarray(texels, np.float32)
        buf = self.ctx.upload(tex.reshape(-1))
        self._keep.append(buf)
        check(lib.rt_bindings_set_miss_record(self.handle, 0, buf.ptr, tex.shape[1]))

    def close(self):
        if self.handle:
            lib.rt_program_destroy(self.handle)
            self.handle = None


PROGRESSIVE, REALTIME = 0, 1
_AOV_IDS = {**{name: k for k, name in enumerate(T.AOV_NAMES)}, T.AOV_POSITION_NAME: T.AOV_POSITION,
            T.AOV_PREVIOUS_POSITION_NAME: T.AOV_PREVIOUS_POSITION}
assert sorted(_AOV_IDS.values()) == list(range(T.AOV_COUNT))


class Comm:
    """rt_comm: the NCCL communicator behind rt_accum_reduce (one process per GPU).

    ``exchange(id_bytes_or_None) -> id_bytes`` is the side channel that carries rank 0's 128-byte unique id to every
    rank: rank 0 calls it with the bytes, the others with None (torch.distributed broadcast, a shared file, MPI ...)."""

    def __init__(self, ctx: Context, world: int, rank: int, exchange):
        self.ctx, self.world, self.rank = ctx, world, rank
        uid = None
        if rank == 0:
            buf = (C.c_uint8 * 128)()
            check(lib.rt_comm_get_unique_id(buf))
            uid = bytes(buf)
        uid = exchange(uid)
        assert len(uid) == 128
        h = C.c_void_p()
        check(lib.rt_comm_create(ctx.handle, (C.c_uint8 * 128).from_buffer_copy(uid), world, rank, C.byref(h)))
        self.handle = h.value

    def nccl_version(self) -> int:
        v = C.c_int()
        check(lib.rt_comm_info(self.handle, None, None, C.byref(v)))
        return v.value

    def reduce(self, send_ptr, recv_ptr, count: int, weight: float, root: int = 0):
        check(lib.rt_accum_reduce(self.ctx.handle, self.handle, send_ptr, recv_ptr, count, weight, root))

    def close(self):
        if self.handle:
            lib.rt_comm_destroy(self.handle)
            self.handle = None


def file_exchange(path: str, timeout_s: float = 120.0):
    """Unique-id side channel over a shared file (no torch.distributed needed): rank 0 writes, the others poll."""
    import time

    def exchange(uid):
        if uid is not None:
            tmp = path + ".tmp"
            with open(tmp, "wb") as f:
                f.write(uid)
            os.replace(tmp, path)
            return uid
        t0 = time.time()
        while time.time() - t0 < timeout_s:
            if os.path.exists(path) and os.path.getsize(path) == 128:
                return open(path, "rb").read()
            time.sleep(0.01)
        raise TimeoutError(f"no NCCL unique id at {path}")
    return exchange


class Renderer:
    """Convenience host for tests/bench: one scene (instances of meshes), one program, fp32 outputs on the device."""

    def __init__(self, ctx: Context, meshes, transforms, materials, env_texels, kind=PROGRESSIVE, width=256, height=256,
                 outputs=None, instance_mesh=None, build_flags: int = 0, aovs=(), adaptive: bool = False, deforming=()):
        """outputs: optional list of caller-owned device buffers (anything with .ptr, e.g. a wrapped torch tensor)
        of width*height RGBA fp32, one per output slot; allocated here when omitted.
        instance_mesh: optional list, one mesh index per transform (instancing: many instances of few BLASes);
        by default instance i is mesh i.
        aovs: names from types.AOV_NAMES, types.AOV_POSITION_NAME or types.AOV_PREVIOUS_POSITION_NAME (progressive program
        only): each gets a zeroed
        width*height RGBA fp32 buffer that every dispatch accumulates next to the beauty output (rt_set_aov_output); read it
        back with aov(name).
        adaptive: sample adaptively (rt_set_adaptive_sampling, progressive program only): zeroed per-pixel sample counts and
        luminance moments that every dispatch binds; adaptive_update() marks converged pixels, which later dispatches skip.
        deforming: indices of the meshes whose vertices set_vertices() may change; their BLASes are built with
        BUILD_FLAG_ALLOW_UPDATE so that it can refit them."""
        self.ctx, self.width, self.height, self.kind = ctx, width, height, kind
        self.deforming = frozenset(int(k) for k in deforming)
        if any(not 0 <= k < len(meshes) for k in self.deforming):
            raise ValueError(f"deforming names meshes {sorted(self.deforming)}, but there are {len(meshes)}")
        # 0 = the application's flags (RtModel.cpp:86-118)
        self.blases = [ctx.build_blas_from_mesh(m, build_flags=build_flags | (T.BUILD_FLAG_ALLOW_UPDATE if k in self.deforming else 0))
                       for k, m in enumerate(meshes)]
        if instance_mesh is None:
            instance_mesh = list(range(len(meshes)))
        assert len(instance_mesh) == len(transforms)
        self.instance_mesh = list(instance_mesh)
        self.transforms = np.asarray(transforms, np.float32).reshape(len(self.instance_mesh), 12).copy()
        self.tlas = ctx.build_tlas([self.blases[k] for k in instance_mesh], self.transforms)
        self.motion = None   # (n, 12) float32 world -> previous-world matrices of the last set_transforms(), None before it
        self._motion_buf = None
        self.prev_transforms = self.transforms.copy()  # the transforms before the last set_transforms()
        self._vertices = {k: np.ascontiguousarray(meshes[k].vertices).copy() for k in self.deforming}  # host copy of each VB
        self._prev_vb = {}        # mesh -> device previous positions (a VERTEX_DTYPE array), from its first set_vertices()
        self._deform_buf = None   # one DeformationDesc per instance, from the first set_vertices()
        self.program = Program(ctx, kind)
        for i, k in enumerate(instance_mesh):
            for ray_type in range(2):
                self.program.set_hit_record(ray_type, i, self.blases[k].vb, self.blases[k].ib, materials[k])
        self.program.set_env(env_texels)
        n_out = 2 if kind == REALTIME else 1
        self.out = list(outputs) if outputs is not None else [ctx.alloc(16 * width * height).zero() for _ in range(n_out)]
        assert len(self.out) == n_out
        unknown = [a for a in aovs if a not in _AOV_IDS]
        if unknown:
            raise ValueError(f"unknown AOV names {unknown}; known: {tuple(_AOV_IDS)}")
        self.aovs = {a: ctx.alloc(16 * width * height).zero() for a in aovs}
        if adaptive and kind != PROGRESSIVE:
            raise ValueError("adaptive sampling needs the progressive program")
        self.adaptive = None  # (counts, moments, active count) device buffers
        if adaptive:
            self.adaptive = (ctx.alloc(4 * width * height).zero(), ctx.alloc(8 * width * height).zero(), ctx.alloc(4))
        self._denoise_bufs = None  # (tmp, out) of denoise(), allocated on first use
        self._last_camera = None   # cameraParams of the last dispatch
        self.reset_temporal()

    def dispatch(self, frame: T.PerFrameConstants, region=None, strips=None):
        """region: (x0, y0, x1, y1) pixel rectangle; strips: (strip_rows, groups, group) strip-interleaved shard."""
        # global root arguments are (re)bound per dispatch, as render() does (ProgressiveRaytracingPipeline.cpp:236-242)
        for slot, o in enumerate(self.out):
            check(lib.rt_set_output(self.ctx.handle, slot, o.ptr, 16 * self.width))
        for name, k in _AOV_IDS.items():  # all of them, so that AOVs another Renderer bound on this context are unbound
            buf = self.aovs.get(name)
            check(lib.rt_set_aov_output(self.ctx.handle, k, buf.ptr if buf is not None else None, 16 * self.width if buf is not None else 0))
        # every call, so that motion another Renderer bound on this context is never inherited
        self.ctx.set_instance_motion(self._motion_buf, len(self.instance_mesh) if self._motion_buf is not None else 0)
        self.ctx.set_instance_deformation(self._deform_buf, len(self.instance_mesh) if self._deform_buf is not None else 0)
        # likewise the adaptive sampling buffers
        self.ctx.set_adaptive_sampling(*(self.adaptive[:2] if self.adaptive is not None else (None, None)))
        check(lib.rt_set_tlas(self.ctx.handle, self.tlas.result.ptr))
        check(lib.rt_set_frame_constants(self.ctx.handle, C.byref(frame)))
        if strips is not None:
            check(lib.rt_dispatch_rays_interleaved(self.ctx.handle, self.program.handle, self.width, self.height, *strips))
        elif region is None:
            check(lib.rt_dispatch_rays(self.ctx.handle, self.program.handle, self.width, self.height, 3))
        else:
            x0, y0, x1, y1 = region
            check(lib.rt_dispatch_rays_region(self.ctx.handle, self.program.handle, self.width, self.height, x0, y0, x1, y1))
        self._last_camera = T.CameraParams.from_buffer_copy(bytes(frame.cameraParams))

    def _need_adaptive(self, what):
        if self.adaptive is None:
            raise ValueError(f"{what} needs a Renderer constructed with adaptive=True")

    def adaptive_update(self, params: T.AdaptiveParams = None) -> int:
        """rt_adaptive_update over the whole image: mark the pixels that have converged under `params` (default
        types.adaptive_defaults()) and return how many pixels are still active (synchronises)."""
        self._need_adaptive("adaptive_update()")
        counts, moments, active = self.adaptive
        self.ctx.adaptive_update(moments, counts, self.width, self.height, params, active)
        return int(active.download(np.uint32, 1)[0])

    def sample_counts(self):
        """(n, converged): the samples accumulated into each pixel as (height, width) uint32 and the converged mask as
        (height, width) bool."""
        self._need_adaptive("sample_counts()")
        c = self.adaptive[0].download(np.uint32).reshape(self.height, self.width)
        return c & np.uint32(~T.ADAPTIVE_CONVERGED & 0xFFFFFFFF), (c & np.uint32(T.ADAPTIVE_CONVERGED)) != 0

    def moments(self) -> np.ndarray:
        """The running luminance moments (m1, m2) of every pixel as (height, width, 2) float32."""
        self._need_adaptive("moments()")
        return self.adaptive[1].download(np.float32).reshape(self.height, self.width, 2)

    def reset_adaptive(self):
        """Start over: zero the sample counts (every pixel active again), the moments, the outputs and the AOVs."""
        self._need_adaptive("reset_adaptive()")
        for b in (*self.adaptive[:2], *self.out, *self.aovs.values()):
            b.zero()

    def set_transforms(self, transforms):
        """Move the instances: rebuild the TLAS with `transforms` (one object->world 3x4 per instance, as the constructor
        took them) and make the instance motion, which the previous-position AOV applies, the change from the transforms
        before this call to these: matrix i = prevObjectToWorld_i * inverse(objectToWorld_i), computed in float64 and
        rounded to float32.  Call it once per frame of a moving sequence (with unchanged transforms for a frame where
        nothing moves): the motion is always that of the last two calls, and none (identity) before the first."""
        new = np.asarray(transforms, np.float32)
        if new.size != 12 * len(self.instance_mesh):
            raise ValueError(f"set_transforms() needs {len(self.instance_mesh)} 3x4 transforms, got an array of {new.size} values")
        new = new.reshape(len(self.instance_mesh), 12)

        def four(t):
            m = np.zeros((t.shape[0], 4, 4))
            m[:, :3, :] = t.astype(np.float64).reshape(-1, 3, 4)
            m[:, 3, 3] = 1.0
            return m
        cur = four(new)
        if np.any(~np.isfinite(new)) or np.any(np.abs(np.linalg.det(cur)) < 1e-30):
            raise ValueError("set_transforms() needs finite, invertible transforms")
        motion = (four(self.transforms) @ np.linalg.inv(cur))[:, :3, :].reshape(-1, 12).astype(np.float32)
        self.tlas = self.ctx.build_tlas([self.blases[k] for k in self.instance_mesh], new)
        self.prev_transforms, self.transforms, self.motion = self.transforms, new.copy(), motion
        if self._motion_buf is None:
            self._motion_buf = self.ctx.alloc(48 * max(len(self.instance_mesh), 1))
        self._motion_buf.upload(motion.reshape(-1))
        if self._deform_buf is not None:
            self._upload_deformation()

    def set_vertices(self, mesh: int, positions, normals):
        """Deform mesh `mesh` (one of the constructor's deforming=): upload (V, 3) positions and normals in place of its
        vertices (same count and order; the hit records keep their buffers), refit its BLAS (PERFORM_UPDATE) and rebuild
        the TLAS.  The vertices from before this call become the mesh's previous positions, which the previous-position
        AOV carries its hit points back through (rt_set_instance_deformation), together with the transforms from before
        the last set_transforms().  Call it once per frame for each deforming mesh, as set_transforms() is called, with
        unchanged positions for a frame where the mesh rests."""
        if mesh not in self.deforming:
            raise ValueError(f"set_vertices() needs a mesh listed in deforming= ({sorted(self.deforming)}), got {mesh}")
        old = self._vertices[mesh]
        pos, nrm = np.asarray(positions, np.float32), np.asarray(normals, np.float32)
        if pos.shape != (old.shape[0], 3) or nrm.shape != (old.shape[0], 3):
            raise ValueError(f"set_vertices() needs ({old.shape[0]}, 3) positions and normals, got {pos.shape} and {nrm.shape}")
        if not (np.isfinite(pos).all() and np.isfinite(nrm).all()):
            raise ValueError("set_vertices() needs finite positions and normals")
        new = np.zeros(old.shape[0], T.VERTEX_DTYPE)
        new["position"], new["normal"] = pos, nrm
        if mesh not in self._prev_vb:
            self._prev_vb[mesh] = self.ctx.alloc(old.nbytes)
        self._prev_vb[mesh].upload(old)
        acc = self.blases[mesh]
        acc.vb.upload(new)
        self.ctx.update_blas(acc, acc._keep)
        self._vertices[mesh] = new
        self.tlas = self.ctx.build_tlas([self.blases[k] for k in self.instance_mesh], self.transforms)
        self._upload_deformation()

    def _upload_deformation(self):
        """One DeformationDesc per instance: the previous positions of its mesh (NULL while it has none) and the
        transform from before the last set_transforms()."""
        n = len(self.instance_mesh)
        descs = (T.DeformationDesc * n)()
        for i, k in enumerate(self.instance_mesh):
            prev = self._prev_vb.get(k)
            if prev is not None:
                descs[i].previous_positions = prev.ptr
                descs[i].stride_bytes = T.VERTEX_DTYPE.itemsize
                descs[i].vertex_count = self._vertices[k].shape[0]
            descs[i].object_to_previous_world[:] = self.prev_transforms[i].tolist()
        if self._deform_buf is None:
            self._deform_buf = self.ctx.alloc(C.sizeof(descs))
        self._deform_buf.upload(np.frombuffer(descs, np.uint8))

    def realtime_band(self, frame: T.PerFrameConstants, band, params: T.DenoiserParams, tmp: "Buffer", final: "Buffer"):
        """One rank's share of a realtime frame sharded by row bands (sharding.band_plan): render rows [r0, r1) of the two
        AOVs, run DenoiseCompositor on exactly those rows, and leave only the core rows [y0, y1) in `final` (a full-size,
        initially zero RGBA32F buffer) — the sum of the ranks' `final` buffers (rt_accum_reduce, weight 1) is the frame."""
        self.dispatch(frame, region=(0, band.r0, self.width, band.r1))
        row = 16 * self.width
        off = band.r0 * row
        check(lib.rt_denoise(self.ctx.handle, self.out[0].ptr + off, self.out[1].ptr + off, tmp.ptr + off, final.ptr + off,
                             self.width, band.r1 - band.r0, C.byref(params)))
        if band.y0 > band.r0:
            check(lib.rt_memset(self.ctx.handle, final.ptr + off, 0, (band.y0 - band.r0) * row))
        if band.r1 > band.y1:
            check(lib.rt_memset(self.ctx.handle, final.ptr + band.y1 * row, 0, (band.r1 - band.y1) * row))

    def image(self, slot=0) -> np.ndarray:
        return self.out[slot].download(np.float32).reshape(self.height, self.width, 4)

    def aov(self, name: str) -> np.ndarray:
        """The accumulated AOV `name` (one of the names passed as aovs=) as (height, width, 4) float32."""
        return self.aovs[name].download(np.float32).reshape(self.height, self.width, 4)

    def denoise(self, params: T.ProgressiveDenoiseParams = None) -> np.ndarray:
        """The beauty output filtered by rt_denoise_progressive with the albedo and normal AOVs as guides, as (height, width,
        4) float32.  Filters the device buffers in place of a host round trip; needs aovs= to include "albedo" and "normal"."""
        if self.kind != PROGRESSIVE or "albedo" not in self.aovs or "normal" not in self.aovs:
            raise ValueError('denoise() needs a progressive Renderer with the "albedo" and "normal" AOVs')
        if self._denoise_bufs is None:
            self._denoise_bufs = (self.ctx.alloc(32 * self.width * self.height), self.ctx.alloc(16 * self.width * self.height))
        tmp, out = self._denoise_bufs
        params = T.progressive_denoise_defaults() if params is None else params
        check(lib.rt_denoise_progressive(self.ctx.handle, self.out[0].ptr, self.aovs["albedo"].ptr, self.aovs["normal"].ptr, tmp.ptr,
                                         out.ptr, self.width, self.height, C.byref(params)))
        return out.download(np.float32).reshape(self.height, self.width, 4)

    def denoise_temporal(self, params: T.TemporalDenoiseParams = None) -> np.ndarray:
        """The last dispatch's beauty output filtered by rt_denoise_temporal, as (height, width, 4) float32: the frames
        filtered since the last reset_temporal() are the history, reprojected through the position AOV.  Needs aovs= to
        include "albedo", "normal" and "position", and a last dispatch of one sample with accumulation off (accumCount 0).
        With the "previous-position" AOV also bound it runs rt_denoise_temporal_motion, which reprojects through that AOV,
        so that instances moved by set_transforms() and meshes deformed by set_vertices() keep their history."""
        if self.kind != PROGRESSIVE or any(a not in self.aovs for a in ("albedo", "normal", T.AOV_POSITION_NAME)):
            raise ValueError('denoise_temporal() needs a progressive Renderer with the "albedo", "normal" and "position" AOVs')
        if self.adaptive is not None:
            raise ValueError("denoise_temporal() filters frames of one sample, which adaptive sampling does not make")
        if self._last_camera is None or self._last_camera.accumCount != 0:
            raise ValueError("denoise_temporal() filters frames of one sample: the last dispatch must have accumCount 0")
        if self._temporal is None:
            px = self.width * self.height
            self._temporal = [self.ctx.alloc(64 * px), self.ctx.alloc(64 * px), self.ctx.alloc(32 * px), self.ctx.alloc(16 * px)]
        prev, hist, tmp, out = self._temporal
        params = T.temporal_denoise_defaults() if params is None else params
        prev_cam = self._prev_camera
        guides = (self.out[0].ptr, self.aovs["albedo"].ptr, self.aovs["normal"].ptr, self.aovs[T.AOV_POSITION_NAME].ptr)
        history = (C.byref(prev_cam) if prev_cam is not None else None, prev.ptr if prev_cam is not None else None, hist.ptr,
                   tmp.ptr, out.ptr, self.width, self.height, C.byref(params))
        if T.AOV_PREVIOUS_POSITION_NAME in self.aovs:
            check(lib.rt_denoise_temporal_motion(self.ctx.handle, *guides, self.aovs[T.AOV_PREVIOUS_POSITION_NAME].ptr, *history))
        else:
            check(lib.rt_denoise_temporal(self.ctx.handle, *guides, *history))
        self._temporal[0], self._temporal[1] = hist, prev  # this frame's history is the next call's prev_history
        self._prev_camera = T.CameraParams.from_buffer_copy(bytes(self._last_camera))
        return out.download(np.float32).reshape(self.height, self.width, 4)

    def temporal_history(self) -> np.ndarray:
        """The history the last denoise_temporal() wrote, as (4, height, width, 4) float32 (planes as in include/rt_core.h)."""
        return self._temporal[0].download(np.float32).reshape(4, self.height, self.width, 4)

    def reset_temporal(self):
        """Drop the history: the next denoise_temporal() filters its frame as a first frame."""
        self._temporal = None
        self._prev_camera = None
