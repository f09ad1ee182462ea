"""ctypes loader for the CPU oracle (``oracle/liboracle.so``).

TEST INFRASTRUCTURE, NOT PRODUCT — see oracle/oracle.h.  Importable only from tests/, from
``__graft_entry__.smoke()`` and from ``bench.py``'s cpu_baseline / ``--impl reference`` legs.
"""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from dxrexperiments_b200 import types as T

_DIR = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_DIR, "liboracle.so")


def build(force: bool = False) -> str:
    srcs = [os.path.join(_DIR, f) for f in os.listdir(_DIR) if f.endswith((".cpp", ".h"))]
    srcs.append(os.path.join(_DIR, "..", "include", "rt_types.h"))
    stale = force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs)
    if stale:
        subprocess.run(["make", "-C", _DIR, "-s"], check=True)
    return _SO


def use_native() -> str:
    """CPU-baseline build of the same sources: -O3 -march=native, compiled ON THE MACHINE THAT RUNS IT, into a temporary
    directory removed at exit (the tree is left untouched and may be read-only, and a library built for another CPU
    never travels with it).  Must be called before the first lib() call; falls back to the portable -O2 library if the
    compile fails.  Returns the flags in use."""
    global _SO
    if _lib is not None:  # already loaded: report what is in use
        return "-O3 -march=native -ffp-contract=off" if _SO.endswith("liboracle_native.so") else "-O2 -ffp-contract=off"
    out_dir = tempfile.mkdtemp(prefix="oracle_native_")
    atexit.register(shutil.rmtree, out_dir, ignore_errors=True)
    try:
        subprocess.run(["make", "-C", _DIR, "-s", "native", f"NATIVE_DIR={out_dir}"], check=True, capture_output=True, timeout=600)
        _SO = os.path.join(out_dir, "liboracle_native.so")
        return "-O3 -march=native -ffp-contract=off"
    except Exception:
        return "-O2 -ffp-contract=off (native build failed)"


_lib = None


def lib():
    global _lib
    if _lib is None:
        if _SO.endswith("liboracle.so"):
            build()
        L = C.CDLL(_SO)
        vp, u32, u64, i32, f32p = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int, C.POINTER(C.c_float)
        L.orc_scene_aabb.argtypes = [vp, u32, vp]
        L.orc_morton_codes.argtypes = [vp, u32, vp, vp]
        L.orc_morton_code_from_centroid.argtypes = [vp, vp]
        L.orc_morton_code_from_centroid.restype = u32
        L.orc_sort_pairs.argtypes = [vp, u32, vp, vp]
        L.orc_build_hierarchy.argtypes = [vp, u32, vp]
        L.orc_treelet_optimise.argtypes = [u32, vp, vp, u32]
        L.orc_init_rand.argtypes = [u32, u32]
        L.orc_init_rand.restype = u32
        L.orc_next_rand.argtypes = [C.POINTER(u32)]
        L.orc_next_rand.restype = C.c_float
        L.orc_blas_build.argtypes = [vp, u32, u32]
        L.orc_blas_build.restype = vp
        L.orc_blas_free.argtypes = [vp]
        L.orc_blas_num_prims.argtypes = [vp]
        L.orc_blas_num_prims.restype = u32
        for name in ("unsorted_prims", "scene_aabb", "morton", "sorted_morton", "perm", "hierarchy"):
            f = getattr(L, "orc_blas_" + name)
            f.argtypes = [vp]
            f.restype = vp
        L.orc_blas_blob.argtypes = [vp, C.POINTER(u64)]
        L.orc_blas_blob.restype = vp
        L.orc_blas_update.argtypes = [vp, vp, u32]
        L.orc_blas_update.restype = i32
        for name in ("orc_blas_sort_cache", "orc_blas_parents", "orc_tlas_sort_cache", "orc_tlas_parents"):
            getattr(L, name).argtypes = [vp]
            getattr(L, name).restype = vp
        L.orc_tlas_update.argtypes = [vp, vp, u32]
        L.orc_tlas_update.restype = i32
        L.orc_tlas_build.argtypes = [vp, u32, u32]
        L.orc_tlas_build.restype = vp
        L.orc_tlas_free.argtypes = [vp]
        L.orc_tlas_blob.argtypes = [vp, C.POINTER(u64)]
        L.orc_tlas_blob.restype = vp
        L.orc_tlas_sorted_morton.argtypes = [vp]
        L.orc_tlas_sorted_morton.restype = vp
        L.orc_tlas_perm.argtypes = [vp]
        L.orc_tlas_perm.restype = vp
        L.orc_trace.argtypes = [vp, vp, u64, u32, u32, vp, vp, i32]
        L.orc_trace_hit_groups.argtypes = [vp, vp, u64, u32, u32, u32, u32, vp, u32, vp, i32]
        L.orc_render_progressive.argtypes = [vp, vp, u32, vp, vp, u32, u32, vp, i32, vp, vp]
        L.orc_render_realtime.argtypes = [vp, vp, u32, vp, vp, u32, u32, vp, vp, i32, vp]
        L.orc_denoise.argtypes = [vp, vp, vp, vp, u32, u32, vp, i32]
        L.orc_primary_ray.argtypes = [vp, u32, u32, u32, u32, C.c_float, vp]
        L.orc_primary_rays.argtypes = [vp, u32, u32, C.c_float, vp]
        L.orc_sample_env.argtypes = [vp, vp, vp]
        L.orc_set_render_options.argtypes = [u32, i32]
        _lib = L
    return _lib


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _view(addr, count, dtype):
    if count == 0 or not addr:
        return np.zeros(0, dtype=dtype)
    nbytes = count * np.dtype(dtype).itemsize
    buf = (C.c_uint8 * nbytes).from_address(addr)
    return np.frombuffer(buf, dtype=dtype, count=count).copy()


# ------------------------------------------------------------------ stage functions

def prims_from_triangles(tris: np.ndarray) -> np.ndarray:
    """(N,3,3) float32 -> rt_primitive records (type 1)."""
    p = np.zeros(tris.shape[0], dtype=T.PRIM_DTYPE)
    p["type"] = 1
    p["v"] = tris.reshape(-1, 9).astype(np.float32)
    return p


def scene_aabb(prims: np.ndarray) -> np.ndarray:
    out = np.zeros(6, np.float32)
    lib().orc_scene_aabb(_ptr(prims), prims.shape[0], _ptr(out))
    return out


def morton_codes(prims: np.ndarray, aabb: np.ndarray) -> np.ndarray:
    out = np.zeros(prims.shape[0], np.uint32)
    aabb = np.ascontiguousarray(aabb, np.float32)
    lib().orc_morton_codes(_ptr(prims), prims.shape[0], _ptr(aabb), _ptr(out))
    return out


def morton_code_from_centroid(centroid, aabb) -> int:
    c = np.ascontiguousarray(centroid, np.float32)
    a = np.ascontiguousarray(aabb, np.float32)
    return int(lib().orc_morton_code_from_centroid(_ptr(c), _ptr(a)))


def sort_pairs(codes: np.ndarray):
    codes = np.ascontiguousarray(codes, np.uint32)
    s = np.zeros_like(codes)
    p = np.zeros_like(codes)
    lib().orc_sort_pairs(_ptr(codes), codes.size, _ptr(s), _ptr(p))
    return s, p


def build_hierarchy(sorted_codes: np.ndarray) -> np.ndarray:
    sorted_codes = np.ascontiguousarray(sorted_codes, np.uint32)
    n = sorted_codes.size
    h = np.zeros(max(2 * n - 1, 0), dtype=T.HIER_DTYPE)
    lib().orc_build_hierarchy(_ptr(sorted_codes), n, _ptr(h))
    return h


def treelet_optimise(hier: np.ndarray, sorted_prims: np.ndarray, build_flags: int = 0) -> np.ndarray:
    """FL/TreeletReorder.cpp:38-109 on a copy of `hier` (2n-1 {parent,left,right}) over n sorted rt_primitive records."""
    h = np.ascontiguousarray(hier, dtype=T.HIER_DTYPE).copy()
    prims = np.ascontiguousarray(sorted_prims, dtype=T.PRIM_DTYPE)
    assert h.shape[0] == 2 * prims.shape[0] - 1
    lib().orc_treelet_optimise(prims.shape[0], _ptr(h), _ptr(prims), build_flags)
    return h


def init_rand(v0: int, v1: int) -> int:
    return int(lib().orc_init_rand(v0 & 0xFFFFFFFF, v1 & 0xFFFFFFFF))


def next_rand(state: int):
    s = C.c_uint32(state)
    v = lib().orc_next_rand(C.byref(s))
    return float(v), int(s.value)


# ------------------------------------------------------------------ acceleration structures

class Blas:
    def __init__(self, geoms, build_flags: int = 0):
        """geoms: list of dicts {vertices (V,k) float32 array or structured, stride, indices (uint16/uint32 or None),
        transform (12,) or None, flags}, or {aabbs (A,6+) float32, stride, flags} for procedural-primitive geometry."""
        descs = self._descs(geoms)
        self.handle = lib().orc_blas_build(descs, len(geoms), build_flags)
        self.n = int(lib().orc_blas_num_prims(self.handle))

    def update(self, geoms):
        """PERFORM_UPDATE with new vertex data (same triangle count and order), in place."""
        descs = self._descs(geoms)
        rc = lib().orc_blas_update(self.handle, descs, len(geoms))
        if rc != 0:
            raise ValueError("update: primitive count differs from the original build")

    def sort_cache(self):
        return _view(lib().orc_blas_sort_cache(self.handle), self.n, np.uint32)

    def parents(self):
        return _view(lib().orc_blas_parents(self.handle), max(2 * self.n - 1, 0), np.uint32)

    def _descs(self, geoms):
        self._keep = []
        descs = (T.GeometryDesc * len(geoms))()
        for d, g in zip(descs, geoms):
            if "aabbs" in g:
                vb = np.ascontiguousarray(g["aabbs"], np.float32)
                self._keep.append(vb)
                d.type = T.GEOMETRY_TYPE_PROCEDURAL_AABBS
                d.vertex_buffer = vb.ctypes.data
                d.vertex_stride_bytes = int(g.get("stride", vb.strides[0]))
                d.vertex_count = vb.shape[0]
                d.flags = int(g.get("flags", T.GEOMETRY_FLAG_OPAQUE))
                continue
            vb = np.ascontiguousarray(g["vertices"])
            self._keep.append(vb)
            d.vertex_buffer = vb.ctypes.data
            d.vertex_stride_bytes = int(g.get("stride", vb.strides[0]))
            d.vertex_count = vb.shape[0]
            ib = g.get("indices")
            if ib is not None:
                ib = np.ascontiguousarray(ib)
                self._keep.append(ib)
                d.index_buffer = ib.ctypes.data
                d.index_count = ib.size
                d.index_format = 16 if ib.dtype == np.uint16 else 32
            tr = g.get("transform")
            if tr is not None:
                tr = np.ascontiguousarray(tr, np.float32)
                self._keep.append(tr)
                d.transform3x4 = tr.ctypes.data
            d.flags = int(g.get("flags", T.GEOMETRY_FLAG_OPAQUE))
        return descs

    @classmethod
    def from_mesh(cls, mesh, flags=T.GEOMETRY_FLAG_OPAQUE, build_flags: int = 0):
        return cls([dict(vertices=mesh.vertices, stride=24, indices=mesh.indices, flags=flags)], build_flags)

    def __del__(self):
        if getattr(self, "handle", None):
            lib().orc_blas_free(self.handle)
            self.handle = None

    def unsorted_prims(self):
        return _view(lib().orc_blas_unsorted_prims(self.handle), self.n, T.PRIM_DTYPE)

    def scene_aabb(self):
        return _view(lib().orc_blas_scene_aabb(self.handle), 6, np.float32)

    def morton(self):
        return _view(lib().orc_blas_morton(self.handle), self.n, np.uint32)

    def sorted_morton(self):
        return _view(lib().orc_blas_sorted_morton(self.handle), self.n, np.uint32)

    def perm(self):
        return _view(lib().orc_blas_perm(self.handle), self.n, np.uint32)

    def hierarchy(self):
        return _view(lib().orc_blas_hierarchy(self.handle), max(2 * self.n - 1, 0), T.HIER_DTYPE)

    def blob(self):
        nbytes = C.c_uint64(0)
        addr = lib().orc_blas_blob(self.handle, C.byref(nbytes))
        return _view(addr, int(nbytes.value), np.uint8)


def make_instance_descs(blas_handles, transforms, ids=None, masks=None, hit_groups=None, flags=None):
    """Array of rt_instance_desc; defaults follow RtScene::build + TopLevelASGenerator (mask 0xFF, flags NONE,
    id = i, hit group = i * 2)."""
    n = len(blas_handles)
    arr = (T.InstanceDesc * n)()
    for i in range(n):
        tr = np.asarray(transforms[i], np.float32).reshape(12)
        arr[i].transform[:] = tr.tolist()
        iid = i if ids is None else ids[i]
        mask = 0xFF if masks is None else masks[i]
        hg = 2 * i if hit_groups is None else hit_groups[i]
        fl = 0 if flags is None else flags[i]
        arr[i].instance_id_and_mask = (iid & 0xFFFFFF) | ((mask & 0xFF) << 24)
        arr[i].hit_group_and_flags = (hg & 0xFFFFFF) | ((fl & 0xFF) << 24)
        arr[i].blas = int(blas_handles[i])
    return arr


class Tlas:
    def __init__(self, blases, transforms, ids=None, masks=None, hit_groups=None, flags=None, build_flags=0):
        self.blases = list(blases)
        descs = make_instance_descs([b.handle for b in self.blases], transforms, ids, masks, hit_groups, flags)
        self.n = len(self.blases)
        self.handle = lib().orc_tlas_build(descs, self.n, build_flags)

    def __del__(self):
        if getattr(self, "handle", None):
            lib().orc_tlas_free(self.handle)
            self.handle = None

    def update(self, transforms, ids=None, masks=None, hit_groups=None, flags=None):
        """PERFORM_UPDATE: same instances in the same order, new transforms / ids / masks / flags."""
        descs = make_instance_descs([b.handle for b in self.blases], transforms, ids, masks, hit_groups, flags)
        if lib().orc_tlas_update(self.handle, descs, self.n) != 0:
            raise ValueError("update: instance count differs from the original build")

    def sort_cache(self):
        return _view(lib().orc_tlas_sort_cache(self.handle), self.n, np.uint32)

    def parents(self):
        return _view(lib().orc_tlas_parents(self.handle), max(2 * self.n - 1, 0), np.uint32)

    def blob(self):
        nbytes = C.c_uint64(0)
        addr = lib().orc_tlas_blob(self.handle, C.byref(nbytes))
        return _view(addr, int(nbytes.value), np.uint8)

    def sorted_morton(self):
        return _view(lib().orc_tlas_sorted_morton(self.handle), self.n, np.uint32)

    def perm(self):
        return _view(lib().orc_tlas_perm(self.handle), self.n, np.uint32)

    def trace(self, rays: np.ndarray, ray_flags: int = 0, mask: int = 0xFF, threads: int = 1, stats=None):
        rays = np.ascontiguousarray(rays, dtype=T.RAY_DTYPE)
        hits = np.zeros(rays.shape[0], dtype=T.HIT_DTYPE)
        st = stats if stats is not None else T.TraceStats()
        lib().orc_trace(self.handle, _ptr(rays), rays.shape[0], ray_flags, mask, _ptr(hits), C.byref(st), threads)
        return hits

    def trace_hit_groups(self, rays: np.ndarray, programs, ray_flags: int = 0, mask: int = 0xFF, ray_contribution: int = 0,
                         geometry_multiplier: int = 0, threads: int = 1):
        """programs: (R, 2) uint32 {any_hit, intersection} per hit-group record.  leaf_slot carries HitKind() << 24."""
        rays = np.ascontiguousarray(rays, dtype=T.RAY_DTYPE)
        hits = np.zeros(rays.shape[0], dtype=T.HIT_DTYPE)
        progs = np.ascontiguousarray(programs, np.uint32).reshape(-1, 2)
        lib().orc_trace_hit_groups(self.handle, _ptr(rays), rays.shape[0], ray_flags, mask, ray_contribution, geometry_multiplier,
                                   _ptr(progs), progs.shape[0], _ptr(hits), threads)
        return hits


# ------------------------------------------------------------------ pipelines

class Records:
    """Hit-group record table indexed by hit-group record index (instance * hitGroupCount + rayType)."""

    def __init__(self, meshes, materials, hit_group_count: int = 2):
        self._keep = []
        n = len(meshes) * hit_group_count
        self.arr = (T.HitRecord * n)()
        for i, (m, mat) in enumerate(zip(meshes, materials)):
            vb = np.ascontiguousarray(m.vertices)
            ib = np.ascontiguousarray(m.indices, np.uint32)
            self._keep += [vb, ib]
            for r in range(hit_group_count):
                rec = self.arr[i * hit_group_count + r]
                rec.vertex_buffer = vb.ctypes.data
                rec.index_buffer = ib.ctypes.data
                rec.material = mat
        self.n = n


def env_cube(texels):
    e = T.EnvCube()
    if texels is None:
        return e, None
    tex = np.ascontiguousarray(texels, np.float32)
    e.texels = tex.ctypes.data
    e.size = tex.shape[1]
    return e, tex


def set_render_options(max_radiance_ray_depth: int = 1, half_render_targets: bool = False):
    """MAX_RADIANCE_RAY_DEPTH (1 = the reference) and R16G16B16A16_FLOAT target emulation; process-wide."""
    lib().orc_set_render_options(max_radiance_ray_depth, 1 if half_render_targets else 0)


def render_progressive(tlas: Tlas, records: Records, env_texels, frame: T.PerFrameConstants, width, height,
                       accum: np.ndarray, threads: int = 1, counts=None, secondary_stats=None):
    e, keep = env_cube(env_texels)
    assert accum.dtype == np.float32 and accum.size == width * height * 4 and accum.flags.c_contiguous
    lib().orc_render_progressive(tlas.handle, records.arr, records.n, C.byref(e), C.byref(frame), width, height,
                                 _ptr(accum), threads, C.byref(counts) if counts is not None else None,
                                 C.byref(secondary_stats) if secondary_stats is not None else None)
    return accum


def render_realtime(tlas: Tlas, records: Records, env_texels, frame, width, height, threads: int = 1, counts=None):
    e, keep = env_cube(env_texels)
    direct = np.zeros((height, width, 4), np.float32)
    spec = np.zeros((height, width, 4), np.float32)
    lib().orc_render_realtime(tlas.handle, records.arr, records.n, C.byref(e), C.byref(frame), width, height,
                              _ptr(direct), _ptr(spec), threads, C.byref(counts) if counts is not None else None)
    return direct, spec


def denoise(direct: np.ndarray, spec: np.ndarray, params: T.DenoiserParams, threads: int = 1):
    h, w = direct.shape[:2]
    direct = np.ascontiguousarray(direct, np.float32)
    spec = np.ascontiguousarray(spec, np.float32)
    tmp = np.zeros_like(direct)
    out = np.zeros_like(direct)
    lib().orc_denoise(_ptr(direct), _ptr(spec), _ptr(tmp), _ptr(out), w, h, C.byref(params), threads)
    return out, tmp


def primary_rays(frame, width, height, jitter_scale=30.0) -> np.ndarray:
    rays = np.zeros(width * height, dtype=T.RAY_DTYPE)
    lib().orc_primary_rays(C.byref(frame), width, height, jitter_scale, _ptr(rays))
    return rays


def sample_env(env_texels, dirs: np.ndarray) -> np.ndarray:
    e, keep = env_cube(env_texels)
    dirs = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
    out = np.zeros_like(dirs)
    L = lib()
    for i in range(dirs.shape[0]):
        L.orc_sample_env(C.byref(e), dirs[i].ctypes.data_as(C.c_void_p), out[i].ctypes.data_as(C.c_void_p))
    return out
