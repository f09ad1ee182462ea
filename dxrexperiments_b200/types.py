"""ctypes / numpy mirrors of ``include/rt_types.h``.

Every structure here is byte-compatible with the C declaration of the same name, which in turn
is byte-compatible with the reference struct it cites (see the header).  Sizes are asserted at
import time so that a drift between the header and this file fails loudly.
"""
import ctypes as C

import numpy as np

F4 = C.c_float * 4


class CameraParams(C.Structure):  # assets/shaders/RaytracingHlslCompat.h:41-50
    _fields_ = [("worldEyePos", F4), ("U", F4), ("V", F4), ("W", F4), ("jitters", C.c_float * 2),
                ("frameCount", C.c_uint32), ("accumCount", C.c_uint32)]


class DirectionalLight(C.Structure):  # :52-56
    _fields_ = [("forwardDir", F4), ("color", F4)]


class PointLight(C.Structure):  # :58-62
    _fields_ = [("worldPos", F4), ("color", F4)]


class DebugOptions(C.Structure):  # :64-77
    _fields_ = [("maxIterations", C.c_uint32), ("cosineHemisphereSampling", C.c_uint32),
                ("showIndirectDiffuseOnly", C.c_uint32), ("showIndirectSpecularOnly", C.c_uint32),
                ("showAmbientOcclusionOnly", C.c_uint32), ("showGBufferAlbedoOnly", C.c_uint32),
                ("showDirectLightingOnly", C.c_uint32), ("showFresnelTerm", C.c_uint32),
                ("noIndirectDiffuse", C.c_uint32), ("environmentStrength", C.c_float), ("debug", C.c_uint32)]


class PerFrameConstants(C.Structure):  # :79-85
    _fields_ = [("cameraParams", CameraParams), ("directionalLight", DirectionalLight),
                ("pointLight", PointLight), ("options", DebugOptions)]


class MaterialParams(C.Structure):  # :87-96
    _fields_ = [("albedo", F4), ("specular", F4), ("emissive", F4), ("reflectivity", C.c_float),
                ("roughness", C.c_float), ("IoR", C.c_float), ("type", C.c_uint32)]


class DenoiserParams(C.Structure):  # include/DenoiseCompositor.h:41-49
    _fields_ = [("exposure", C.c_float), ("gamma", C.c_float), ("tonemap", C.c_uint32),
                ("gammaCorrect", C.c_uint32), ("maxKernelSize", C.c_int32), ("debugVisualize", C.c_uint32)]


class ProgressiveDenoiseParams(C.Structure):  # rt_progressive_denoise_params (include/rt_types.h)
    _fields_ = [("iterations", C.c_uint32), ("normal_exponent_log2", C.c_uint32), ("sigma_luminance", C.c_float),
                ("sigma_albedo", C.c_float)]


def progressive_denoise_defaults() -> ProgressiveDenoiseParams:
    """RT_PROGRESSIVE_DENOISE_DEFAULTS (include/rt_types.h): the parameters rt_denoise_progressive is used with unless told
    otherwise (DESIGN.md 4.4 records how they were chosen)."""
    return ProgressiveDenoiseParams(5, 7, 4.0, 0.1)


class TemporalDenoiseParams(C.Structure):  # rt_temporal_denoise_params (include/rt_types.h)
    _fields_ = [("spatial", ProgressiveDenoiseParams), ("alpha_color", C.c_float), ("alpha_moments", C.c_float),
                ("normal_cos", C.c_float), ("position_tolerance", C.c_float)]


def temporal_denoise_defaults() -> TemporalDenoiseParams:
    """RT_TEMPORAL_DENOISE_DEFAULTS (include/rt_types.h): the parameters rt_denoise_temporal is used with unless told
    otherwise (DESIGN.md 4.4.2 records how they were chosen)."""
    return TemporalDenoiseParams(progressive_denoise_defaults(), 0.2, 0.2, 0.9, 0.02)


class AdaptiveParams(C.Structure):  # rt_adaptive_params (include/rt_types.h)
    _fields_ = [("threshold", C.c_float), ("floor", C.c_float), ("min_samples", C.c_uint32), ("max_samples", C.c_uint32)]


def adaptive_defaults() -> AdaptiveParams:
    """RT_ADAPTIVE_DEFAULTS (include/rt_types.h): the parameters rt_adaptive_update is used with unless told otherwise
    (DESIGN.md 4.6 records how they were chosen)."""
    return AdaptiveParams(0.1, 0.1, 8, 1024)


# bit 31 of an adaptive sample count (RT_ADAPTIVE_CONVERGED): the pixel has converged and dispatches skip it
ADAPTIVE_CONVERGED = 0x80000000


class DeformationDesc(C.Structure):  # rt_deformation_desc (include/rt_types.h), one per InstanceIndex()
    _fields_ = [("previous_positions", C.c_void_p), ("stride_bytes", C.c_uint32), ("vertex_count", C.c_uint32),
                ("object_to_previous_world", C.c_float * 12)]


class GeometryDesc(C.Structure):
    _fields_ = [("vertex_buffer", C.c_void_p), ("vertex_count", C.c_uint32), ("vertex_stride_bytes", C.c_uint32),
                ("index_buffer", C.c_void_p), ("index_count", C.c_uint32), ("index_format", C.c_uint32),
                ("transform3x4", C.c_void_p), ("flags", C.c_uint32), ("type", C.c_uint32)]


class InstanceDesc(C.Structure):  # D3D12_RAYTRACING_FALLBACK_INSTANCE_DESC
    _fields_ = [("transform", C.c_float * 12), ("instance_id_and_mask", C.c_uint32),
                ("hit_group_and_flags", C.c_uint32), ("blas", C.c_uint64)]


class EnvCube(C.Structure):
    _fields_ = [("texels", C.c_void_p), ("size", C.c_uint32), ("_pad", C.c_uint32)]


class HitRecord(C.Structure):
    _fields_ = [("vertex_buffer", C.c_void_p), ("index_buffer", C.c_void_p), ("material", MaterialParams)]


class TraceStats(C.Structure):
    _fields_ = [("rays", C.c_uint64), ("internal_visits", C.c_uint64), ("leaf_visits", C.c_uint64),
                ("instance_visits", C.c_uint64), ("max_stack", C.c_uint64)]


class RayCounts(C.Structure):
    _fields_ = [("primary", C.c_uint64), ("secondary", C.c_uint64), ("shadow", C.c_uint64)]


class PrebuildInfo(C.Structure):
    _fields_ = [("result_bytes", C.c_uint64), ("scratch_bytes", C.c_uint64), ("update_scratch_bytes", C.c_uint64)]


class AsInfo(C.Structure):  # rt_as_info
    _fields_ = [("count", C.c_uint32), ("top_level", C.c_uint32), ("build_flags", C.c_uint32), ("has_procedural", C.c_uint32),
                ("blob_bytes", C.c_uint64), ("total_bytes", C.c_uint64), ("compacted_bytes", C.c_uint64)]


assert C.sizeof(PerFrameConstants) == 188
assert C.sizeof(MaterialParams) == 64
assert C.sizeof(DenoiserParams) == 24
assert C.sizeof(ProgressiveDenoiseParams) == 16
assert C.sizeof(TemporalDenoiseParams) == 32
assert C.sizeof(AdaptiveParams) == 16
assert C.sizeof(DeformationDesc) == 64
assert C.sizeof(InstanceDesc) == 64
assert C.sizeof(HitRecord) == 80
assert C.sizeof(GeometryDesc) == 48

# numpy record layouts of the wavefront records and of the acceleration-structure blob
RAY_DTYPE = np.dtype([("origin", "<f4", 3), ("tmin", "<f4"), ("direction", "<f4", 3), ("tmax", "<f4")])
HIT_DTYPE = np.dtype([("t", "<f4"), ("bary", "<f4", 2), ("primitive_index", "<u4"), ("instance_index", "<u4"),
                      ("geometry_index", "<u4"), ("instance_id", "<u4"), ("leaf_slot", "<u4")])
NODE_DTYPE = np.dtype([("center", "<f4", 3), ("flags", "<u4"), ("halfDim", "<f4", 3), ("right", "<u4")])
PRIM_DTYPE = np.dtype([("type", "<u4"), ("v", "<f4", 9)])
META_DTYPE = np.dtype([("geom", "<u4"), ("prim", "<u4"), ("flags", "<u4")])
PACKED_TRI_DTYPE = np.dtype([("v", "<f4", 9), ("prim", "<u4"), ("geom", "<u4"), ("flags", "<u4")])  # csrc/common.cuh rt_packed_tri
HIER_DTYPE = np.dtype([("parent", "<u4"), ("left", "<u4"), ("right", "<u4")])
BVH_METADATA_DTYPE = np.dtype([("w2o", "<f4", 12), ("id_mask", "<u4"), ("hg_flags", "<u4"), ("blas", "<u8"),
                               ("o2w", "<f4", 12), ("instance_index", "<u4")])
VERTEX_DTYPE = np.dtype([("position", "<f4", 3), ("normal", "<f4", 3)])
assert RAY_DTYPE.itemsize == 32 and HIT_DTYPE.itemsize == 32 and NODE_DTYPE.itemsize == 32
assert PRIM_DTYPE.itemsize == 40 and META_DTYPE.itemsize == 12 and BVH_METADATA_DTYPE.itemsize == 116
assert VERTEX_DTYPE.itemsize == 24

NO_HIT = 0xFFFFFFFF
LEAF_FLAG = 0x80000000

PROCEDURAL_FLAG = 0x40000000
RAY_FLAG_NONE = 0x00
RAY_FLAG_FORCE_OPAQUE = 0x01
RAY_FLAG_FORCE_NON_OPAQUE = 0x02
RAY_FLAG_CULL_OPAQUE = 0x40
RAY_FLAG_CULL_NON_OPAQUE = 0x80
RAY_FLAG_ACCEPT_FIRST_HIT_AND_END_SEARCH = 0x04
RAY_FLAG_SKIP_CLOSEST_HIT_SHADER = 0x08
RAY_FLAG_CULL_BACK_FACING_TRIANGLES = 0x10
RAY_FLAG_CULL_FRONT_FACING_TRIANGLES = 0x20
BUILD_FLAG_NONE = 0
BUILD_FLAG_ALLOW_UPDATE = 0x1
BUILD_FLAG_ALLOW_COMPACTION = 0x2
BUILD_FLAG_PREFER_FAST_TRACE = 0x4
BUILD_FLAG_PREFER_FAST_BUILD = 0x8
BUILD_FLAG_MINIMIZE_MEMORY = 0x10
BUILD_FLAG_PERFORM_UPDATE = 0x20
COPY_MODE_CLONE, COPY_MODE_COMPACT = 0, 1
INSTANCE_FLAG_NONE = 0
INSTANCE_FLAG_TRIANGLE_CULL_DISABLE = 0x1
INSTANCE_FLAG_TRIANGLE_FRONT_COUNTERCLOCKWISE = 0x2
INSTANCE_FLAG_FORCE_OPAQUE = 0x4
INSTANCE_FLAG_FORCE_NON_OPAQUE = 0x8
GEOMETRY_FLAG_NONE = 0
GEOMETRY_FLAG_OPAQUE = 0x1
GEOMETRY_TYPE_TRIANGLES, GEOMETRY_TYPE_PROCEDURAL_AABBS = 0, 1
PRIMITIVE_TYPE_TRIANGLE, PRIMITIVE_TYPE_PROCEDURAL = 1, 2
ANYHIT_NONE, ANYHIT_ACCEPT, ANYHIT_IGNORE, ANYHIT_END_SEARCH, ANYHIT_CUTOUT = 0, 1, 2, 3, 4
INTERSECTION_NONE, INTERSECTION_BOX, INTERSECTION_SPHERE = 0, 1, 2
HIT_KIND_TRIANGLE_FRONT_FACE = 0xFE
# rt_aov (include/rt_core.h): AOV outputs of the progressive program, in id order
(AOV_DIRECT, AOV_INDIRECT_DIFFUSE, AOV_INDIRECT_SPECULAR, AOV_ALBEDO, AOV_FRESNEL, AOV_NORMAL, AOV_POSITION, AOV_PREVIOUS_POSITION,
 AOV_COUNT) = range(9)
# the names of AOVs 0-5: the five debug-view terms and the normal
AOV_NAMES = ("direct", "indirect-diffuse", "indirect-specular", "albedo", "fresnel", "normal")
# the world-position AOV (what rt_denoise_temporal reprojects through), kept out of AOV_NAMES, which names AOVs 0-5 only
AOV_POSITION_NAME = "position"
# the same hit point carried into the previous frame by its instance's motion (what rt_denoise_temporal_motion reprojects
# through), also kept out of AOV_NAMES
AOV_PREVIOUS_POSITION_NAME = "previous-position"


def parse_blas_blob(blob: np.ndarray):
    """Split a BLAS blob ([BVHOffsets][2N-1 AABBNode][N Primitive][N PrimitiveMetaData]) into arrays."""
    blob = np.ascontiguousarray(blob, dtype=np.uint8)
    hdr = blob[:16].view("<u4")
    off_boxes, off_prims, off_meta, total = (int(x) for x in hdr)
    n = (off_meta - off_prims) // 40
    nodes = blob[off_boxes:off_prims].view(NODE_DTYPE)
    prims = blob[off_prims:off_meta].view(PRIM_DTYPE)
    meta = blob[off_meta:off_meta + 12 * n].view(META_DTYPE)
    return {"n": n, "header": hdr.copy(), "nodes": nodes, "prims": prims, "meta": meta, "total": total}


def parse_tlas_blob(blob: np.ndarray):
    """Split a TLAS blob ([BVHOffsets][I-1 internal + I leaf AABBNode][I BVHMetadata]) into arrays."""
    blob = np.ascontiguousarray(blob, dtype=np.uint8)
    hdr = blob[:16].view("<u4")
    off_boxes, off_meta, _, total = (int(x) for x in hdr)
    n = (total - off_meta) // 116
    nodes = blob[off_boxes:off_meta].view(NODE_DTYPE)
    meta = blob[off_meta:off_meta + 116 * n].view(BVH_METADATA_DTYPE)
    return {"n": n, "header": hdr.copy(), "nodes": nodes, "meta": meta, "total": total}
