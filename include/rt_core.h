/*
 * rt_core.h — C ABI of the B200 ray-tracing core (librt_core.so).
 *
 * This is the drop-in boundary: the DXRFramework-style host classes (RtContext, RtModel, RtScene,
 * RtProgram, RtBindings, RtState, the two RaytracingPipelines and the DenoiseCompositor) call
 * these entry points where the reference calls the COM interfaces of the D3D12 Raytracing
 * Fallback Layer (externals/D3D12RaytracingFallback/Include/D3D12RaytracingFallback.h:46-171).
 * Each function cites the reference interface it replaces.  Paths are relative to /root/reference.
 *
 * Conventions
 *   - plain C: pointers, sizes and the POD structs of rt_types.h; no CUDA / torch / C++ types.
 *   - return value: 0 (RT_OK) on success, a negative rt_status otherwise; rt_last_error() returns a
 *     thread-local description of the last failure (the reference throws: FL/Util.h:14-27).
 *   - every device pointer argument is a CUDA device address valid in the context's device.
 *   - all work is stream-ordered on the context's stream (default: a private non-blocking stream;
 *     rt_context_set_stream adopts the caller's, e.g. torch's current stream).  Nothing here
 *     synchronises the host except rt_sync, rt_download, rt_get_ray_counts and rt_get_status.
 *   - a context is thread-compatible, not thread-safe (the reference records on one command list).
 *   - there is NO CPU fallback: without a CUDA device every call fails with RT_ERR_CUDA.
 */
#ifndef RT_CORE_H
#define RT_CORE_H

#include "rt_types.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef enum rt_status {
    RT_OK = 0,
    RT_ERR_INVALID_ARG = -1, /* E_INVALIDARG in the reference */
    RT_ERR_CUDA = -2,        /* a CUDA runtime call failed (device removed / out of memory / no device) */
    RT_ERR_TOO_SMALL = -3,   /* scratch or result buffer smaller than rt_*_prebuild reported */
    RT_ERR_UNSUPPORTED = -4,
    RT_ERR_OVERFLOW = -5     /* traversal stack overflow was detected on the device (see rt_get_status) */
} rt_status;

typedef struct rt_context rt_context;
typedef struct rt_program rt_program;

typedef enum rt_program_kind {
    RT_PROGRAM_PROGRESSIVE = 0, /* assets/shaders/ProgressiveRaytracing.hlsl */
    RT_PROGRAM_REALTIME = 1     /* assets/shaders/RealtimeRaytracing.hlsl */
} rt_program_kind;

/* D3D12_RAYTRACING_ACCELERATION_STRUCTURE_PREBUILD_INFO */
typedef struct rt_prebuild_info {
    uint64_t result_bytes;
    uint64_t scratch_bytes;
    uint64_t update_scratch_bytes;
} rt_prebuild_info;

/* Byte offsets of the intermediate build products inside the scratch buffer of the LAST build of
 * that size; white-box parity tests download them after rt_blas_build / rt_tlas_build. */
typedef struct rt_scratch_layout {
    uint64_t scene_aabb;     /* 6 floats {min xyz, max xyz}                          (FL/SceneAABBCalculator.cpp) */
    uint64_t morton_codes;   /* n x u32, load order                                  (FL/CalculateMortonCodes.hlsli) */
    uint64_t sorted_codes;   /* n x u32                                               (FL/BitonicSort.cpp)           */
    uint64_t sorted_indices; /* n x u32: sorted slot -> load-order primitive          (FL/BitonicSort.cpp)           */
    uint64_t hierarchy;      /* (2n-1) x rt_hierarchy_node                            (FL/BuildBVHSplits.hlsli)
                                NOT produced by bottom-level builds with PREFER_FAST_BUILD and without ALLOW_UPDATE: those emit
                                the hierarchy and fit the boxes in one bottom-up kernel; the child links of the blob's nodes
                                carry the same topology                                                                  */
    uint64_t primitives;     /* BLAS: n x 48-byte load-order records {float v[9]; u32 primitiveIndex, geometryIndex,
                                geometryFlags} = Primitive + PrimitiveMetaData of FL/BottomLevelLoadTriangles.hlsli      */
    uint64_t metadata;       /* same offset as `primitives` (the metadata lives in the same records)                  */
    uint64_t total;
} rt_scratch_layout;

const char *rt_last_error(void);
/* Library version string; also proves the native library (not a fallback) is what got loaded. */
const char *rt_version(void);

/* ---- context: RtContext::create / D3D12CreateRaytracingFallbackDevice (libs/DXRFramework/RtContext.cpp:12-29) */
int rt_context_create(int device_ordinal, rt_context **out);
int rt_context_destroy(rt_context *ctx);
int rt_context_set_stream(rt_context *ctx, void *cuda_stream /* cudaStream_t */);
int rt_sync(rt_context *ctx); /* DeviceResources::WaitForGpu */
int rt_get_status(rt_context *ctx); /* syncs; RT_ERR_OVERFLOW if any traversal overflowed its stack */
/* Number of kernel launches issued through this context since creation (bench.py's gpu_launches). */
uint64_t rt_launch_count(const rt_context *ctx);

/* ---- buffers: CreateBuffer / AllocateUploadBuffer (libs/DXRFramework/Helpers/DirectXRaytracingHelper.h) */
int rt_malloc(rt_context *ctx, uint64_t bytes, void **dev);
int rt_free(rt_context *ctx, void *dev);
int rt_memset(rt_context *ctx, void *dev, int value, uint64_t bytes);
int rt_upload(rt_context *ctx, void *dev, const void *host, uint64_t bytes);   /* async if host is pinned */
int rt_download(rt_context *ctx, void *host, const void *dev, uint64_t bytes); /* synchronises */
int rt_host_alloc_pinned(uint64_t bytes, void **host);
int rt_host_free_pinned(void *host);

/* ---- acceleration structures
 * ID3D12RaytracingFallbackDevice::GetRaytracingAccelerationStructurePrebuildInfo and
 * ID3D12RaytracingFallbackCommandList::BuildRaytracingAccelerationStructure
 * (FL/FallbackLayer.cpp:317-338, FL/GpuBVH2Builder.cpp:137-205,349-455), as called by
 * RtModel::build (libs/DXRFramework/RtModel.cpp:86-118) and RtScene::build (RtScene.cpp:18-52).
 *
 * The result buffer receives the reference's blob ([BVHOffsets][2N-1 AABBNode][N Primitive]
 * [N PrimitiveMetaData], or the TLAS layout) followed, 64-byte aligned, by this library's
 * traversal section (rt_core's own wide nodes; opaque to callers).  A TLAS refers to its BLASes
 * by the device address of their result buffers (rt_instance_desc.blas), the analogue of the
 * Fallback Layer's WRAPPED_GPU_POINTER.  Buffers must stay alive while anything refers to them. */
/* Limits: one acceleration structure holds at most 2^24 - 1 primitives (instances): node and primitive indices are 24 bit
 * in the reference's node format (FL/RayTracingHelper.hlsli:112-118); more is RT_ERR_INVALID_ARG — split the mesh into
 * several BLASes under one TLAS.  Scratch and result buffers must be 64-byte aligned. */
int rt_blas_prebuild(rt_context *ctx, const rt_geometry_desc *geoms, uint32_t n_geoms, uint32_t build_flags,
                     rt_prebuild_info *info);
int rt_blas_build(rt_context *ctx, const rt_geometry_desc *geoms, uint32_t n_geoms, uint32_t build_flags,
                  void *scratch, uint64_t scratch_bytes, void *result, uint64_t result_bytes);
int rt_tlas_prebuild(rt_context *ctx, uint32_t n_instances, uint32_t build_flags, rt_prebuild_info *info);
/* instance_descs: DEVICE array of n rt_instance_desc (ELEMENTS_LAYOUT_ARRAY). */
int rt_tlas_build(rt_context *ctx, const rt_instance_desc *instance_descs, uint32_t n_instances, uint32_t build_flags,
                  void *scratch, uint64_t scratch_bytes, void *result, uint64_t result_bytes);
/* The same builds from D3D12_ELEMENTS_LAYOUT_ARRAY_OF_POINTERS inputs (FL/Util.h:101-114 GetGeometryDesc; FL/TopLevelLoadAABBs.hlsli:38-49,
 * FL/LoadInstancesPass.cpp:55-60; exercised by UT:653, 878-934): `geoms` is a HOST array of host pointers to geometry descriptors;
 * `desc_ptrs` is a DEVICE array of n device addresses, one per instance descriptor. */
int rt_blas_prebuild_ptrs(rt_context *ctx, const rt_geometry_desc *const *geoms, uint32_t n_geoms, uint32_t build_flags,
                          rt_prebuild_info *info);
int rt_blas_build_ptrs(rt_context *ctx, const rt_geometry_desc *const *geoms, uint32_t n_geoms, uint32_t build_flags, void *scratch,
                       uint64_t scratch_bytes, void *result, uint64_t result_bytes);
int rt_tlas_build_ptrs(rt_context *ctx, const rt_instance_desc *const *desc_ptrs, uint32_t n_instances, uint32_t build_flags,
                       void *scratch, uint64_t scratch_bytes, void *result, uint64_t result_bytes);
/* Acceleration-structure updates (D3D12_RAYTRACING_ACCELERATION_STRUCTURE_BUILD_FLAG_ALLOW_UPDATE / PERFORM_UPDATE,
 * FL/GpuBVH2Builder.cpp:152-204, FL/ComputeAABBs.hlsli:38-67,160-164, unit tests UT:1054-1475).
 *   - build_flags | RT_BUILD_FLAG_ALLOW_UPDATE: rt_*_prebuild reports 4n + 4(2n-1) more result bytes and the same
 *     scratch bytes (UT:1085-1086); the build also stores the sort cache (load-order element -> sorted slot) and the
 *     parent of every node.
 *   - build_flags | ALLOW_UPDATE | PERFORM_UPDATE on the SAME result buffer with the same element count and order:
 *     the elements are re-loaded into their cached slots and the boxes re-fitted on the stored topology (no Morton
 *     codes, no sort, no hierarchy pass).  RT_ERR_INVALID_ARG if the buffer does not hold such a build (the
 *     reference does not check).  PERFORM_UPDATE without ALLOW_UPDATE is RT_ERR_INVALID_ARG.
 * rt_update_cache_layout: byte offsets of the two caches inside an ALLOW_UPDATE result buffer (the reference puts
 * them at BVHOffsets.totalSize; here they follow the traversal section). */
int rt_update_cache_layout(uint32_t n_elements, int top_level, uint64_t *sort_cache_offset, uint64_t *parents_offset);

/* ID3D12RaytracingFallbackCommandList::CopyRaytracingAccelerationStructure (FL/GpuBVH2Builder.cpp:330-347,
 * FL/GpuBvh2Copy.hlsl:17-27).  mode: RT_COPY_MODE_CLONE or RT_COPY_MODE_COMPACT (D3D12's values 0 and 1); any other
 * mode is RT_ERR_INVALID_ARG as in the reference.  CLONE copies everything, COMPACT drops the update caches (the copy
 * cannot be updated).  A bottom-level buffer is position independent (offsets only): its bytes can also be moved with
 * rt_download / rt_upload to another device or to disk.  A top-level buffer stores the addresses of its BLASes and
 * stays valid only while they do.  Reads the 144 header bytes back (synchronises) to validate dst_bytes. */
typedef enum rt_copy_mode { RT_COPY_MODE_CLONE = 0, RT_COPY_MODE_COMPACT = 1 } rt_copy_mode;
int rt_as_copy(rt_context *ctx, void *dst, uint64_t dst_bytes, const void *src, int mode);
/* EmitRaytracingAccelerationStructurePostbuildInfo, COMPACTED_SIZE (FL/GpuBVH2Builder.cpp:459-470,
 * FL/GetBVHCompactedSize.hlsl:22-63): dst_sizes[i] (DEVICE, u64) = bytes rt_as_copy(COMPACT) of sources[i] needs;
 * `sources` is a HOST array of n device addresses.  Stream ordered, no host synchronisation. */
int rt_as_emit_postbuild_info(rt_context *ctx, uint64_t *dst_sizes, uint32_t n, const void *const *sources);
typedef struct rt_as_info {
    uint32_t count;      /* triangles or instances */
    uint32_t top_level;  /* 1 for a TLAS */
    uint32_t build_flags;
    uint32_t has_procedural; /* BLAS built from procedural-AABB geometry / TLAS reaching such a BLAS */
    uint64_t blob_bytes;      /* BVHOffsets.totalSize: the reference-format blob at the head of the buffer */
    uint64_t total_bytes;     /* bytes in use = result_bytes of the matching prebuild */
    uint64_t compacted_bytes; /* bytes a COMPACT copy needs */
} rt_as_info;
/* Host-side query of a finished acceleration structure (synchronises). */
int rt_as_get_info(rt_context *ctx, const void *as, rt_as_info *info);
int rt_build_scratch_layout(uint32_t n_elements, int top_level, rt_scratch_layout *layout);
/* Size in bytes of the reference-format blob at the head of a result buffer holding n elements. */
uint64_t rt_blob_bytes(uint32_t n_elements, int top_level);

/* ---- programs and shader-table bindings
 * RtProgram::create / RtState (libs/DXRFramework/RtProgram.h:38-128, RtState.h:18-30) and
 * RtBindings::apply (RtBindings.cpp:100-164).  Shaders are compiled into the library, so a program
 * is chosen by kind; the entry-point names given to RtProgram::Desc are validated on the host side. */
int rt_program_create(rt_context *ctx, rt_program_kind kind, uint32_t hit_group_count, uint32_t miss_count,
                      rt_program **out);
int rt_program_destroy(rt_program *prog);
/* Hit record of (ray_type, instance): VB SRV, IB SRV, 16 dwords MaterialParams
 * (src/ProgressiveRaytracingPipeline.cpp:220-227).  vertex_buffer: rt_vertex[], index_buffer: uint32[]. */
int rt_bindings_set_hit_record(rt_program *prog, uint32_t ray_type, uint32_t instance, const void *vertex_buffer,
                               const void *index_buffer, const rt_material_params *material);
/* Miss record of ray_type: the environment cube (6 x size x size RGBA fp32 device texels), or NULL. */
int rt_bindings_set_miss_record(rt_program *prog, uint32_t ray_type, const float *env_cube_texels, uint32_t size);

/* ---- per-dispatch state: SetComputeRootConstantBufferView / RootDescriptorTable /
 * SetTopLevelAccelerationStructure (src/ProgressiveRaytracingPipeline.cpp:236-242) */
int rt_set_frame_constants(rt_context *ctx, const rt_per_frame_constants *frame);
/* slot 0: gOutput (progressive) / gDirectLightingOutput (realtime); slot 1: gIndirectSpecularOutput.
 * RGBA fp32, pitch in bytes (>= width*16).  The reference's targets are R16G16B16A16_FLOAT
 * (src/DXRExperimentsApp.cpp:28); fp32 is a declared deviation (DESIGN.md). */
int rt_set_output(rt_context *ctx, uint32_t slot, float *rgba, uint64_t pitch_bytes);
/* AOV outputs of the progressive program (new work: the reference has no counterpart; its nearest relative is the
 * DebugOptions switches, assets/shaders/RaytracingHlslCompat.h:64-77, each of which REPLACES the beauty frame with one
 * component).  A bound AOV is accumulated next to gOutput from the same rays, with the same running mean and the same
 * fp16 rounding under half_render_targets, so AOV k equals the beauty output of the same dispatches with debug view k
 * switched on, bit for bit.  AOVs 0-4 hold, for a primary hit:
 *   DIRECT             albedo * direct / pi            (showDirectLightingOnly)
 *   INDIRECT_DIFFUSE   albedo * indirect / pi          (showIndirectDiffuseOnly)
 *   INDIRECT_SPECULAR  reflectivity * spec * fresnel   (showIndirectSpecularOnly)
 *   ALBEDO             albedo                          (showGBufferAlbedoOnly)
 *   FRESNEL            fresnel                         (showFresnelTerm)
 * and for a primary miss the environment times environmentStrength; they are clamped at 0 with alpha 1 like gOutput.
 * NORMAL holds (N, 1) for a hit and (0, 0, 0, 0) for a miss, without the clamp, so its w is the fraction of samples that
 * hit.  N is the normalised interpolated vertex normal exactly as shade() receives it: the OBJECT-space normal, which
 * the reference does not transform by the instance.  POSITION is stored like NORMAL (no clamp, w = coverage) with P the
 * world-space primary hit point o + t*d (HitWorldPosition, o including the RayGen's jitter) in place of N: it is what
 * rt_denoise_temporal reprojects through.  PREVIOUS_POSITION is stored exactly like POSITION with P' in place of P: the
 * same hit point carried into the previous frame's world by the motion of the instance it lies on
 * (rt_set_instance_motion) and, on a deforming mesh, by the motion of its vertices (rt_set_instance_deformation, which
 * adds a term Dw to the P' below).  With M the bound matrix of InstanceIndex() = i, P' = M * (P, 1), each row evaluated as
 * ((m0*Px + m1*Py) + m2*Pz) + m3; P' = P (a copy, no arithmetic) when no motion is bound or i >= n.  No binding
 * therefore gives a PREVIOUS_POSITION equal to POSITION bit for bit, and so does an identity matrix (x*1 and adding +0
 * are exact; the one exception is a coordinate of -0, which comes out +0).  It is what
 * rt_denoise_temporal_motion reprojects through.  Debug views change gOutput only; the AOVs keep these definitions. */
typedef enum rt_aov {
    RT_AOV_DIRECT = 0,
    RT_AOV_INDIRECT_DIFFUSE = 1,
    RT_AOV_INDIRECT_SPECULAR = 2,
    RT_AOV_ALBEDO = 3,
    RT_AOV_FRESNEL = 4,
    RT_AOV_NORMAL = 5,
    RT_AOV_POSITION = 6,
    RT_AOV_PREVIOUS_POSITION = 7,
    RT_AOV_COUNT = 8
} rt_aov;
/* Binds AOV `aov` (an rt_aov id; others are RT_ERR_INVALID_ARG) to a caller-owned RGBA fp32 image; NULL unbinds.  A
 * dispatch checks pitch_bytes >= width*16 for every bound AOV.  A dispatch with any AOV bound is RT_ERR_INVALID_ARG for
 * a realtime program (its outputs already are AOVs) and in the showAmbientOcclusionOnly view (which traces AO rays
 * instead of lighting).  The maxIterations early-out leaves the AOVs untouched, as it leaves gOutput. */
int rt_set_aov_output(rt_context *ctx, uint32_t aov, float *rgba, uint64_t pitch_bytes);
/* Per-instance motion for RT_AOV_PREVIOUS_POSITION (new work: the reference has no counterpart).  world_to_previous_world
 * is a DEVICE array of n row-major 3x4 fp32 matrices; matrix i maps this frame's world space to the previous frame's for
 * the instance with InstanceIndex() == i.  A host computes it as prevObjectToWorld_i * inverse(objectToWorld_i).  It is
 * context state like rt_set_tlas, read by the dispatches that write PREVIOUS_POSITION; the caller keeps the array alive
 * and unchanged until they are done.  NULL with n = 0 unbinds.  RT_ERR_INVALID_ARG: NULL with n > 0 or a pointer with
 * n = 0, a pointer not 16-byte aligned, n > 2^24 - 1.  Only rigid (per-instance) motion is described here; a deforming
 * mesh's moved vertices are described by rt_set_instance_deformation. */
int rt_set_instance_motion(rt_context *ctx, const float *world_to_previous_world, uint32_t n);
/* Per-vertex motion of deforming meshes for RT_AOV_PREVIOUS_POSITION (new work: the reference has no counterpart).
 * descs is a DEVICE array of n rt_deformation_desc (rt_types.h); entry i describes the instance with InstanceIndex() == i:
 *   previous_positions holds last frame's position of every vertex, indexed like the hit record's vertex buffer and in
 *     that buffer's space (xyz = the first 3 floats of each stride_bytes element), NULL for a rigid instance;
 *   object_to_previous_world maps that space into the previous frame's world: prevObjectToWorld_i, times the geometry's
 *     transform3x4 if the BLAS was built with one.  Only its 3x3 is applied.
 * For a primary hit P on primitive prim with barycentrics (bu, bv), record indices i0 i1 i2 and record vertex positions
 * v_k (this frame's vertex buffer: the one the refitted BLAS was built from, as the reference assumes for normals), in
 * fp32 operation by operation:
 *   b0 = (1 - bu) - bv, b1 = bu, b2 = bv                 (interpolate_normal's weights)
 *   d_k = previous_positions[i_k] - v_k                  (per component)
 *   D = (d0*b0 + d1*b1) + d2*b2
 *   Dw_r = (m_r0*D.x + m_r1*D.y) + m_r2*D.z              (r = 0..2, m = object_to_previous_world)
 *   P' = [rt_set_instance_motion's rule: M_i * (P, 1), or P] + Dw
 * That follows from prevO2W * (X + D) = M_i * P + L(prevO2W) * D with M_i = prevO2W * inverse(O2W), so it composes with
 * rigid motion.  Dw is left out (P' is exactly the value above) when nothing is bound, i >= n or previous_positions is
 * NULL.  It is also left out, and rt_get_status reports RT_ERR_INVALID_ARG (as for a missing hit record), when an index
 * is >= vertex_count or stride_bytes is < 12 or not a multiple of 4.  Previous positions equal to the current ones
 * therefore give the AOV without the binding bit for bit, except that a coordinate of -0 may come out +0.  The scope is
 * per-vertex linear motion within each triangle: the hit point moves with the barycentric blend of its vertices'
 * displacements; topology changes (other vertex or index counts) are not described.  Context state like
 * rt_set_instance_motion, read only by dispatches that write PREVIOUS_POSITION; the caller keeps descs and the arrays
 * it points to alive and unchanged until they are done.  NULL with n = 0 unbinds.  RT_ERR_INVALID_ARG: NULL with n > 0
 * or a pointer with n = 0, descs not 16-byte aligned, n > 2^24 - 1. */
int rt_set_instance_deformation(rt_context *ctx, const rt_deformation_desc *descs, uint32_t n);
/* Adaptive sampling of the progressive program (new work: the reference has no counterpart; it accumulates every pixel
 * with the one global accumCount).  counts is a DEVICE array of width x height uint32 in image order (y * width + x):
 * bits 0-30 hold n_p, the samples accumulated into pixel p, and bit 31 (RT_ADAPTIVE_CONVERGED) marks p converged.
 * moments is a DEVICE array of width x height (m1, m2) fp32 pairs: the running means of L and L*L, with
 * L = (r*0.299f + g*0.587f) + b*0.114f of the sample written to gOutput after its clamp at 0 (whatever gOutput shows:
 * the beauty frame, a debug view or the ambient-occlusion view).  moments stays fp32 under half_render_targets (L*L
 * overflows fp16 beyond L = 256).  Context state like rt_set_instance_motion: the caller keeps both arrays alive until
 * the dispatches that use them are done.  NULL, NULL unbinds.  RT_ERR_INVALID_ARG: exactly one of the two NULL, counts
 * not 4-byte or moments not 8-byte aligned, and (at dispatch) a realtime program dispatched while they are bound.
 * While bound, every progressive dispatch (region, interleaved, multi-band, instrumented, debug capture) does this:
 *   a pixel of the launch with bit 31 set is skipped: it traces no ray, is not counted by rt_get_ray_counts, takes no
 *     hit slot, and writes nothing to gOutput, an AOV, counts or moments;
 *   every other pixel is sampled exactly as without the binding, except that every running mean (gOutput, the AOVs and
 *     the moments) uses n_p in place of accumCount: v' = (n_p*v + s) / (n_p + 1); the pixel then stores n_p + 1.
 * accumCount keeps its other two roles: the maxIterations early-out and (on the host) the jitter sequence.  So with
 * counts starting at 0 and no rt_adaptive_update, dispatch k writes exactly what the unbound pipeline writes with
 * accumCount = k, bit for bit, in every output and AOV. */
int rt_set_adaptive_sampling(rt_context *ctx, uint32_t *counts, float *moments);
/* Marks converged pixels: sets bit 31 of counts[p] (never clears it, so the active set only shrinks) when
 *   n_p >= max_samples, or
 *   n_p >= min_samples and e_q <= threshold for every q of p's 3 x 3 window inside the image (Cycles' one-pixel
 *   dilation: an unconverged neighbour keeps p active),
 * with n = counts & 0x7FFFFFFF, sigma_p = sqrtf(fmaxf(0, m2 - m1*m1) / float(n_p - 1)) for n_p >= 2 (+inf below),
 * e_p = sigma_p / (m1 + floor).  A NaN error never passes.  active_count (DEVICE, may be NULL) receives the number of
 * pixels without bit 31 after the update.  At most two operations (a memset and a kernel) on the context's stream, no
 * host synchronisation.  A host may also set or clear bit 31 itself, e.g. to freeze or reopen a region.
 * RT_ERR_INVALID_ARG: a null moments / counts / params, an empty image, counts or active_count not 4-byte or moments not
 * 8-byte aligned, parameters out of range (rt_types.h), or counts / active_count overlapping moments or each other. */
int rt_adaptive_update(rt_context *ctx, const float *moments, uint32_t *counts, uint32_t width, uint32_t height,
                       const rt_adaptive_params *params, uint32_t *active_count);
int rt_set_tlas(rt_context *ctx, const void *tlas_result);
/* Two things that are constants of the reference and options here (defaults = the reference's shaders / this library's
 * declared fp32 deviation):
 *   max_radiance_ray_depth — MAX_RADIANCE_RAY_DEPTH, 1 in assets/shaders/RaytracingCommon.hlsli:11.  2 lets the Phong-lobe
 *     bounce continue one level (BASELINE config 3, "2-bounce"): a secondary hit on a reflective material shoots one more
 *     incoherent closest-hit ray, whose hit is shaded with direct light only (no shadow rays at depth 2:
 *     MAX_SHADOW_RAY_DEPTH 2; no indirect diffuse below depth 0: ProgressiveRaytracing.hlsl:107).  Parity with the
 *     reference is pinned at 1; at 2 the CPU oracle follows the same shader source with the constant changed.
 *   half_render_targets — 1: every value stored to an output (accumulation, AOVs, both denoiser passes) is rounded to fp16
 *     and back, which is what the reference's R16G16B16A16_FLOAT targets hold (src/DXRExperimentsApp.cpp:28, :121); the
 *     buffers stay RGBA fp32.  0 (default): full fp32, needed for multi-GPU sums and long accumulations. */
typedef struct rt_render_options {
    uint32_t max_radiance_ray_depth; /* 1 or 2 */
    uint32_t half_render_targets;    /* 0 or 1 */
} rt_render_options;
int rt_set_render_options(rt_context *ctx, const rt_render_options *options);

/* RtContext::raytrace -> DispatchRays (libs/DXRFramework/RtContext.cpp:192-222,
 * FL/UberShaderRayTracingProgram.cpp:213-272).  `depth` is accepted and ignored, as in the reference. */
int rt_dispatch_rays(rt_context *ctx, rt_program *prog, uint32_t width, uint32_t height, uint32_t depth);
/* Same, restricted to the pixel rectangle [x0,x1) x [y0,y1) of the width x height launch: screen-tile
 * sharding across GPUs (SURVEY.md 8e).  Pixels outside the rectangle are not touched. */
int rt_dispatch_rays_region(rt_context *ctx, rt_program *prog, uint32_t width, uint32_t height, uint32_t x0,
                            uint32_t y0, uint32_t x1, uint32_t y1);
/* Same, restricted to every `groups`-th horizontal strip of `strip_rows` image rows (a power of two >= 4), starting
 * with strip `group`: screen-tile sharding of one frame across GPUs with a balanced load (SURVEY.md 8e ii; the
 * reference is single-GPU, libs/DXRFramework/RtContext.cpp:23).  One dispatch covers all of the group's strips, so
 * the kernels stay as large as a contiguous region of the same area.  Pixels of other groups are not touched. */
int rt_dispatch_rays_interleaved(rt_context *ctx, rt_program *prog, uint32_t width, uint32_t height, uint32_t strip_rows,
                                 uint32_t groups, uint32_t group);
/* Rays traced by all dispatches since the last reset (synchronises). */
int rt_get_ray_counts(rt_context *ctx, rt_ray_counts *counts, int reset);
/* Instrumented traversal: while enabled, dispatches run trace kernels that count node visits and triangle tests
 * per stage (primary / incoherent secondary / shadow).  These counts are the n_int and n_leaf of the roofline's
 * algorithmic bytes per ray (SURVEY.md 8d); instrumented passes are never the ones that are timed. */
int rt_enable_trace_stats(rt_context *ctx, int enable);
int rt_get_trace_stats(rt_context *ctx, rt_trace_stats *primary, rt_trace_stats *secondary, rt_trace_stats *shadow, int reset);
/* Optional per-stage device timing (CUDA events around the trace kernels; synchronises the host once per
 * dispatch while enabled, so it is for profiling runs, not for the headline measurement).  Times are
 * accumulated milliseconds: primary closest-hit, incoherent secondary closest-hit, shadow any-hit. */
int rt_enable_stage_timing(rt_context *ctx, int enable);
int rt_get_stage_timing(rt_context *ctx, double *primary_ms, double *secondary_ms, double *shadow_ms, int reset);

/* Parity instrumentation (test infrastructure of the boundary, never on a timed path): while capture is enabled a
 * dispatch runs as ONE pixel band (the same kernels, bit-identical results) and its stage products stay readable:
 * the camera rays' hits written by the ray-generation kernel (the north star's "primary-ray hit triangle IDs"),
 * the compacted secondary / shadow ray queues and what the queue traversal kernels answered.  Queues are planar:
 * `plane` selects the ray kind (secondary: 0 indirect diffuse, 1 Phong lobe; shadow: 0 directional, 1 point light,
 * 2-3 ambient-occlusion debug view).  There is no reference counterpart (the Fallback Layer keeps this state in
 * registers of its uber shader, FL/TraverseShader.hlsli:21-73); the oracle re-traces the downloaded rays. */
typedef enum rt_debug_array {
    RT_DEBUG_PRIMARY_HITS = 0,       /* pixels x {float t, u, v; uint32 PrimitiveIndex (0xFFFFFFFF = miss)}, pixel order of the dispatch;
                                        under adaptive sampling a skipped (converged) pixel traces nothing and its entry here and
                                        in RT_DEBUG_PRIMARY_RECORDS keeps whatever an earlier dispatch left */
    RT_DEBUG_PRIMARY_RECORDS = 1,    /* pixels x uint32 hit-group record index (InstanceContribution + ray type) */
    RT_DEBUG_SLOT_INFO = 2,          /* hit_slots x {uint32 pixel, record, flags, 0} */
    RT_DEBUG_SECONDARY_RAYS = 3,     /* hit_slots x rt_ray per plane; tmax < 0 marks an inactive slot */
    RT_DEBUG_SECONDARY_HITS = 4,     /* hit_slots x {t, u, v, PrimitiveIndex} per plane */
    RT_DEBUG_SECONDARY_RECORDS = 5,  /* hit_slots x uint32 per plane */
    RT_DEBUG_SHADOW0_RAYS = 6,       /* hit_slots x rt_ray per plane (depth-0 shadow rays) */
    RT_DEBUG_SHADOW0_VISIBILITY = 7, /* hit_slots x uint8 per plane: 1 = unoccluded */
    RT_DEBUG_SHADOW1_RAYS = 8,       /* shadow1_pairs x rt_ray per plane (shadow rays of the secondary hits) */
    RT_DEBUG_SHADOW1_VISIBILITY = 9  /* shadow1_pairs x uint8 per plane */
} rt_debug_array;
int rt_enable_debug_capture(rt_context *ctx, int enable);
int rt_debug_counts(rt_context *ctx, uint32_t *pixels, uint32_t *hit_slots, uint32_t *shadow1_pairs); /* synchronises */
int rt_debug_download(rt_context *ctx, int array, uint32_t plane, void *host, uint64_t host_bytes);   /* synchronises */

/* DenoiseCompositor::dispatch (src/DenoiseCompositor.cpp:109-148): pass H (joint = direct, input =
 * indirect specular -> tmp) then pass V (-> out, + direct, exposure, Reinhard, gamma).  RGBA fp32, tightly packed. */
int rt_denoise(rt_context *ctx, const float *direct, const float *indirect_specular, float *tmp, float *out,
               uint32_t width, uint32_t height, const rt_denoiser_params *params);
/* Denoiser for the accumulated frame of the progressive program (new work: the reference has no counterpart; its nearest
 * relative is DenoiseCompositor::dispatch, which filters indirect specular only).  Spatial SVGF without its temporal part
 * (Schied et al. 2017): an edge-avoiding a-trous wavelet filter (Dammertz et al. 2010) guided by the AOVs.  Inputs are
 * RGBA fp32 images, tightly packed, width x height: beauty = gOutput, albedo = RT_AOV_ALBEDO, normal = RT_AOV_NORMAL
 * (N = .xyz, coverage c = .w).  Per pixel p, with L = (r*0.299f + g*0.587f) + b*0.114f:
 *   wN(p,q) = max(0, (Np.x*Nq.x + Np.y*Nq.y) + Np.z*Nq.z), squared normal_exponent_log2 times.  For the centre tap q = p
 *     every edge-stopping factor is 1.  Taps outside the image or with weight 0 contribute nothing.
 *   A pixel with c == 0 (sky) is copied unchanged; its N = 0 gives wN = 0, so it never contributes to a neighbour.
 *   var0 = max(0, m2 - m1*m1), m1 / m2 the wN-weighted means of L / L*L over the 7 x 7 window.
 *   Iteration i = 0 .. iterations-1, step s = 2^i, kernel b = (1/16, 1/4, 3/8, 1/4, 1/16) over the 5 x 5 taps
 *   q = p + s*(dx, dy), summed dy outer, dx inner:
 *     g(p) = sum (h(dy)*h(dx))*wN * var / sum (h(dy)*h(dx))*wN over the 3 x 3 neighbours, h = (1/4, 1/2, 1/4);
 *     w = ((b(dx)*b(dy))*wN) * expf(-(|Lp-Lq|*invL + |dA|_1*invA)), |dA|_1 = (|dr| + |dg|) + |db| of the albedo;
 *     invL = 1/(sigma_luminance*sqrtf(g(p)) + 1e-10f), invA = 1/sigma_albedo or 0 when sigma_albedo = 0;
 *     C' = sum w*C / sum w, var' = sum (w*w)*var / (sum w)^2; L is recomputed from C every iteration.
 *   out = (C, 1) after the last iteration; under half_render_targets the store rounds through fp16 (intermediates fp32).
 * tmp holds 2 * width * height RGBA fp32 (C, var) ping-pong images.  1 + iterations launches on the context's stream, no
 * host synchronisation.  RT_ERR_INVALID_ARG: a null pointer, a buffer not 16-byte aligned, an empty image, parameters out
 * of range, or out / tmp overlapping an input or each other.  The inputs are only read. */
int rt_denoise_progressive(rt_context *ctx, const float *beauty, const float *albedo, const float *normal,
                           float *tmp /* 2 * width * height RGBA fp32 */, float *out,
                           uint32_t width, uint32_t height, const rt_progressive_denoise_params *params);
/* The same filter with SVGF's temporal pass in front of it (Schied et al. 2017), for frames of one sample each
 * (accumulation off) from a moving camera.  Inputs as rt_denoise_progressive plus position = RT_AOV_POSITION (P = .xyz);
 * prev_camera (host memory) is the camera of the previous frame, as rt_set_frame_constants received it.  A history image
 * is 4 planes of width x height RGBA fp32: 0 = (integrated C.rgb, history length n), 1 = (m1, m2, 0, 0) the integrated
 * luminance moments, 2 = this frame's normal AOV, 3 = this frame's position AOV.  The call reads prev_history and writes
 * history; the caller swaps them every frame.  prev_camera and prev_history are both NULL for a first frame (or after a
 * reset).  Per pixel p, with L, wN and the window as above and c the coverage of the normal AOV:
 *   Reproject (only if c == 1 and prev_history != NULL): o' = prev eye + (jitters[0]*30, jitters[1]*30, 0), the origin of
 *     the progressive primary ray; r = Pp - o'; zc = dot(r, W')/dot(W', W'), no history if !(zc > 0);
 *     sx = (dot(r, U')/dot(U', U'))/zc, sy = -((dot(r, V')/dot(V', V'))/zc) (the inverse of the primary ray: U', V', W'
 *     are orthogonal); fx = ((sx + 1)*0.5)*width - 0.5, fy likewise; dot(a, b) = (a.x*b.x + a.y*b.y) + a.z*b.z.
 *   Bilinear fetch: x0 = floor(fx), y0 = floor(fy), ax = fx - x0, ay = fy - y0; taps (x0, y0), (x0+1, y0), (x0, y0+1),
 *     (x0+1, y0+1) in that order with weights (1-ax)*(1-ay), ax*(1-ay), (1-ax)*ay, ax*ay.  A tap is dropped when it lies
 *     outside the image, its weight is 0, its coverage (plane 2 .w) is not 1, dot(Nq, Np) < normal_cos, or
 *     |Pq - Pp| > position_tolerance*|Pp - o'| (|v| = sqrtf(dot(v, v))).  C_h, n_h, m1_h, m2_h are the weighted sums over
 *     the remaining taps divided by the sum of their weights; with none left (or no fx, fy inside (-1, width) x
 *     (-1, height)) they are 0.
 *   Blend: n = min(n_h + 1, 32); a = max(1/n, alpha_color), am = max(1/n, alpha_moments); C = (1 - a)*C_h + a*C_cur;
 *     m1 = (1 - am)*m1_h + am*L(C_cur), m2 = (1 - am)*m2_h + am*(L*L).
 *   Variance: var0 = max(0, m2 - m1*m1) if n >= 4, else the 7 x 7 window estimate over the integrated C.
 *   Then the a-trous iterations of rt_denoise_progressive run unchanged on (C, var0) and write out.
 * Without history every pixel has n = 1 and C = C_cur, so out equals rt_denoise_progressive's bit for bit.  The history
 * is fp32 always; only out is rounded through fp16 under half_render_targets.  tmp holds 2 * width * height RGBA fp32.
 * 2 + iterations launches on the context's stream, no host synchronisation.  RT_ERR_INVALID_ARG: a null pointer (other
 * than the prev_camera / prev_history pair), exactly one of that pair NULL, a buffer not 16-byte aligned, an empty image,
 * parameters out of range, or history / tmp / out overlapping an input, prev_history or each other.  The inputs and
 * prev_history are only read. */
int rt_denoise_temporal(rt_context *ctx, const float *beauty, const float *albedo, const float *normal, const float *position,
                        const rt_camera_params *prev_camera, const float *prev_history,
                        float *history /* 4 * width * height RGBA fp32 */, float *tmp /* 2 * width * height RGBA fp32 */,
                        float *out, uint32_t width, uint32_t height, const rt_temporal_denoise_params *params);
/* rt_denoise_temporal for scenes whose instances move between frames.  previous_position = RT_AOV_PREVIOUS_POSITION
 * (Q = .xyz: where this frame's primary hit point was in the previous frame's world, rt_set_instance_motion and
 * rt_set_instance_deformation).  Q takes
 * the place of Pp in exactly two places of the rule above:
 *   the reprojection: r = Q - o';
 *   the position test: a tap is dropped when |Pq - Q| > position_tolerance*|Q - o'|.
 * Everything else is unchanged: the normal test compares this frame's normal AOV with the history's (the normal AOV is
 * object-space, so a rigid instance motion leaves it unchanged), and history plane 3 stores this frame's P, which the
 * next frame's Pq is.  previous_position == position therefore gives rt_denoise_temporal's out and history bit for bit.
 * A deforming mesh (a BLAS refit with moved vertices) keeps its history when its previous positions are bound with
 * rt_set_instance_deformation; the normal test still sees its changed normals.  previous_position is required; its alignment and overlap rules are those of the other inputs,
 * and it is only read.  Launches and RT_ERR_INVALID_ARG cases otherwise as rt_denoise_temporal. */
int rt_denoise_temporal_motion(rt_context *ctx, const float *beauty, const float *albedo, const float *normal,
                               const float *position, const float *previous_position, const rt_camera_params *prev_camera,
                               const float *prev_history, float *history /* 4 * width * height RGBA fp32 */,
                               float *tmp /* 2 * width * height RGBA fp32 */, float *out, uint32_t width, uint32_t height,
                               const rt_temporal_denoise_params *params);

/* ---- wavefront primitives exposed for parity tests and benchmarks */
/* Fallback_TraceRay without shader call-outs (FL/TraverseShader.hlsli:21-73): n rays -> n hits. */
int rt_trace_rays(rt_context *ctx, const void *tlas_result, const rt_ray *rays, uint64_t n, uint32_t ray_flags,
                  uint32_t instance_mask, rt_hit *hits);
/* Same with per-ray work counters accumulated into *stats (device memory, 5 x u64 = rt_trace_stats). */
int rt_trace_rays_stats(rt_context *ctx, const void *tlas_result, const rt_ray *rays, uint64_t n, uint32_t ray_flags,
                        uint32_t instance_mask, rt_hit *hits, rt_trace_stats *stats_dev);
/*
 * Fallback_TraceRay WITH the hit groups' any-hit and intersection programs, over triangle and procedural-AABB geometry
 * (replaces: the Traverse loop's shader call-outs FL/TraverseFunction.hlsli:651-722 — InvokeAnyHit :102-117,
 * Fallback_ReportHit :136-158 — and the hit-group lookup GetAnyHitAndIntersectionStateId; on the host side
 * RtProgram::Desc::addHitGroup(idx, closestHit, anyHit, intersection), libs/DXRFramework/RtProgram.h:51).
 * `programs` is a HOST array with one entry per hit-group record, indexed by
 * ray_contribution + GeometryContributionToHitGroupIndex * geometry_multiplier + InstanceContributionToHitGroupIndex;
 * records beyond n_programs have no any-hit and no intersection program.  hits[i].leaf_slot carries HitKind() in bits
 * 31:24 (0xFE for triangles); for a procedural hit bary[] holds the intersection program's two attribute floats.
 * rt_dispatch_rays / rt_trace_rays know hit groups of type TRIANGLES only: given a TLAS that reaches procedural
 * primitives they report every ray as a miss and rt_get_status returns RT_ERR_UNSUPPORTED.
 */
int rt_trace_rays_hit_groups(rt_context *ctx, const void *tlas_result, const rt_ray *rays, uint64_t n, uint32_t ray_flags,
                             uint32_t instance_mask, uint32_t ray_contribution, uint32_t geometry_multiplier,
                             const rt_hit_group_programs *programs, uint32_t n_programs, rt_hit *hits);
/* RayGen's camera rays (ProgressiveRaytracing.hlsl:17-31) written out as records. */
int rt_generate_primary_rays(rt_context *ctx, const rt_per_frame_constants *frame, uint32_t width, uint32_t height,
                             float jitter_scale, rt_ray *rays);
/* buf[i] *= scale  (i < count floats): turns a rank's running mean into its share of the global mean
 * before the NCCL sum of the accumulation buffers (SURVEY.md 8e). */
int rt_scale_buffer(rt_context *ctx, float *buf, uint64_t count, float scale);


/* ---- multi-GPU accumulation (SURVEY.md 8e): one process per GPU, replicated acceleration structures, the frame split
 * by sample index (frameCount = global sample index) and / or by screen strips (rt_dispatch_rays_interleaved), and ONE
 * NCCL reduce per output frame.  New work of this library: the reference has no multi-GPU path (NodeMask is always 0,
 * libs/DXRFramework/RtContext.cpp:23, FL/GpuBVH2Builder.cpp:17).  libnccl.so.2 is bound at run time on first use
 * (RT_NCCL_LIB overrides the name); without it these calls return RT_ERR_UNSUPPORTED and everything else works.
 *   rank 0: rt_comm_get_unique_id -> hand the 128 bytes to every rank over any side channel (file, MPI, a
 *   torch.distributed broadcast) -> all ranks: rt_comm_create (collective) -> per frame: rt_accum_reduce. */
#define RT_COMM_ID_BYTES 128
typedef struct rt_comm rt_comm;
int rt_comm_get_unique_id(uint8_t *id /* RT_COMM_ID_BYTES */);
int rt_comm_create(rt_context *ctx, const uint8_t *id, int world_size, int rank, rt_comm **out);
int rt_comm_destroy(rt_comm *comm);
int rt_comm_info(const rt_comm *comm, int *world_size, int *rank, int *nccl_version);
/* recv[i] = sum over ranks r of weight_r * send_r[i], i < count floats, on rank `root` (root = -1: on every rank).
 * `weight` is this rank's share of the frame's samples (its spp / total spp for running-mean accumulation buffers,
 * 1 for sums); it is applied inside the reduction, not by a separate pass.  Stream-ordered on the context's stream;
 * recv may equal send (in place) and is ignored on non-root ranks.  Strip-sharded ranks pass full-frame buffers that
 * are zero outside their strips. */
int rt_accum_reduce(rt_context *ctx, rt_comm *comm, const float *send, float *recv, uint64_t count, float weight, int root);

#ifdef __cplusplus
}
#endif
#endif /* RT_CORE_H */
