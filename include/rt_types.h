/*
 * rt_types.h — plain-C data types shared by every layer of the B200 ray-tracing core.
 *
 * These are the byte-compatible restatements of the structs the reference passes across
 * its host/shader boundary, so that a maintainer can hand the reference's own structs to the
 * C ABI in rt_core.h unchanged:
 *
 *   rt_per_frame_constants  == PerFrameConstants   (assets/shaders/RaytracingHlslCompat.h:79-85, 188 B)
 *   rt_material_params      == MaterialParams      (assets/shaders/RaytracingHlslCompat.h:87-96,  64 B)
 *   rt_denoiser_params      == DenoiserParams      (include/DenoiseCompositor.h:41-49,             24 B)
 *   rt_instance_desc        == D3D12_RAYTRACING_FALLBACK_INSTANCE_DESC
 *                              (externals/D3D12RaytracingFallback/src/RayTracingHlslCompat.h:236-242, 64 B)
 *   rt_geometry_desc        ~= D3D12_RAYTRACING_GEOMETRY_DESC (triangles only), the arguments
 *                              libs/DXRFramework/RtModel.cpp:95-101 passes to AddVertexBuffer
 *   rt_aabb_node / rt_bvh_offsets / rt_primitive / rt_primitive_meta / rt_bvh_metadata
 *                           == AABBNode / BVHOffsets / Primitive / PrimitiveMetaData / BVHMetadata
 *                              (externals/D3D12RaytracingFallback/src/RayTracingHlslCompat.h:142-255,368-421)
 *
 * No CUDA, torch or C++ types appear here; the header compiles as C99 and C++11.
 */
#ifndef RT_TYPES_H
#define RT_TYPES_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ frame constants */

typedef struct rt_camera_params {
    float worldEyePos[4];
    float U[4];
    float V[4];
    float W[4];
    float jitters[2];
    uint32_t frameCount;
    uint32_t accumCount;
} rt_camera_params; /* 80 B */

typedef struct rt_directional_light {
    float forwardDir[4];
    float color[4]; /* rgb * a */
} rt_directional_light; /* 32 B */

typedef struct rt_point_light {
    float worldPos[4];
    float color[4];
} rt_point_light; /* 32 B */

typedef struct rt_debug_options {
    uint32_t maxIterations;
    uint32_t cosineHemisphereSampling;
    uint32_t showIndirectDiffuseOnly;
    uint32_t showIndirectSpecularOnly;
    uint32_t showAmbientOcclusionOnly;
    uint32_t showGBufferAlbedoOnly;
    uint32_t showDirectLightingOnly;
    uint32_t showFresnelTerm;
    uint32_t noIndirectDiffuse;
    float environmentStrength;
    uint32_t debug;
} rt_debug_options; /* 44 B */

typedef struct rt_per_frame_constants {
    rt_camera_params cameraParams;
    rt_directional_light directionalLight;
    rt_point_light pointLight;
    rt_debug_options options;
} rt_per_frame_constants; /* 188 B */

typedef struct rt_material_params {
    float albedo[4];
    float specular[4];
    float emissive[4];
    float reflectivity;
    float roughness;
    float IoR;
    uint32_t type; /* 0 diffuse, 1 glossy, 2 specular */
} rt_material_params; /* 64 B */

typedef struct rt_denoiser_params {
    float exposure;
    float gamma;
    uint32_t tonemap;
    uint32_t gammaCorrect;
    int32_t maxKernelSize;
    uint32_t debugVisualize; /* 0 composite, 1 denoised, 2 input, 3 joint */
} rt_denoiser_params; /* 24 B */

/* rt_denoise_progressive (rt_core.h); new work, no reference counterpart. */
typedef struct rt_progressive_denoise_params {
    uint32_t iterations;           /* 0..5: a-trous steps 1, 2, 4, 8, 16 */
    uint32_t normal_exponent_log2; /* 0..8: the normal weight is max(0, Np.Nq)^(2^this) */
    float sigma_luminance;         /* > 0 */
    float sigma_albedo;            /* >= 0, 0 = no albedo term */
} rt_progressive_denoise_params; /* 16 B */
/* Defaults, chosen on the CPU restatement of the filter (DESIGN.md 4.4). */
#define RT_PROGRESSIVE_DENOISE_DEFAULTS {5u, 7u, 4.0f, 0.1f}

/* rt_denoise_temporal (rt_core.h); new work, no reference counterpart. */
typedef struct rt_temporal_denoise_params {
    rt_progressive_denoise_params spatial; /* the a-trous stage, exactly as rt_denoise_progressive */
    float alpha_color;                     /* (0, 1]: floor of the current frame's blend weight (SVGF: 0.2) */
    float alpha_moments;                   /* (0, 1]: the same for the luminance moments (SVGF: 0.2) */
    float normal_cos;                      /* [-1, 1]: a history tap is rejected when dot(Nq, Np) < this */
    float position_tolerance;              /* >= 0: ... or when |Pq - Pp| > this * |Pp - o_prev| */
} rt_temporal_denoise_params; /* 32 B */
/* Defaults, chosen on the CPU restatement of the filter (DESIGN.md 4.4.2). */
#define RT_TEMPORAL_DENOISE_DEFAULTS {RT_PROGRESSIVE_DENOISE_DEFAULTS, 0.2f, 0.2f, 0.9f, 0.02f}

/* rt_adaptive_update (rt_core.h); new work, no reference counterpart. */
typedef struct rt_adaptive_params {
    float threshold;      /* >= 0, finite: a pixel may converge once its relative standard error is at most this */
    float floor;          /* > 0, finite: added to the mean luminance in the relative error's denominator */
    uint32_t min_samples; /* >= 1: no pixel converges on its error with fewer samples */
    uint32_t max_samples; /* min_samples .. 2^31 - 1: every pixel converges at this many samples */
} rt_adaptive_params; /* 16 B */
/* Defaults, chosen on the CPU restatement of the rule (DESIGN.md 4.6). */
#define RT_ADAPTIVE_DEFAULTS {0.1f, 0.1f, 8u, 1024u}
/* Bit 31 of a sample count: the pixel has converged and dispatches skip it. */
#define RT_ADAPTIVE_CONVERGED 0x80000000u

/* rt_set_instance_deformation (rt_core.h); new work, no reference counterpart.  One per InstanceIndex(). */
typedef struct rt_deformation_desc {
    const float *previous_positions;   /* DEVICE; NULL = the instance is rigid */
    uint32_t stride_bytes;             /* >= 12, a multiple of 4: xyz are the first 3 floats of an element */
    uint32_t vertex_count;             /* elements of previous_positions */
    float object_to_previous_world[12]; /* row-major 3x4; only its 3x3 is applied */
} rt_deformation_desc; /* 64 B, 16-byte aligned in an array */

/* Interleaved vertex the hit shaders read: libs/DXRFramework/RtModel.cpp:13-17 (stride 24). */
typedef struct rt_vertex {
    float position[3];
    float normal[3];
} rt_vertex;

/* ------------------------------------------------------------------ acceleration structure inputs */

/* D3D12_RAYTRACING_GEOMETRY_TYPE (FL/LoadPrimitivesPass.cpp:73,124-127). */
enum {
    RT_GEOMETRY_TYPE_TRIANGLES = 0,
    RT_GEOMETRY_TYPE_PROCEDURAL_AABBS = 1
};

enum {
    RT_GEOMETRY_FLAG_NONE = 0,
    RT_GEOMETRY_FLAG_OPAQUE = 0x1,
    RT_GEOMETRY_FLAG_NO_DUPLICATE_ANYHIT = 0x2
};

enum {
    RT_INSTANCE_FLAG_NONE = 0,
    RT_INSTANCE_FLAG_TRIANGLE_CULL_DISABLE = 0x1,
    RT_INSTANCE_FLAG_TRIANGLE_FRONT_COUNTERCLOCKWISE = 0x2,
    RT_INSTANCE_FLAG_FORCE_OPAQUE = 0x4,
    RT_INSTANCE_FLAG_FORCE_NON_OPAQUE = 0x8
};

enum {
    RT_RAY_FLAG_NONE = 0x00,
    RT_RAY_FLAG_FORCE_OPAQUE = 0x01,
    RT_RAY_FLAG_FORCE_NON_OPAQUE = 0x02,
    RT_RAY_FLAG_ACCEPT_FIRST_HIT_AND_END_SEARCH = 0x04,
    RT_RAY_FLAG_SKIP_CLOSEST_HIT_SHADER = 0x08,
    RT_RAY_FLAG_CULL_BACK_FACING_TRIANGLES = 0x10,
    RT_RAY_FLAG_CULL_FRONT_FACING_TRIANGLES = 0x20,
    RT_RAY_FLAG_CULL_OPAQUE = 0x40,
    RT_RAY_FLAG_CULL_NON_OPAQUE = 0x80
};

enum {
    RT_BUILD_FLAG_NONE = 0,
    RT_BUILD_FLAG_ALLOW_UPDATE = 0x1,
    RT_BUILD_FLAG_ALLOW_COMPACTION = 0x2,
    RT_BUILD_FLAG_PREFER_FAST_TRACE = 0x4,
    RT_BUILD_FLAG_PREFER_FAST_BUILD = 0x8,
    RT_BUILD_FLAG_MINIMIZE_MEMORY = 0x10,
    RT_BUILD_FLAG_PERFORM_UPDATE = 0x20
};

/*
 * One geometry of a bottom-level build.  `vertex_buffer`/`index_buffer`/`transform3x4`
 * are DEVICE pointers for rt_core (HOST pointers for the CPU oracle, which reuses the struct).
 * index_format: 0 = no index buffer, 16 = uint16, 32 = uint32.
 * (externals/D3D12RaytracingFallback/src/LoadPrimitivesPass.cpp:60-115)
 * type == RT_GEOMETRY_TYPE_PROCEDURAL_AABBS (D3D12_RAYTRACING_GEOMETRY_AABBS_DESC, LoadPrimitivesPass.cpp:122-152,
 * FL/LoadProceduralGeometry.hlsl): `vertex_buffer` is the AABB buffer ({float min[3], max[3]} at the start of every
 * `vertex_stride_bytes`), `vertex_count` is AABBCount; index buffer and transform are ignored.
 */
typedef struct rt_geometry_desc {
    const void *vertex_buffer;
    uint32_t vertex_count;
    uint32_t vertex_stride_bytes;
    const void *index_buffer;
    uint32_t index_count;
    uint32_t index_format;
    const float *transform3x4; /* 12 floats, row major, or NULL */
    uint32_t flags;            /* RT_GEOMETRY_FLAG_* */
    uint32_t type;             /* RT_GEOMETRY_TYPE_* (0 = triangles, so zero-initialised descs keep their meaning) */
} rt_geometry_desc;

/* 64 B, byte-compatible with D3D12_RAYTRACING_FALLBACK_INSTANCE_DESC. */
typedef struct rt_instance_desc {
    float transform[12];            /* object -> world, 3x4 row major */
    uint32_t instance_id_and_mask;  /* id : 24 | mask : 8 (mask in the high byte) */
    uint32_t hit_group_and_flags;   /* InstanceContributionToHitGroupIndex : 24 | flags : 8 */
    uint64_t blas;                  /* device address of a built BLAS blob (oracle: host address) */
} rt_instance_desc;

#define RT_INSTANCE_ID(d) ((d).instance_id_and_mask & 0xFFFFFFu)
#define RT_INSTANCE_MASK(d) ((d).instance_id_and_mask >> 24)
#define RT_INSTANCE_HIT_GROUP(d) ((d).hit_group_and_flags & 0xFFFFFFu)
#define RT_INSTANCE_FLAGS(d) ((d).hit_group_and_flags >> 24)

/* ------------------------------------------------------------------ acceleration structure blob */

typedef struct rt_bvh_offsets {
    uint32_t offsetToBoxes;
    uint32_t offsetToVertices;          /* TLAS: offsetToLeafNodeMetaData */
    uint32_t offsetToPrimitiveMetaData; /* TLAS: unused (0) */
    uint32_t totalSize;
} rt_bvh_offsets; /* 16 B */

typedef struct rt_aabb_node {
    float center[3];
    uint32_t flags; /* internal: left index (24 bit); leaf: slot | 0x80000000 */
    float halfDim[3];
    uint32_t right; /* internal: right index; leaf: number of triangles (1) */
} rt_aabb_node; /* 32 B */

#define RT_NODE_LEAF_FLAG 0x80000000u
#define RT_NODE_PROCEDURAL_FLAG 0x40000000u

#pragma pack(push, 1)
#define RT_PRIMITIVE_TYPE_TRIANGLE 1u   /* TRIANGLE_TYPE, FL/RayTracingHlslCompat.h:140 */
#define RT_PRIMITIVE_TYPE_PROCEDURAL 2u /* PROCEDURAL_PRIMITIVE_TYPE, :141 */
typedef struct rt_primitive {
    uint32_t type; /* 1 = triangle (v = 3 vertices), 2 = procedural (v[0..5] = AABB min, max; v[6..8] = 0) */
    float v[9];
} rt_primitive; /* 40 B */

typedef struct rt_primitive_meta {
    uint32_t geometryContributionToHitGroupIndex;
    uint32_t primitiveIndex;
    uint32_t geometryFlags;
} rt_primitive_meta; /* 12 B */

typedef struct rt_bvh_metadata {
    rt_instance_desc instanceDesc; /* transform replaced by world -> object */
    float objectToWorld[12];
    uint32_t instanceIndex;
} rt_bvh_metadata; /* 116 B */
#pragma pack(pop)

typedef struct rt_hierarchy_node {
    uint32_t parent;
    uint32_t left;
    uint32_t right;
} rt_hierarchy_node; /* 12 B */

/* ------------------------------------------------------------------ rays and hits (wavefront records) */

typedef struct rt_ray {
    float origin[3];
    float tmin;
    float direction[3];
    float tmax;
} rt_ray; /* 32 B */

#define RT_NO_HIT 0xFFFFFFFFu

typedef struct rt_hit {
    float t;
    float bary[2];
    uint32_t primitive_index; /* PrimitiveIndex(): index within its geometry, pre-sort; RT_NO_HIT on miss */
    uint32_t instance_index;  /* InstanceIndex() */
    uint32_t geometry_index;  /* GeometryContributionToHitGroupIndex */
    uint32_t instance_id;     /* InstanceID() */
    uint32_t leaf_slot;       /* sorted triangle slot inside the BLAS (debug / parity) */
} rt_hit; /* 32 B */

/*
 * Hit groups with any-hit / intersection shaders (RtProgram::Desc::addHitGroup(idx, chs, ahs, is), RtProgram.h:51).
 * The reference links DXIL entry points; here the "shader library" is CUDA code compiled into librt_core, and a hit
 * group names its programs by id.  One entry per hit-group record, indexed exactly as the shader table is
 * (RayContributionToHitGroupIndex + GeometryContributionToHitGroupIndex * Multiplier + InstanceContribution...,
 * FL/TraverseFunction.hlsli:658-661,684-687).
 */
enum {
    RT_ANYHIT_NONE = 0,       /* no any-hit shader in the hit group (state id 0): the hit is accepted */
    RT_ANYHIT_ACCEPT = 1,     /* a no-op shader, e.g. the application's ShadowAnyHit (ProgressiveRaytracing.hlsl:172-176) */
    RT_ANYHIT_IGNORE = 2,     /* IgnoreHit() on every candidate */
    RT_ANYHIT_END_SEARCH = 3, /* AcceptHitAndEndSearch() on every candidate */
    RT_ANYHIT_CUTOUT = 4,     /* alpha-test stand-in: IgnoreHit() when (int(8*attr.x) + int(8*attr.y)) is odd */
    RT_ANYHIT_COUNT = 5
};
enum {
    RT_INTERSECTION_NONE = 0,   /* hit group of type TRIANGLES */
    RT_INTERSECTION_BOX = 1,    /* the primitive's AABB itself: ReportHit(entry t, or exit t when the origin is inside) */
    RT_INTERSECTION_SPHERE = 2, /* sphere inscribed in the AABB (centre = box centre, radius = smallest half extent) */
    RT_INTERSECTION_COUNT = 3
};
#define RT_HIT_KIND_TRIANGLE_FRONT_FACE 0xFEu /* the only triangle hit kind the reference reports (:688) */
#define RT_HIT_KIND_BOX_ENTER 0u
#define RT_HIT_KIND_BOX_EXIT 1u
#define RT_HIT_KIND_SPHERE_ENTER 0u
#define RT_HIT_KIND_SPHERE_EXIT 1u

typedef struct rt_hit_group_programs {
    uint32_t any_hit;      /* RT_ANYHIT_* */
    uint32_t intersection; /* RT_INTERSECTION_* */
} rt_hit_group_programs;

/* Per-ray traversal work counters used for the roofline (SURVEY.md section 8d). */
typedef struct rt_trace_stats {
    uint64_t rays;
    uint64_t internal_visits; /* internal nodes popped (each tests both children) */
    uint64_t leaf_visits;     /* triangles tested */
    uint64_t instance_visits; /* TLAS leaves entered */
    uint64_t max_stack;       /* deepest traversal stack seen */
} rt_trace_stats;

/* Environment cube: 6 faces (+X,-X,+Y,-Y,+Z,-Z) of size x size RGBA fp32 texels, mip 0 only. */
typedef struct rt_env_cube {
    const float *texels;
    uint32_t size;
    uint32_t _pad;
} rt_env_cube;

/* Per-(instance) hit-group record: what RtBindings writes per hit record for ray type 0
 * (src/ProgressiveRaytracingPipeline.cpp:220-227): VB SRV, IB SRV, 16 dwords of MaterialParams. */
typedef struct rt_hit_record {
    const rt_vertex *vertex_buffer;
    const uint32_t *index_buffer;
    rt_material_params material;
} rt_hit_record; /* 80 B */

/* Counts of rays actually traced by one dispatch (primary + secondary + shadow). */
typedef struct rt_ray_counts {
    uint64_t primary;
    uint64_t secondary; /* incoherent closest-hit rays: indirect diffuse + Phong lobe */
    uint64_t shadow;    /* any-hit rays */
} rt_ray_counts;

#ifdef __cplusplus
}
#endif

#endif /* RT_TYPES_H */
