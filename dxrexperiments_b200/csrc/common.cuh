// common.cuh — shared device/host helpers of librt_core.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/rt_core.h"

#define RT_STR2(x) #x
#define RT_STR(x) RT_STR2(x)

// ---------------------------------------------------------------------------------------------
// error handling
void rt_set_error(const char *fmt, ...);

#define RT_CUDA(call)                                                                              \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            rt_set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            return RT_ERR_CUDA;                                                                    \
        }                                                                                          \
    } while (0)

#define RT_REQUIRE(cond, msg)                                   \
    do {                                                        \
        if (!(cond)) {                                          \
            rt_set_error("invalid argument: %s (%s)", msg, #cond); \
            return RT_ERR_INVALID_ARG;                          \
        }                                                       \
    } while (0)

#define RT_LAUNCH_CHECK()                                                                \
    do {                                                                                 \
        cudaError_t e_ = cudaGetLastError();                                             \
        if (e_ != cudaSuccess) {                                                         \
            rt_set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e_), __FILE__, __LINE__); \
            return RT_ERR_CUDA;                                                          \
        }                                                                                \
    } while (0)

// ---------------------------------------------------------------------------------------------
// context

#define RT_MAX_BANDS 8
struct rt_workspace {  // wavefront queues, grown on demand (pipeline.cu)
    void *base = nullptr;
    uint64_t bytes = 0;
};

struct rt_context {
    int device = 0;
    int num_sms = 148;
    cudaStream_t stream = nullptr;
    bool owns_stream = false;
    uint64_t launches = 0;

    rt_per_frame_constants frame{};
    float *output[2] = {nullptr, nullptr};
    uint64_t pitch[2] = {0, 0};
    float *aov[RT_AOV_COUNT] = {};  // rt_set_aov_output: progressive AOV images, nullptr = unbound
    uint64_t aov_pitch[RT_AOV_COUNT] = {};
    const float *motion = nullptr;  // rt_set_instance_motion: n_motion row-major 3x4 world -> previous-world matrices (device)
    uint32_t n_motion = 0;
    const rt_deformation_desc *deform = nullptr;  // rt_set_instance_deformation: n_deform descriptors (device)
    uint32_t n_deform = 0;
    uint32_t *adaptive_counts = nullptr;  // rt_set_adaptive_sampling: width x height n_p | converged << 31 (device), nullptr = unbound
    float *adaptive_moments = nullptr;    // width x height (m1, m2) fp32 (device)
    const void *tlas = nullptr;
    rt_render_options render_options{1u, 0u};

    rt_workspace ws;
    cudaStream_t side_stream = nullptr;  // shadow depth-0 wave of a dispatch, overlapped with the secondary-ray chain
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // pixel bands 1.. of a dispatch (band 0 runs on `stream` / `side_stream`): {main, shadow-wave} streams, {fork, join, band-join} events
    cudaStream_t band_streams[RT_MAX_BANDS][2] = {};
    cudaEvent_t band_events[RT_MAX_BANDS][3] = {};
    cudaEvent_t ev_band_fork = nullptr;
    uint32_t *status = nullptr;          // device word: bit0 = traversal stack overflow, bit1 = procedural primitives reached by a triangles-only dispatch
    rt_hit_group_programs *hit_programs = nullptr;  // device copy of the table rt_trace_rays_hit_groups was last given
    unsigned long long *ray_counts = nullptr;  // device u64[32]: [0..2] rays traced; [8..12], [16..20], [24..28] rt_trace_stats of the primary / secondary / shadow stages
    // stage timing (optional)
    bool timing = false;
    bool collect_stats = false;  // instrumented trace kernels (rt_enable_trace_stats)
    bool capture = false;        // rt_enable_debug_capture: dispatches run as one band and keep their stage products
    uint64_t dbg_pixels = 0;     // pixels of the last captured dispatch (its workspace layout)
    cudaEvent_t ev[8] = {};
    bool ev_ready = false;
    double t_primary = 0, t_secondary = 0, t_shadow = 0;
    uint64_t n_secondary_timed = 0;
};

static_assert(sizeof(rt_deformation_desc) == 64, "rt_deformation_desc is four 16-byte loads");

struct rt_hit_record_dev {  // device copy of rt_hit_record
    const float *vb;        // rt_vertex[] viewed as floats (stride 6)
    const uint32_t *ib;
    rt_material_params mat;
};

struct rt_program {
    rt_context *ctx = nullptr;
    rt_program_kind kind = RT_PROGRAM_PROGRESSIVE;
    uint32_t hit_group_count = 0, miss_count = 0;
    // host mirror + device table of hit records indexed by instance * hit_group_count + ray_type
    rt_hit_record_dev *host_recs = nullptr;
    rt_hit_record_dev *dev_recs = nullptr;
    uint32_t n_recs = 0, cap_recs = 0;
    bool dirty = true;
    const float *env_texels = nullptr;
    uint32_t env_size = 0;
};

// ---------------------------------------------------------------------------------------------
// layout of the library's traversal section appended to every result buffer

#define RT_EXT_MAGIC 0x58425452u /* "RTBX" */

struct rt_ext_header {  // 128 bytes, located at align64(reference blob size)
    uint32_t magic;
    uint32_t count;         // number of leaves (triangles or instances)
    uint32_t root_ref;      // reference of the root (leaf ref if count == 1)
    uint32_t top_level;     // 1 for a TLAS
    uint64_t off_wide;      // byte offset from the start of the result buffer to the wide (BVH2) nodes
    uint64_t off_leaf;      // ... to the packed triangles (BLAS) / packed instances (TLAS)
    float root_center[3];   // root box (TLAS: tested once per ray; BLAS: informational)
    uint32_t _pad0;
    float root_half[3];
    uint32_t _pad1;
    uint64_t off_wide4;     // ... to the 4-wide nodes (rt_wide4_node), one per BVH2 internal node, same indexing
    // ALLOW_UPDATE builds only (0 otherwise): the two arrays FL/GpuBVH2Builder.cpp:82-92 appends for PERFORM_UPDATE
    uint64_t off_sort_cache;  // count x u32: load-order element -> sorted slot (RearrangeTriangles.hlsl:25-28)
    uint64_t off_parents;     // (2*count-1) x u32: parent of every node (ComputeAABBs.hlsli:160-164)
    uint32_t build_flags;     // RT_BUILD_FLAG_* of the build that produced this buffer
    uint32_t has_procedural;  // BLAS: built from >= 1 procedural-AABB geometry; TLAS: some instance's BLAS was
    uint64_t total_bytes;      // bytes of the result buffer in use (what rt_*_prebuild reported as result_bytes)
    uint64_t compacted_bytes;  // bytes a COMPACT copy needs: total_bytes minus the two update caches
    uint64_t _pad2[2];
};
static_assert(sizeof(rt_ext_header) == 128, "ext header");

// Wide node: an internal BVH2 node carrying BOTH child boxes (center/halfDim as the reference stores
// them) and child references.  64 B = 4 x 16-byte loads.  ref: bit31 set -> leaf slot in the low bits.
struct __align__(16) rt_wide_node {
    float lc[3];
    uint32_t left;
    float lh[3];
    uint32_t right;
    float rc[3];
    uint32_t _p0;
    float rh[3];
    uint32_t _p1;
};
static_assert(sizeof(rt_wide_node) == 64, "wide node");

// 4-wide node: the (up to) four descendants of BVH2 node i reached by opening, twice, the internal child with the
// largest surface area (k_collapse4).  wide4[i] exists for EVERY BVH2 internal node i, so no allocation or queue is
// needed to build it; a traversal that starts at node 0 only ever touches the nodes reachable through wide4 links.
// One 128-byte line = 8 x 16-byte loads: q[2k] = {center_k.xyz, ref_k}, q[2k+1] = {half_k.xyz, -}.
// Boxes are the reference's own center/half values, so a child box test is the arithmetic of RayBoxTest unchanged.
// Empty slot: ref = RT_WIDE4_EMPTY, center 0, half -1 (the slab test then fails for every ray).
struct __align__(16) rt_wide4_node {
    struct {
        float c[3];
        uint32_t ref;
        float h[3];
        uint32_t _p;
    } child[4];
};
static_assert(sizeof(rt_wide4_node) == 128, "wide4 node");
#define RT_WIDE4_EMPTY 0x7fffffffu

// Packed triangle: 9 floats + PrimitiveMetaData in 48 B = 3 x 16-byte loads.
struct __align__(16) rt_packed_tri {
    float v[9];
    uint32_t primitive_index;
    uint32_t geometry_index;
    uint32_t geometry_flags;
};
static_assert(sizeof(rt_packed_tri) == 48, "packed tri");
// A procedural primitive travels in the same 48-byte record: v[0..5] = AABB min, max, v[6..8] = 0, and this bit in
// geometry_flags (never a D3D12 geometry flag); the reference-format Primitive / PrimitiveMetaData carry type 2 and
// the plain flags.
#define RT_PACKED_PROCEDURAL 0x80000000u

// Packed instance (TLAS leaf): world->object 3x4, ids, and the BLAS traversal pointers. 96 B.
struct __align__(16) rt_packed_instance {
    float w2o[12];
    uint32_t instance_id_and_mask;
    uint32_t hit_group_and_flags;
    uint32_t instance_index;
    uint32_t blas_root_ref;
    const rt_wide_node *blas_wide;
    const rt_packed_tri *blas_tris;
    const rt_wide4_node *blas_wide4;
    uint64_t _pad;
};
static_assert(sizeof(rt_packed_instance) == 96, "packed instance");
#define RT_PACKED_INSTANCE_IDENTITY 0x80000000u /* in rt_packed_instance.hit_group_and_flags only */

static inline __host__ __device__ uint64_t align_up(uint64_t x, uint64_t a) { return (x + a - 1) / a * a; }

// ---------------------------------------------------------------------------------------------
// small device vector helpers (explicitly unfused where bit-parity with the oracle matters)

struct f3 {
    float x, y, z;
};
__device__ __forceinline__ f3 mk3(float x, float y, float z) { return f3{x, y, z}; }
// Exact (never contracted) arithmetic: nvcc will not fuse __fmul_rn/__fadd_rn into FMAs.
__device__ __forceinline__ float mul_(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float add_(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub_(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float div_(float a, float b) { return __fdiv_rn(a, b); }

// Rec. 601 luma: reinhardToneMap's luminance (DenoiseCommon.hlsli:33-38), the edge-stopping luminance of
// rt_denoise_progressive and the luminance whose moments adaptive sampling (rt_set_adaptive_sampling) accumulates.
__device__ __forceinline__ float luminance(float r, float g, float b) { return (r * 0.299f + g * 0.587f) + b * 0.114f; }

__device__ __forceinline__ f3 xform_point(const float *m, f3 v) {
    return mk3(add_(add_(add_(mul_(m[0], v.x), mul_(m[1], v.y)), mul_(m[2], v.z)), m[3]),
               add_(add_(add_(mul_(m[4], v.x), mul_(m[5], v.y)), mul_(m[6], v.z)), m[7]),
               add_(add_(add_(mul_(m[8], v.x), mul_(m[9], v.y)), mul_(m[10], v.z)), m[11]));
}
__device__ __forceinline__ f3 xform_vector(const float *m, f3 v) {
    return mk3(add_(add_(mul_(m[0], v.x), mul_(m[1], v.y)), mul_(m[2], v.z)),
               add_(add_(mul_(m[4], v.x), mul_(m[5], v.y)), mul_(m[6], v.z)),
               add_(add_(mul_(m[8], v.x), mul_(m[9], v.y)), mul_(m[10], v.z)));
}

static inline int rt_div_up(uint64_t a, uint64_t b) { return int((a + b - 1) / b); }
