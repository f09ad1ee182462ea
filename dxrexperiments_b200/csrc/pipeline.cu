// pipeline.cu — wavefront ray-generation / closest-hit / miss pipeline for sm_100a.
//
// Replaces the Fallback Layer's uber-shader state machine (FL/UberShaderRayTracingProgram.cpp:213-272,
// FL/StateMachineLib.hlsl, dxrfallbackcompiler.dll) for the two shader libraries of the application:
//   assets/shaders/ProgressiveRaytracing.hlsl (RayGen :11-39, shade :80-148, closest-hit/miss :150-164)
//   assets/shaders/RealtimeRaytracing.hlsl    (RayGen :22-46, shadeAOV :65-103, closest-hit/miss :105-126)
// The recursion "TraceRay inside closest-hit" becomes explicit stages with compacted ray queues:
//
//   K1 primary   : raygen + closest-hit traversal, 8x4 pixel tile per warp            -> hit records
//   K2 shade0    : miss -> environment -> output; hit -> depth-0 shade(), emits 2 shadow rays (4 in the AO
//                  debug view) and up to 2 secondary rays per hit pixel into compacted queues
//   K3 secondary : closest-hit traversal of the incoherent secondary rays (the headline metric)
//   K4 shadow0   : any-hit traversal of the depth-0 shadow rays
//   K5 shade1    : depth-1 shade() of every secondary hit, emits its 2 shadow rays (compacted)
//   K6 shadow1   : any-hit traversal of the depth-1 shadow rays
//   K7 resolve   : recombines exactly the expression tree of shade()/shadeAOV() and accumulates
//
// Queue layout: every ray queue is PLANAR by ray kind — ray k of hit slot s lives at k * plane + s (plane = pixels of
// the dispatch for the depth-0 queues, twice that for the depth-1 shadow queue), not at s * kinds + k.  A warp of a
// trace kernel therefore holds rays of ONE kind from neighbouring pixels: all directional-light shadow rays are
// parallel, all point-light rays converge on one point, Phong-lobe rays cluster around the mirror directions, and
// only the cosine-hemisphere plane is truly incoherent.  Interleaved queues put two unrelated directions in adjacent
// lanes and halved the SIMT efficiency of the shadow kernels (profiles/r1_ncu_trace_w4.md: 13.8-18.2 of 32 lanes).
// Rays are "sorted by kind" by construction, with no sorting pass.
//
// Random numbers are a pure function of (pixel, frameCount) and are re-derived at each depth exactly as the
// shaders re-initialise their seed, so no RNG state travels through the queues.
#include <cuda_fp16.h>

#include <cstdio>
#include <cstdlib>

#include "shade.cuh"
#include "trace.cuh"
#include "trace_persistent.cuh"

namespace {

constexpr int kBlock = 128;

struct Launch {
    rt_per_frame_constants f;
    uint32_t width, height;  // full launch dimensions
    uint32_t x0, y0, rw, rh; // pixel rectangle handled by this dispatch (rh counts the dispatch's own rows: "virtual" rows)
    uint32_t v0;             // first virtual row of this band of the dispatch
    uint32_t stripShift, stripGroups, stripGroup;  // strip-interleaved dispatch (stripGroups > 1): virtual row -> image row, see image_row()
    float jitterScale;
    uint32_t realtime;
    uint32_t shadowsPerHit;  // 2, or 4 in the ambient-occlusion debug view
    uint32_t maxDepth;       // MAX_RADIANCE_RAY_DEPTH: 1 (reference) or 2 (rt_set_render_options)
    uint32_t halfTargets;    // stores round through fp16 (R16G16B16A16_FLOAT emulation)
};

struct WS {
    uint32_t plane;     // P: plane stride of the depth-0 queues (the depth-1 shadow queue uses 2P)
    float4 *hitA;       // [P]  primary hit: t, u, v, primitive
    uint32_t *hitRec;   // [P]  hit-group record index
    uint32_t *counters; // [0] hit slots, [1] depth-1 shadow pairs
    uint4 *slotInfo;    // [P]  pixel (region-linear), record, flags, -
    float4 *S0, *S1, *S2;
    float *S3;
    rt_ray *shadowQ0;   // [4P]
    uint8_t *vis0;
    rt_ray *secQ;       // [2P]
    float4 *secHitA;
    uint32_t *secRec;
    uint32_t *secShadow; // [2P] index of the depth-1 shadow pair, or ~0
    float4 *T0, *T1, *T2;
    rt_ray *shadowQ1;   // [4P]
    uint8_t *vis1;
    // depth-2 wave (maxDepth == 2 only): the Phong-lobe ray of every secondary hit, same planar indexing as secQ
    rt_ray *terQ;       // [2P]
    float4 *terHitA;    // [2P]
    uint32_t *terRec;   // [2P]
    float4 *terRad;     // [2P] radiance returned by the depth-2 hit (or the environment)
    float2 *T3;         // [2P] {brdf, pdf} of the depth-1 lobe sample
};

enum : uint32_t {
    SLOT_DEBUG2_DIR = 1u,    // debug == 2 and the directional light was selected
    SLOT_DEBUG2_POINT = 2u,  // debug == 2 and the point light was selected
    SLOT_HAS_SPEC = 4u,
    SLOT_HAS_DIFFUSE = 8u,
    SLOT_UNIFORM = 16u,
    SLOT_AO = 32u,
};

// Image row of row `r` of a band.  A plain (region) dispatch covers rows y0 .. y0+rh-1.  A strip-interleaved dispatch
// (rt_dispatch_rays_interleaved: screen-tile sharding across GPUs) covers the strips of 2^stripShift rows whose index is
// congruent to stripGroup modulo stripGroups, packed into consecutive virtual rows.
__device__ __forceinline__ uint32_t image_row(const Launch &L, uint32_t r) {
    const uint32_t v = L.v0 + r;
    if (L.stripGroups <= 1) return L.y0 + v;
    return (((v >> L.stripShift) * L.stripGroups + L.stripGroup) << L.stripShift) + (v & ((1u << L.stripShift) - 1u));
}

__device__ __forceinline__ void store_ray(rt_ray *q, f3 o, float tmin, f3 d, float tmax) {
    float4 *p = reinterpret_cast<float4 *>(q);
    p[0] = make_float4(o.x, o.y, o.z, tmin);
    p[1] = make_float4(d.x, d.y, d.z, tmax);
}

__device__ __forceinline__ uint32_t warp_alloc(bool want, uint32_t *counter) {
    const unsigned active = __ballot_sync(0xffffffffu, want);
    if (!want) return 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(active) - 1;
    uint32_t base = 0;
    if (lane == leader) base = atomicAdd(counter, uint32_t(__popc(active)));
    base = __shfl_sync(active, base, leader);
    return base + __popc(active & ((1u << lane) - 1));
}

__device__ __forceinline__ void warp_count_add(unsigned long long *dst, uint32_t v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(dst, (unsigned long long)v);
}

__device__ __forceinline__ void flush_stats(const TraceCtr &c, uint32_t rays, unsigned long long *stats) {
    // block-level reduction would be cheaper; this path only runs in instrumented (untimed) passes
    uint32_t v[4] = {rays, c.internal, c.leaf, c.inst};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
    }
    uint32_t m = c.max_stack;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (v[k]) atomicAdd(&stats[k], (unsigned long long)v[k]);
        atomicMax(&stats[4], (unsigned long long)m);
    }
}

#ifndef RT_DISPATCH_BANDS
#define RT_DISPATCH_BANDS 2  // pixel bands per dispatch (1 = off, at most RT_MAX_BANDS)
#endif
// ------------------------------------------------------------------------------------------------ K1
#ifndef RT_PRIMARY_MIN_BLOCKS
#define RT_PRIMARY_MIN_BLOCKS 7  // 72 registers: the kernel is latency-bound (26 % of the warp slots active at 6 blocks); A/B round 2: 5 / 6 / 7 / 8
                                 // blocks per SM = 5363 / 5767 / 6103 / 5802 Mrays/s on C2, 3053 / 3160 / 3329 / 3035 on 1.31 M triangles
#endif
// Adaptive sampling (rt_set_adaptive_sampling): the per-pixel sample counts (bit 31: converged) and luminance moments, in
// image order.  Only the ADAPTIVE instantiations of k_primary, k_primary_inst, k_shade_primary and k_resolve read them.
struct Adaptive {
    uint32_t *counts;
    float2 *moments;
};

__device__ __forceinline__ size_t image_index(const Launch &L, uint32_t x, uint32_t y) { return size_t(y) * L.width + x; }

// INST: also store each pixel's InstanceIndex() to inst[p], which the previous-position AOV looks its motion up by (the
// hit-group record does not determine the instance: it is RayContribution + InstanceContributionToHitGroupIndex).
// ADAPTIVE: a converged pixel traces nothing and is not counted.
template <bool STATS, bool INST, bool ADAPTIVE>
__device__ __forceinline__ void primary_tile(const Launch &L, const void *tlas, const WS &ws, uint32_t *status, unsigned long long *stats,
                                             uint32_t *inst, const uint32_t *counts) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t tilesX = (L.rw + 7) / 8;
    const uint32_t tile = blockIdx.x * (kBlock / 32) + warp;
    const uint32_t lx = (tile % tilesX) * 8 + (lane & 7), ly = (tile / tilesX) * 4 + (lane >> 3);
    const bool inside = lx < L.rw && ly < L.rh &&
                        (!ADAPTIVE || !(counts[image_index(L, L.x0 + lx, image_row(L, ly))] & RT_ADAPTIVE_CONVERGED));
    TraceCtr ctr{0, 0, 0, 0};
    if (inside) {
        const uint32_t x = L.x0 + lx, y = image_row(L, ly);
        f3 o, d;
        primary_ray(L.f, L.width, L.height, x, y, L.jitterScale, o, d);
        TraceAccel A = resolve_tlas(tlas, status);
        TraceHit h;
        if (STATS)  // instrumented: BVH2 in the reference's visit order
            trace_ray<false, STATS>(A, o.x, o.y, o.z, 0.0f, d.x, d.y, d.z, RT_RAY_MAX_T, RT_RAY_FLAG_CULL_BACK_FACING_TRIANGLES, 0xFF, 0, 0, h,
                                    &ctr, status);
        else
            trace_ray4(A, o.x, o.y, o.z, 0.0f, d.x, d.y, d.z, RT_RAY_MAX_T, RT_RAY_FLAG_CULL_BACK_FACING_TRIANGLES, 0xFF, 0, h, status);
        const uint32_t p = ly * L.rw + lx;
        ws.hitA[p] = make_float4(h.t, h.u, h.v, __uint_as_float(h.prim));
        ws.hitRec[p] = h.record;
        if (INST) inst[p] = h.inst_index;
    }
    if (STATS) flush_stats(ctr, inside ? 1u : 0u, stats);
}

template <bool STATS, bool ADAPTIVE>
__global__ void __launch_bounds__(kBlock, RT_PRIMARY_MIN_BLOCKS) k_primary(const __grid_constant__ Launch L, const void *tlas, WS ws, uint32_t *status,
                                                    unsigned long long *stats, const uint32_t *counts) {
    primary_tile<STATS, false, ADAPTIVE>(L, tlas, ws, status, stats, nullptr, counts);
}

// k_primary for a dispatch with the previous-position AOV bound
template <bool STATS, bool ADAPTIVE>
__global__ void __launch_bounds__(kBlock, RT_PRIMARY_MIN_BLOCKS) k_primary_inst(const __grid_constant__ Launch L, const void *tlas, WS ws,
                                                                                uint32_t *status, unsigned long long *stats, uint32_t *inst,
                                                                                const uint32_t *counts) {
    primary_tile<STATS, true, ADAPTIVE>(L, tlas, ws, status, stats, inst, counts);
}

// ------------------------------------------------------------------------------------------------ light helpers
// evaluateDirectionalLight / evaluatePointLight without the visibility factor
// (S/RaytracingCommon.hlsli:126-147); the shadow ray is queued instead of traced.
struct LightEval {
    f3 dirPre;      // color.rgb * color.a * NoL
    f3 dirL;
    f3 pointPre;    // color.rgb * color.a * NoL
    f3 pointL;
    float pointDist, falloff;
};
__device__ __forceinline__ LightEval eval_lights(const rt_per_frame_constants &f, f3 p, f3 n) {
    LightEval e;
    const rt_directional_light &dl = f.directionalLight;
    e.dirL = normalize3(-mk3(dl.forwardDir[0], dl.forwardDir[1], dl.forwardDir[2]));
    float NoL = saturatef(dot3(n, e.dirL));
    e.dirPre = mk3(dl.color[0], dl.color[1], dl.color[2]) * dl.color[3] * NoL;
    const rt_point_light &pl = f.pointLight;
    f3 path = mk3(pl.worldPos[0], pl.worldPos[1], pl.worldPos[2]) - p;
    e.pointDist = length3(path);
    e.pointL = normalize3(path);
    float NoLp = saturatef(dot3(n, e.pointL));
    e.falloff = 1.0f / (2 * RT_M_PI * e.pointDist * e.pointDist);
    e.pointPre = mk3(pl.color[0], pl.color[1], pl.color[2]) * pl.color[3] * NoLp;
    return e;
}

// n: the samples already in the running mean (accumCount, or the pixel's count under adaptive sampling)
__device__ __forceinline__ void write_pixel(const Launch &L, float *out, uint64_t pitch, uint32_t x, uint32_t y, f3 c, bool accumulate,
                                            uint32_t n) {
    float4 *px = reinterpret_cast<float4 *>(reinterpret_cast<uint8_t *>(out) + size_t(y) * pitch) + x;
    float4 cur = make_float4(fmaxf(c.x, 0.0f), fmaxf(c.y, 0.0f), fmaxf(c.z, 0.0f), 1.0f);
    if (accumulate) {  // RayGen: S/ProgressiveRaytracing.hlsl:36-38
        float4 prev = *px;
        const float fn = float(n), fn1 = float(n + 1);
        cur = make_float4((fn * prev.x + cur.x) / fn1, (fn * prev.y + cur.y) / fn1, (fn * prev.z + cur.z) / fn1,
                          (fn * prev.w + cur.w) / fn1);
    }
    if (L.halfTargets)  // what an R16G16B16A16_FLOAT target holds after the store (and returns as `prev` next frame)
        cur = make_float4(__half2float(__float2half_rn(cur.x)), __half2float(__float2half_rn(cur.y)), __half2float(__float2half_rn(cur.z)),
                          __half2float(__float2half_rn(cur.w)));
    *px = cur;
}

// AOV outputs of a progressive dispatch (rt_set_aov_output): one RGBA fp32 image per rt_aov id, bit k of `mask` set when
// AOV k is bound.  Only the <true> instantiations of k_shade_primary and k_resolve read it.
struct AovOut {
    float *ptr[RT_AOV_COUNT];
    uint64_t pitch[RT_AOV_COUNT];
    uint32_t mask;
    uint32_t n_motion;      // rt_set_instance_motion: matrices bound (0: none)
    const float4 *motion;   // 3 rows of (m0, m1, m2, m3) per instance
    const uint32_t *inst;   // [P] InstanceIndex() of each pixel's primary hit (k_primary_inst), previous-position AOV only
    const rt_deformation_desc *deform;  // rt_set_instance_deformation: n_deform descriptors (0: none)
    uint32_t n_deform;
};

// P' of the previous-position AOV for the primary hit P of workspace pixel p on primitive prim of record R at
// barycentrics (bu, bv) (include/rt_core.h states the rule).
__device__ __forceinline__ f3 previous_position(const AovOut &a, uint32_t p, f3 P, const rt_hit_record_dev &R, uint32_t prim, float bu,
                                                float bv, uint32_t *status) {
    const uint32_t i = a.inst[p];
    if (i < a.n_motion) {
        const float4 *m = a.motion + 3 * size_t(i);
        const float4 r0 = __ldg(m), r1 = __ldg(m + 1), r2 = __ldg(m + 2);
        P = mk3(((r0.x * P.x + r0.y * P.y) + r0.z * P.z) + r0.w, ((r1.x * P.x + r1.y * P.y) + r1.z * P.z) + r1.w,
                ((r2.x * P.x + r2.y * P.y) + r2.z * P.z) + r2.w);
    }
    if (i >= a.n_deform) return P;
    // the descriptor as four 16-byte loads: {pointer, stride_bytes, vertex_count}, then the three rows of the 3x4
    const uint4 *q = reinterpret_cast<const uint4 *>(a.deform + i);
    const uint4 h = __ldg(q);
    const float *prev = reinterpret_cast<const float *>(uint64_t(h.x) | (uint64_t(h.y) << 32));
    if (prev == nullptr) return P;
    const uint32_t *idx = R.ib + size_t(prim) * 3;
    const uint32_t i0 = __ldg(idx), i1 = __ldg(idx + 1), i2 = __ldg(idx + 2);
    if (h.z < 12u || (h.z & 3u) || i0 >= h.w || i1 >= h.w || i2 >= h.w) {
        atomicOr(status, 8u);  // rt_get_status -> RT_ERR_INVALID_ARG, as for a missing hit record
        return P;
    }
    const size_t s = h.z / 4u;
    const float *q0 = prev + i0 * s, *q1 = prev + i1 * s, *q2 = prev + i2 * s;
    const float *v0 = R.vb + size_t(i0) * 6, *v1 = R.vb + size_t(i1) * 6, *v2 = R.vb + size_t(i2) * 6;
    const f3 d0 = mk3(__ldg(q0) - __ldg(v0), __ldg(q0 + 1) - __ldg(v0 + 1), __ldg(q0 + 2) - __ldg(v0 + 2));
    const f3 d1 = mk3(__ldg(q1) - __ldg(v1), __ldg(q1 + 1) - __ldg(v1 + 1), __ldg(q1 + 2) - __ldg(v1 + 2));
    const f3 d2 = mk3(__ldg(q2) - __ldg(v2), __ldg(q2 + 1) - __ldg(v2 + 1), __ldg(q2 + 2) - __ldg(v2 + 2));
    const float b0 = 1.f - bu - bv, b1 = bu, b2 = bv;
    const f3 D = (d0 * b0 + d1 * b1) + d2 * b2;
    const float4 *m = reinterpret_cast<const float4 *>(q + 1);
    const float4 r0 = __ldg(m), r1 = __ldg(m + 1), r2 = __ldg(m + 2);
    return mk3(P.x + ((r0.x * D.x + r0.y * D.y) + r0.z * D.z), P.y + ((r1.x * D.x + r1.y * D.y) + r1.z * D.z),
               P.z + ((r2.x * D.x + r2.y * D.y) + r2.z * D.z));
}

// AOVs 0-4 accumulate exactly as the beauty frame does, so each one equals the matching debug view bit for bit.
__device__ __forceinline__ void write_aov(const Launch &L, const AovOut &a, int k, uint32_t x, uint32_t y, f3 c, uint32_t n) {
    if (a.mask & (1u << k)) write_pixel(L, a.ptr[k], a.pitch[k], x, y, c, true, n);
}

// The normal and position AOVs: the running mean of (N or P, coverage) without write_pixel's clamp at 0, so that negative
// components survive and `w` is the fraction of samples that hit.
__device__ __forceinline__ void write_geometry_aov(const Launch &L, const AovOut &a, int k, uint32_t x, uint32_t y, f3 n, float coverage,
                                                   uint32_t cnt) {
    if (!(a.mask & (1u << k))) return;
    float4 *px = reinterpret_cast<float4 *>(reinterpret_cast<uint8_t *>(a.ptr[k]) + size_t(y) * a.pitch[k]) + x;
    const float4 prev = *px;
    const float fn = float(cnt), fn1 = float(cnt + 1);
    float4 cur = make_float4((fn * prev.x + n.x) / fn1, (fn * prev.y + n.y) / fn1, (fn * prev.z + n.z) / fn1, (fn * prev.w + coverage) / fn1);
    if (L.halfTargets)
        cur = make_float4(__half2float(__float2half_rn(cur.x)), __half2float(__float2half_rn(cur.y)), __half2float(__float2half_rn(cur.z)),
                          __half2float(__float2half_rn(cur.w)));
    *px = cur;
}

// Adaptive sampling: fold the sample c (clamped as write_pixel clamps it) into pixel i's luminance moments and count it.
__device__ __forceinline__ void write_moments(const Adaptive &ad, size_t i, f3 c, uint32_t n) {
    const float l = luminance(fmaxf(c.x, 0.0f), fmaxf(c.y, 0.0f), fmaxf(c.z, 0.0f));
    const float2 m = ad.moments[i];
    const float fn = float(n), fn1 = float(n + 1);
    ad.moments[i] = make_float2((fn * m.x + l) / fn1, (fn * m.y + l * l) / fn1);
    ad.counts[i] = n + 1;
}

// ------------------------------------------------------------------------------------------------ K2
// Coherence binning (north star: "rays compacted and sorted ... between bounces"): a block shades one 16x16 pixel tile
// and hands out the tile's hit slots bin by bin, the bin being {hit-group record (material / instance), direction octant of
// the indirect-diffuse ray}.  The hits of a tile lie close together in space, so after the binning 32 consecutive slots —
// one warp of the queue kernels, for every ray kind of those slots — hold rays that start near each other, on the same
// material, and head into the same octant: they walk the same part of the tree.  The sort is a counting sort in shared
// memory inside the shading kernel (one global atomic per block); no pass over the queues, no extra launch.
// The reference has no counterpart: the Fallback Layer traces in fixed 8x8 pixel groups and never reorders rays
// (FL/UberShaderRayTracingProgram.cpp:268-272).
constexpr int kShadeTile = 16;                     // pixels per tile edge
constexpr int kShadeThreads = kShadeTile * kShadeTile;
constexpr int kBins = 32;                          // 4 record classes x 8 octants

__device__ __forceinline__ uint32_t octant_of(f3 d) {
    return (d.x < 0.0f ? 1u : 0u) | (d.y < 0.0f ? 2u : 0u) | (d.z < 0.0f ? 4u : 0u);
}

// The shading kernels are latency-bound (ncu: long-scoreboard stalls, 41-47 % of the warp slots occupied at 52-64 registers): register
// budgets for more resident blocks are worth ~1 % of a stage-timed frame (A/B: k_shade_secondary 8 -> 10 blocks of 128: 99.8 -> 94.4 us,
// k_resolve 9 -> 12 blocks of 128: 61.5 -> 60.1 us; in the overlapped dispatch the gain hides behind the other band's traversal).
// k_shade_primary stays at its natural 64 registers: 5 blocks of 256 (48 registers) spill 240 bytes per thread, +67 MB of DRAM
// writes per frame, 138 -> 154 us under ncu.
#ifndef RT_SHADE1_MIN_BLOCKS
#define RT_SHADE1_MIN_BLOCKS 10
#endif
#ifndef RT_RESOLVE_MIN_BLOCKS
#define RT_RESOLVE_MIN_BLOCKS 12
#endif
// AOV: write the AOV outputs of the primary misses and the normal, position and previous-position AOVs of every pixel
// (progressive program only).  ADAPTIVE: a converged pixel is treated as outside the launch, the running means use the
// pixel's count, and a miss folds its sample into the moments here (a hit does so in k_resolve).
template <bool AOV, bool ADAPTIVE>
__global__ void __launch_bounds__(kShadeThreads) k_shade_primary(const __grid_constant__ Launch L, WS ws, const rt_hit_record_dev *recs,
                                                                 uint32_t n_recs, const float *env, uint32_t envSize, float *out0,
                                                                 uint64_t pitch0, float *out1, uint64_t pitch1,
                                                                 unsigned long long *rayCounts, uint32_t *status, const AovOut aov,
                                                                 const Adaptive ad) {
    __shared__ uint32_t s_count[kBins], s_offset[kBins], s_base;
    const uint32_t tilesX = (L.rw + kShadeTile - 1) / kShadeTile;
    const uint32_t lx = (blockIdx.x % tilesX) * kShadeTile + (threadIdx.x % kShadeTile);
    const uint32_t ly = (blockIdx.x / tilesX) * kShadeTile + (threadIdx.x / kShadeTile);
    const uint32_t p = ly * L.rw + lx;
    bool inRange = lx < L.rw && ly < L.rh;
    uint32_t n = L.f.cameraParams.accumCount;
    if (ADAPTIVE && inRange) {
        n = ad.counts[image_index(L, L.x0 + lx, image_row(L, ly))];
        if (n & RT_ADAPTIVE_CONVERGED) inRange = false;
    }
    if (threadIdx.x < kBins) s_count[threadIdx.x] = 0;
    bool isHit = false;
    float4 hA = make_float4(0, 0, 0, 0);
    uint32_t x = 0, y = 0;
    f3 o = mk3(0, 0, 0), d = mk3(0, 0, 1);
    if (inRange) {
        x = L.x0 + lx, y = image_row(L, ly);
        primary_ray(L.f, L.width, L.height, x, y, L.jitterScale, o, d);
        hA = ws.hitA[p];
        isHit = __float_as_uint(hA.w) != RT_NO_HIT;
        if (!isHit) {  // PrimaryMiss
            f3 c = sample_env(env, envSize, d) * L.f.options.environmentStrength;
            if (L.realtime) {
                write_pixel(L, out0, pitch0, x, y, c, false, n);
                write_pixel(L, out1, pitch1, x, y, mk3(0, 0, 0), false, n);
            } else {
                write_pixel(L, out0, pitch0, x, y, c, true, n);
                if (AOV) {  // every debug view shows the environment for a miss
                    write_aov(L, aov, RT_AOV_DIRECT, x, y, c, n);
                    write_aov(L, aov, RT_AOV_INDIRECT_DIFFUSE, x, y, c, n);
                    write_aov(L, aov, RT_AOV_INDIRECT_SPECULAR, x, y, c, n);
                    write_aov(L, aov, RT_AOV_ALBEDO, x, y, c, n);
                    write_aov(L, aov, RT_AOV_FRESNEL, x, y, c, n);
                    write_geometry_aov(L, aov, RT_AOV_NORMAL, x, y, mk3(0, 0, 0), 0.0f, n);
                    write_geometry_aov(L, aov, RT_AOV_POSITION, x, y, mk3(0, 0, 0), 0.0f, n);
                    write_geometry_aov(L, aov, RT_AOV_PREVIOUS_POSITION, x, y, mk3(0, 0, 0), 0.0f, n);
                }
                if (ADAPTIVE) write_moments(ad, image_index(L, x, y), c, n);
            }
        }
    }
    // ---- shade first (everything stays in registers), allocate the slot afterwards: the bin needs the sampled direction
    uint32_t nShadow = 0, nSecondary = 0, rec = 0, flags = 0, bin = 0;
    f3 pos = mk3(0, 0, 0);
    float4 s0 = make_float4(0, 0, 0, 0), s1 = s0, s2 = s0;
    float s3 = 0.0f;
    float shTmax[4] = {-1.0f, -1.0f, -1.0f, -1.0f}, shTmin = RT_RAY_EPSILON, secTmax[2] = {-1.0f, -1.0f};
    f3 shDir[4] = {mk3(0, 0, 1), mk3(0, 0, 1), mk3(0, 0, 1), mk3(0, 0, 1)}, secDir[2] = {mk3(0, 0, 1), mk3(0, 0, 1)};
    if (isHit) {
        rec = ws.hitRec[p];
        if (rec >= n_recs) rec = 0, atomicOr(status, 8u);  // a hit on an instance without a bound record: rt_get_status -> RT_ERR_INVALID_ARG
        const rt_hit_record_dev &R = recs[rec];
        const uint32_t prim = __float_as_uint(hA.w);
        const f3 N = normalize3(interpolate_normal(R, prim, hA.y, hA.z));
        if (AOV) write_geometry_aov(L, aov, RT_AOV_NORMAL, x, y, N, 1.0f, n);
        pos = o + hA.x * d;  // HitWorldPosition
        if (AOV) write_geometry_aov(L, aov, RT_AOV_POSITION, x, y, pos, 1.0f, n);
        if (AOV && (aov.mask & (1u << RT_AOV_PREVIOUS_POSITION)))
            write_geometry_aov(L, aov, RT_AOV_PREVIOUS_POSITION, x, y, previous_position(aov, p, pos, R, prim, hA.y, hA.z, status), 1.0f, n);
        const rt_debug_options &opt = L.f.options;
        if (!L.realtime && opt.showAmbientOcclusionOnly) {
            // evaluateAO: S/RaytracingCommon.hlsli:98-124 — 4 shadow rays, tMax 10
            flags = SLOT_AO;
            uint32_t seed = init_rand(x + y * L.width, L.f.cameraParams.frameCount);
            float nol[4], pdf[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (opt.cosineHemisphereSampling) {
                    shDir[i] = cos_hemisphere(seed, N);
                    nol[i] = saturatef(dot3(N, shDir[i]));
                    pdf[i] = nol[i] / RT_M_PI;
                } else {
                    shDir[i] = uniform_hemisphere(seed, N);
                    nol[i] = saturatef(dot3(N, shDir[i]));
                    pdf[i] = 1.0f / (2.0f * RT_M_PI);
                }
                shTmax[i] = 10.0f;
            }
            nShadow = 4;
            s0 = make_float4(nol[0], nol[1], nol[2], nol[3]);
            s1 = make_float4(pdf[0], pdf[1], pdf[2], pdf[3]);
            bin = octant_of(shDir[0]);
        } else {
            uint32_t seed = init_rand(x + y * L.width, L.f.cameraParams.frameCount);
            LightEval le = eval_lights(L.f, pos, N);
            bool useDir = true, usePoint = true;
            if (!L.realtime && opt.debug == 2) {
                if (next_rand(seed) < 0.5f) usePoint = false, flags |= SLOT_DEBUG2_DIR;
                else useDir = false, flags |= SLOT_DEBUG2_POINT;
            }
            shDir[0] = le.dirL, shTmax[0] = useDir ? RT_RAY_MAX_T : -1.0f;
            shDir[1] = le.pointL, shTmax[1] = usePoint ? le.pointDist - RT_RAY_EPSILON : -1.0f;
            shDir[2] = shDir[3] = le.dirL;  // unused planes of the AO layout: inactive
            nShadow = (useDir ? 1 : 0) + (usePoint ? 1 : 0);
            // indirect diffuse: S/ProgressiveRaytracing.hlsl:57-78,107-110
            float uniformNoL = 0.0f;
            const bool hasDiffuse = !L.realtime && !opt.noIndirectDiffuse;
            if (hasDiffuse) {
                if (opt.cosineHemisphereSampling) secDir[0] = cos_hemisphere(seed, N);
                else {
                    secDir[0] = uniform_hemisphere(seed, N);
                    uniformNoL = saturatef(dot3(N, secDir[0]));
                    flags |= SLOT_UNIFORM;
                }
                flags |= SLOT_HAS_DIFFUSE;
                secTmax[0] = RT_RAY_MAX_T;
            }
            // indirect specular: S/ProgressiveRaytracing.hlsl:114-131
            f3 fres = mk3(0, 0, 0);
            float pdf = 1.0f, brdf = 0.0f;
            const bool hasSpec = (R.mat.type == 1 || R.mat.type == 2) && R.mat.reflectivity > 0.001f;
            if (hasSpec) {
                float exponent = expf((1.0f - R.mat.roughness) * 12.0f);
                f3 mirror = reflect3(d, N);
                secDir[1] = phong_lobe(seed, mirror, exponent, pdf, brdf);
                fres = fresnel_schlick(d, N, mk3(R.mat.specular[0], R.mat.specular[1], R.mat.specular[2]));
                flags |= SLOT_HAS_SPEC;
                secTmax[1] = RT_RAY_MAX_T;
            }
            nSecondary = (hasDiffuse ? 1 : 0) + (hasSpec ? 1 : 0);
            s0 = make_float4(le.dirPre.x, le.dirPre.y, le.dirPre.z, le.falloff);
            s1 = make_float4(le.pointPre.x, le.pointPre.y, le.pointPre.z, pdf);
            s2 = make_float4(fres.x, fres.y, fres.z, brdf);
            s3 = uniformNoL;
            bin = octant_of(hasDiffuse ? secDir[0] : secDir[1]);
        }
        bin |= ((rec >> 1) & 3u) << 3;  // records come in pairs per instance (ray types): the instance / material class
    }
    // ---- slot allocation: counting sort of the tile's hits by bin
    const int lane = threadIdx.x & 31;
    uint32_t slot = 0xffffffffu;
    __syncthreads();  // s_count cleared
    uint32_t inWarp = 0, warpBase = 0;
    {
        const unsigned hitMask = __ballot_sync(0xffffffffu, isHit);
        if (isHit) {
            const unsigned same = __match_any_sync(hitMask, bin);
            inWarp = __popc(same & ((1u << lane) - 1u));
            const int leader = __ffs(same) - 1;
            if (lane == leader) warpBase = atomicAdd(&s_count[bin], uint32_t(__popc(same)));
            warpBase = __shfl_sync(same, warpBase, leader);
        }
    }
    __syncthreads();
    if (threadIdx.x < 32) {  // exclusive scan of the 32 bin counts, one global allocation for the tile
        const uint32_t c = s_count[lane];
        uint32_t incl = c;
#pragma unroll
        for (int o2 = 1; o2 < 32; o2 <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o2);
            if (lane >= o2) incl += v;
        }
        s_offset[lane] = incl - c;
        if (lane == 31 && incl) s_base = atomicAdd(&ws.counters[0], incl);
    }
    __syncthreads();
    if (isHit) slot = s_base + s_offset[bin] + warpBase + inWarp;
    if (isHit) {
        const size_t pl = ws.plane;
        for (uint32_t k = 0; k < L.shadowsPerHit; ++k)
            store_ray(&ws.shadowQ0[size_t(k) * pl + slot], pos, (flags & SLOT_AO) || k < 2 ? shTmin : 0.0f, shDir[k], shTmax[k]);
        // (in the AO debug view both secondary rays are inactive: tmax < 0)
        store_ray(&ws.secQ[slot], pos, RT_RAY_EPSILON, secDir[0], secTmax[0]);
        store_ray(&ws.secQ[pl + slot], pos, RT_RAY_EPSILON, secDir[1], secTmax[1]);
        if (!(flags & SLOT_AO)) {
            ws.S2[slot] = s2;
            ws.S3[slot] = s3;
        }
        ws.S0[slot] = s0;
        ws.S1[slot] = s1;
        ws.slotInfo[slot] = make_uint4(p, rec, flags, 0);
    }
    warp_count_add(&rayCounts[0], inRange ? 1u : 0u);
    warp_count_add(&rayCounts[1], nSecondary);
    warp_count_add(&rayCounts[2], nShadow);
}

// ------------------------------------------------------------------------------------------------ K3 / K4 / K6
template <bool ANY, bool STATS>
__global__ void __launch_bounds__(kBlock) k_trace_queue(const void *tlas, const rt_ray *rays, const uint32_t *count, uint32_t mult,
                                                        uint32_t plane, float4 *hitA, uint32_t *hitRec, uint8_t *vis, uint32_t *status,
                                                        unsigned long long *stats) {
    const uint32_t cnt = count[0], n = cnt * mult;
    TraceAccel A = resolve_tlas(tlas, status);
    TraceCtr ctr{0, 0, 0, 0};
    uint32_t traced = 0;
    for (uint32_t li = blockIdx.x * blockDim.x + threadIdx.x; li < n; li += gridDim.x * blockDim.x) {
        const uint32_t kind = li / cnt, i = kind * plane + (li - kind * cnt);  // planar queue: kind-major
        const float4 *rp = reinterpret_cast<const float4 *>(rays + i);
        const float4 a = rp[0], b = rp[1];
        TraceHit h;
        if (b.w < 0.0f) {  // inactive slot
            if (ANY) vis[i] = 1;
            else hitA[i] = make_float4(0, 0, 0, __uint_as_float(RT_NO_HIT)), hitRec[i] = 0xffffffffu;
            continue;
        }
        if (ANY) {
            // shootShadowRay: S/RaytracingCommon.hlsli:84-96 (ray contribution 1, miss index 1)
            bool hit = trace_ray<true, STATS>(A, a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w,
                                              RT_RAY_FLAG_ACCEPT_FIRST_HIT_AND_END_SEARCH | RT_RAY_FLAG_SKIP_CLOSEST_HIT_SHADER, 0xFF, 1, 0,
                                              h, &ctr, status);
            vis[i] = hit ? 0 : 1;
        } else {
            // shootSecondaryRay: flags 0 (no culling), contribution 0
            trace_ray<false, STATS>(A, a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, 0, 0xFF, 0, 0, h, &ctr, status);
            hitA[i] = make_float4(h.t, h.u, h.v, __uint_as_float(h.prim));
            hitRec[i] = h.record;
        }
        if (STATS) traced++;
    }
    if (STATS) flush_stats(ctr, traced, stats);
}

// ------------------------------------------------------------------------------------------------ K5
// Depth-1 shade()/shadeAOV() of a secondary hit.  At depth 1 shootSecondaryRay returns 0 and shadow rays
// are still traced (MAX_SHADOW_RAY_DEPTH 2); the Phong-lobe sample is still drawn (and its 0*brdf/pdf
// term kept literally, so a zero pdf produces the same NaN as the shader).
__global__ void __launch_bounds__(kBlock, RT_SHADE1_MIN_BLOCKS) k_shade_secondary(const __grid_constant__ Launch L, WS ws, const rt_hit_record_dev *recs,
                                                            uint32_t n_recs, const float *env, uint32_t envSize,
                                                            unsigned long long *rayCounts, uint32_t *status) {
    const uint32_t cnt = ws.counters[0], n = cnt * 2;
    for (uint32_t base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
        const uint32_t lr = base + threadIdx.x;
        // planar queue: plane 0 = indirect-diffuse rays, plane 1 = Phong-lobe rays; r is the physical index
        const uint32_t kindPlane = lr >= cnt ? 1u : 0u, hitSlot = lr - kindPlane * cnt;
        const uint32_t r = lr < n ? kindPlane * ws.plane + hitSlot : 0xffffffffu;
        bool wantShadow = false;
        f3 pos = mk3(0, 0, 0), terDir = mk3(0, 0, 1);
        float terTmax = -1.0f;
        LightEval le;
        uint32_t kind = 0, rec = 0;
        f3 specTerm = mk3(0, 0, 0);
        bool useDir = true, usePoint = true;
        if (lr < n) {
            const float4 *rp = reinterpret_cast<const float4 *>(ws.secQ + r);
            const float4 a = rp[0], b = rp[1];
            if (b.w >= 0.0f) {
                const float4 hA = ws.secHitA[r];
                const f3 o = mk3(a.x, a.y, a.z), d = mk3(b.x, b.y, b.z);
                if (__float_as_uint(hA.w) == RT_NO_HIT) {
                    kind = 1;
                    f3 c = sample_env(env, envSize, d) * L.f.options.environmentStrength;
                    ws.T0[r] = make_float4(c.x, c.y, c.z, __uint_as_float(kind));
                } else {
                    kind = 2;
                    rec = ws.secRec[r];
                    if (rec >= n_recs) rec = 0, atomicOr(status, 8u);
                    const rt_hit_record_dev &R = recs[rec];
                    const f3 N = normalize3(interpolate_normal(R, __float_as_uint(hA.w), hA.y, hA.z));
                    pos = o + hA.x * d;
                    const uint32_t pix = ws.slotInfo[hitSlot].x;
                    const uint32_t x = L.x0 + pix % L.rw, y = image_row(L, pix / L.rw);
                    uint32_t seed = init_rand(x + y * L.width, L.f.cameraParams.frameCount);
                    le = eval_lights(L.f, pos, N);
                    if (!L.realtime && L.f.options.debug == 2) {
                        if (next_rand(seed) < 0.5f) usePoint = false, kind |= 16u;
                        else useDir = false, kind |= 32u;
                    }
                    f3 fres = mk3(0, 0, 0), spec = mk3(0, 0, 0);
                    if ((R.mat.type == 1 || R.mat.type == 2) && R.mat.reflectivity > 0.001f) {
                        float exponent = expf((1.0f - R.mat.roughness) * 12.0f);
                        float pdf, brdf;
                        f3 mirror = reflect3(d, N);
                        const f3 lobe = phong_lobe(seed, mirror, exponent, pdf, brdf);
                        spec = spec + mk3(0, 0, 0) * brdf / pdf;
                        fres = fresnel_schlick(d, N, mk3(R.mat.specular[0], R.mat.specular[1], R.mat.specular[2]));
                        if (L.maxDepth >= 2) {  // shootSecondaryRay at depth 1 traces instead of returning 0
                            terDir = lobe, terTmax = RT_RAY_MAX_T;
                            ws.T3[r] = make_float2(brdf, pdf);
                        }
                    }
                    // depth 1: the whole (zero or NaN) term; depth 2: the Fresnel factor, k_resolve multiplies the traced radiance in
                    specTerm = L.maxDepth >= 2 ? fres : R.mat.reflectivity * spec * fres;
                    wantShadow = true;
                }
            } else {
                ws.T0[r] = make_float4(0, 0, 0, __uint_as_float(0u));
            }
        }
        if (L.maxDepth >= 2 && lr < n) store_ray(&ws.terQ[r], pos, RT_RAY_EPSILON, terDir, terTmax);  // inactive (tmax < 0) unless a lobe ray was drawn
        warp_count_add(&rayCounts[1], terTmax >= 0.0f ? 1u : 0u);
        const uint32_t sh = warp_alloc(wantShadow, &ws.counters[1]);
        if (wantShadow) {
            store_ray(&ws.shadowQ1[sh], pos, RT_RAY_EPSILON, le.dirL, useDir ? RT_RAY_MAX_T : -1.0f);
            store_ray(&ws.shadowQ1[2 * size_t(ws.plane) + sh], pos, RT_RAY_EPSILON, le.pointL, usePoint ? le.pointDist - RT_RAY_EPSILON : -1.0f);
            ws.secShadow[r] = sh;
            ws.T0[r] = make_float4(le.dirPre.x, le.dirPre.y, le.dirPre.z, __uint_as_float(kind));
            ws.T1[r] = make_float4(le.pointPre.x, le.pointPre.y, le.pointPre.z, le.falloff);
            ws.T2[r] = make_float4(specTerm.x, specTerm.y, specTerm.z, __uint_as_float(rec));
        }
        warp_count_add(&rayCounts[2], wantShadow ? ((useDir ? 1u : 0u) + (usePoint ? 1u : 0u)) : 0u);
    }
}

// ------------------------------------------------------------------------------------------------ K5b (maxDepth == 2)
// shade() / shadeAOV() of a depth-2 hit: direct light without shadow rays (MAX_SHADOW_RAY_DEPTH 2: visibility 1), no indirect
// diffuse (currentDepth < 1 only), the lobe sample drawn and its 0 * brdf / pdf term kept literally, exactly as depth 1 does
// when the radiance depth is 1.
__global__ void __launch_bounds__(kBlock) k_shade_tertiary(const __grid_constant__ Launch L, WS ws, const rt_hit_record_dev *recs,
                                                           uint32_t n_recs, const float *env, uint32_t envSize, uint32_t *status) {
    const uint32_t cnt = ws.counters[0], n = cnt * 2;
    for (uint32_t lr = blockIdx.x * blockDim.x + threadIdx.x; lr < n; lr += gridDim.x * blockDim.x) {
        const uint32_t kindPlane = lr >= cnt ? 1u : 0u, hitSlot = lr - kindPlane * cnt;
        const uint32_t r = kindPlane * ws.plane + hitSlot;
        const float4 *rp = reinterpret_cast<const float4 *>(ws.terQ + r);
        const float4 a = rp[0], b = rp[1];
        if (b.w < 0.0f) continue;  // no lobe ray from this secondary hit
        const float4 hA = ws.terHitA[r];
        const f3 o = mk3(a.x, a.y, a.z), d = mk3(b.x, b.y, b.z);
        f3 rad;
        if (__float_as_uint(hA.w) == RT_NO_HIT) {
            rad = sample_env(env, envSize, d) * L.f.options.environmentStrength;
        } else {
            uint32_t rec = ws.terRec[r];
            if (rec >= n_recs) rec = 0, atomicOr(status, 8u);
            const rt_hit_record_dev &R = recs[rec];
            const f3 N = normalize3(interpolate_normal(R, __float_as_uint(hA.w), hA.y, hA.z));
            const f3 pos = o + hA.x * d;
            const uint32_t pix = ws.slotInfo[hitSlot].x;
            const uint32_t x = L.x0 + pix % L.rw, y = image_row(L, pix / L.rw);
            uint32_t seed = init_rand(x + y * L.width, L.f.cameraParams.frameCount);
            const LightEval le = eval_lights(L.f, pos, N);
            f3 direct = mk3(0, 0, 0);
            const f3 dirC = le.dirPre * 1.0f, pointC = le.pointPre * 1.0f * le.falloff;  // visibility 1
            if (!L.realtime && L.f.options.debug == 2) {
                if (next_rand(seed) < 0.5f) direct = direct + dirC * 2.0f;
                else direct = direct + pointC * 2.0f;
            } else {
                direct = direct + dirC;
                direct = direct + pointC;
            }
            f3 fres = mk3(0, 0, 0), spec = mk3(0, 0, 0);
            if ((R.mat.type == 1 || R.mat.type == 2) && R.mat.reflectivity > 0.001f) {
                float exponent = expf((1.0f - R.mat.roughness) * 12.0f);
                float pdf, brdf;
                (void)phong_lobe(seed, reflect3(d, N), exponent, pdf, brdf);
                spec = spec + mk3(0, 0, 0) * brdf / pdf;
                fres = fresnel_schlick(d, N, mk3(R.mat.specular[0], R.mat.specular[1], R.mat.specular[2]));
            }
            const f3 albedo = mk3(R.mat.albedo[0], R.mat.albedo[1], R.mat.albedo[2]);
            const f3 specTerm = R.mat.reflectivity * spec * fres;
            if (L.realtime) rad = albedo * direct / RT_M_PI + specTerm;
            else rad = (mk3(R.mat.emissive[0], R.mat.emissive[1], R.mat.emissive[2]) * R.mat.emissive[3] + albedo * ((direct + mk3(0, 0, 0)) / RT_M_PI)) + specTerm;
        }
        ws.terRad[r] = make_float4(rad.x, rad.y, rad.z, 1.0f);
    }
}

// ------------------------------------------------------------------------------------------------ K7
__device__ __forceinline__ f3 secondary_radiance(const Launch &L, const WS &ws, const rt_hit_record_dev *recs, uint32_t r) {
    const float4 t0 = ws.T0[r];
    const uint32_t kind = __float_as_uint(t0.w);
    if ((kind & 15u) == 0) return mk3(0, 0, 0);
    if ((kind & 15u) == 1) return mk3(t0.x, t0.y, t0.z);
    const float4 t1 = ws.T1[r];
    float4 t2 = ws.T2[r];
    if (L.maxDepth >= 2) {  // t2.xyz is the Fresnel factor: put the traced reflection in (shade(): spec += refl * brdf / pdf)
        const rt_material_params &mm = recs[__float_as_uint(t2.w)].mat;
        f3 term = mk3(0, 0, 0);
        if ((mm.type == 1 || mm.type == 2) && mm.reflectivity > 0.001f) {
            const float4 tr = ws.terRad[r];
            const float2 bp = ws.T3[r];
            f3 spec = mk3(0, 0, 0);
            spec = spec + mk3(tr.x, tr.y, tr.z) * bp.x / bp.y;
            term = mm.reflectivity * spec * mk3(t2.x, t2.y, t2.z);
        }
        t2.x = term.x, t2.y = term.y, t2.z = term.z;
    }
    const uint32_t sh = ws.secShadow[r];
    const float v0 = float(ws.vis1[sh]), v1 = float(ws.vis1[2 * size_t(ws.plane) + sh]);
    const rt_material_params &m = recs[__float_as_uint(t2.w)].mat;
    f3 direct = mk3(0, 0, 0);
    const f3 dirC = mk3(t0.x, t0.y, t0.z) * v0;
    const f3 pointC = mk3(t1.x, t1.y, t1.z) * v1 * t1.w;
    if (kind & 16u) direct = direct + dirC * 2.0f;
    else if (kind & 32u) direct = direct + pointC * 2.0f;
    else {
        direct = direct + dirC;
        direct = direct + pointC;
    }
    const f3 albedo = mk3(m.albedo[0], m.albedo[1], m.albedo[2]);
    const f3 specTerm = mk3(t2.x, t2.y, t2.z);
    if (L.realtime) return albedo * direct / RT_M_PI + specTerm;  // shadeAOV return value
    const f3 diffuseComponent = (direct + mk3(0, 0, 0)) / RT_M_PI;
    return (mk3(m.emissive[0], m.emissive[1], m.emissive[2]) * m.emissive[3] + albedo * diffuseComponent) + specTerm;
}

// AOV: also write AOVs 0-4 of every hit slot (progressive program only).  ADAPTIVE: the running means use the pixel's
// count, and every slot folds its sample into the moments and counts it.
template <bool AOV, bool ADAPTIVE>
__global__ void __launch_bounds__(kBlock, RT_RESOLVE_MIN_BLOCKS) k_resolve(const __grid_constant__ Launch L, WS ws, const rt_hit_record_dev *recs, float *out0,
                                                    uint64_t pitch0, float *out1, uint64_t pitch1, const AovOut aov, const Adaptive ad) {
    const uint32_t n = ws.counters[0];
    for (uint32_t s = blockIdx.x * blockDim.x + threadIdx.x; s < n; s += gridDim.x * blockDim.x) {
        const uint4 info = ws.slotInfo[s];
        const uint32_t x = L.x0 + info.x % L.rw, y = image_row(L, info.x / L.rw);
        const uint32_t np = ADAPTIVE ? ad.counts[image_index(L, x, y)] : L.f.cameraParams.accumCount;
        const rt_material_params &m = recs[info.y].mat;
        const uint32_t flags = info.z;
        f3 color;
        if (flags & SLOT_AO) {
            const float4 nol = ws.S0[s], pdf = ws.S1[s];
            const uint8_t *v = ws.vis0 + s;
            const size_t pl = ws.plane;
            float vis = 0.0f;
            vis += float(v[0]) * nol.x / pdf.x;
            vis += float(v[pl]) * nol.y / pdf.y;
            vis += float(v[2 * pl]) * nol.z / pdf.z;
            vis += float(v[3 * pl]) * nol.w / pdf.w;
            const float ao = vis / 4.0f;
            write_pixel(L, out0, pitch0, x, y, mk3(ao, ao, ao), true, np);
            if (ADAPTIVE) write_moments(ad, image_index(L, x, y), mk3(ao, ao, ao), np);
            continue;
        }
        const float4 s0 = ws.S0[s], s1 = ws.S1[s], s2 = ws.S2[s];
        const float v0 = float(ws.vis0[s]), v1 = float(ws.vis0[size_t(ws.plane) + s]);
        f3 direct = mk3(0, 0, 0);
        const f3 dirC = mk3(s0.x, s0.y, s0.z) * v0;
        const f3 pointC = mk3(s1.x, s1.y, s1.z) * v1 * s0.w;
        if (flags & SLOT_DEBUG2_DIR) direct = direct + dirC * 2.0f;
        else if (flags & SLOT_DEBUG2_POINT) direct = direct + pointC * 2.0f;
        else {
            direct = direct + dirC;
            direct = direct + pointC;
        }
        f3 indirect = mk3(0, 0, 0);
        if (flags & SLOT_HAS_DIFFUSE) {
            const f3 rad = secondary_radiance(L, ws, recs, s);
            f3 c = mk3(0, 0, 0);
            if (flags & SLOT_UNIFORM) {
                const float pdfU = 1.0f / (2.0f * RT_M_PI);
                c = c + rad * ws.S3[s] / pdfU;
            } else {
                c = c + rad * RT_M_PI;
            }
            indirect = indirect + c / 1.0f;
        }
        f3 spec = mk3(0, 0, 0);
        const f3 fres = mk3(s2.x, s2.y, s2.z);
        if (flags & SLOT_HAS_SPEC) {
            const f3 refl = secondary_radiance(L, ws, recs, ws.plane + s);
            spec = spec + refl * s2.w / s1.w;
        }
        const f3 albedo = mk3(m.albedo[0], m.albedo[1], m.albedo[2]);
        if (L.realtime) {
            // aov.directLighting / aov.indirectSpecular: S/RealtimeRaytracing.hlsl:95-100
            write_pixel(L, out0, pitch0, x, y, albedo * direct / RT_M_PI, false, np);
            write_pixel(L, out1, pitch1, x, y, m.reflectivity * spec * fres, false, np);
            continue;
        }
        if (AOV) {  // the expressions of the debug views below, so that each AOV equals its view bit for bit
            write_aov(L, aov, RT_AOV_DIRECT, x, y, albedo * direct / RT_M_PI, np);
            write_aov(L, aov, RT_AOV_INDIRECT_DIFFUSE, x, y, albedo * indirect / RT_M_PI, np);
            write_aov(L, aov, RT_AOV_INDIRECT_SPECULAR, x, y, m.reflectivity * spec * fres, np);
            write_aov(L, aov, RT_AOV_ALBEDO, x, y, albedo, np);
            write_aov(L, aov, RT_AOV_FRESNEL, x, y, fres, np);
        }
        const rt_debug_options &opt = L.f.options;
        const f3 diffuseComponent = (direct + indirect) / RT_M_PI;
        if (opt.showIndirectDiffuseOnly) color = albedo * indirect / RT_M_PI;
        else if (opt.showIndirectSpecularOnly) color = m.reflectivity * spec * fres;
        else if (opt.showFresnelTerm) color = fres;
        else if (opt.showGBufferAlbedoOnly) color = albedo;
        else if (opt.showDirectLightingOnly) color = albedo * direct / RT_M_PI;
        else color = (mk3(m.emissive[0], m.emissive[1], m.emissive[2]) * m.emissive[3] + albedo * diffuseComponent) + m.reflectivity * spec * fres;
        write_pixel(L, out0, pitch0, x, y, color, true, np);
        if (ADAPTIVE) write_moments(ad, image_index(L, x, y), color, np);
    }
}

// ------------------------------------------------------------------------------------------------ standalone kernels
// Traversal with the hit groups' any-hit / intersection programs and procedural primitives (SURVEY 8f-4): one thread
// per ray over the BVH2 wide nodes in the reference's visit order, so every candidate reaches the programs in the
// order the reference's traversal would present it.
template <bool ANY>
__global__ void __launch_bounds__(kBlock) k_trace_rays_hit_groups(const void *tlas, const rt_ray *rays, uint64_t n, uint32_t rayFlags,
                                                                  uint32_t mask, uint32_t rayContribution, uint32_t geomMultiplier,
                                                                  HitPrograms programs, rt_hit *hits, uint32_t *status) {
    const TraceAccel A = resolve_tlas(tlas);
    for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x) {
        const float4 *rp = reinterpret_cast<const float4 *>(rays + i);
        const float4 a = rp[0], b = rp[1];
        TraceHit h;
        trace_ray<ANY, false, true>(A, a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, rayFlags, mask, rayContribution, geomMultiplier, h, nullptr,
                                    status, programs);
        uint4 *hp = reinterpret_cast<uint4 *>(hits + i);
        hp[0] = make_uint4(__float_as_uint(h.t), __float_as_uint(h.u), __float_as_uint(h.v), h.prim);
        hp[1] = make_uint4(h.inst_index, h.geom_index, h.inst_id, h.leaf_slot);
    }
}

template <bool STATS>
__global__ void __launch_bounds__(kBlock) k_trace_rays(const void *tlas, const rt_ray *rays, uint64_t n, uint32_t rayFlags, uint32_t mask,
                                                       rt_hit *hits, unsigned long long *stats, uint32_t *status) {
    TraceAccel A = resolve_tlas(tlas, status);
    TraceCtr c{0, 0, 0, 0};
    for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x) {
        const float4 *rp = reinterpret_cast<const float4 *>(rays + i);
        const float4 a = rp[0], b = rp[1];
        TraceHit h;
        if (rayFlags & RT_RAY_FLAG_ACCEPT_FIRST_HIT_AND_END_SEARCH)
            trace_ray<true, STATS>(A, a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, rayFlags, mask, 0, 0, h, &c, status);
        else
            trace_ray<false, STATS>(A, a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, rayFlags, mask, 0, 0, h, &c, status);
        uint4 *hp = reinterpret_cast<uint4 *>(hits + i);
        hp[0] = make_uint4(__float_as_uint(h.t), __float_as_uint(h.u), __float_as_uint(h.v), h.prim);
        hp[1] = make_uint4(h.inst_index, h.geom_index, h.inst_id, h.leaf_slot);
    }
    if (STATS) {
        atomicAdd(&stats[1], (unsigned long long)c.internal);
        atomicAdd(&stats[2], (unsigned long long)c.leaf);
        atomicAdd(&stats[3], (unsigned long long)c.inst);
        atomicMax(&stats[4], (unsigned long long)c.max_stack);
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&stats[0], (unsigned long long)n);
    }
}

__global__ void __launch_bounds__(kBlock) k_primary_rays(const __grid_constant__ Launch L, rt_ray *rays) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= L.width * L.height) return;
    f3 o, d;
    primary_ray(L.f, L.width, L.height, p % L.width, p / L.width, L.jitterScale, o, d);
    store_ray(rays + p, o, 0.0f, d, RT_RAY_MAX_T);
}

__global__ void k_scale(float *buf, uint64_t n, float s) {
    for (uint64_t i = blockIdx.x * uint64_t(blockDim.x) + threadIdx.x; i < n; i += uint64_t(gridDim.x) * blockDim.x) buf[i] *= s;
}

// ------------------------------------------------------------------------------------------------ host
// `part` of `parts`: the dispatch may run as several independent pixel bands, each with its own workspace of P pixels.
// inst: the pixels' InstanceIndex() array, which exists only while the previous-position AOV is bound (nullptr otherwise).
int ensure_workspace(rt_context *ctx, uint64_t P, WS &ws, uint32_t part = 0, uint32_t parts = 1, uint32_t **inst = nullptr) {
    uint64_t o = 0;
    auto take = [&](uint64_t bytes) {
        uint64_t r = o;
        o = align_up(o + bytes, 256);
        return r;
    };
    const uint64_t oHitA = take(16 * P), oHitRec = take(4 * P), oCnt = take(256), oSlot = take(16 * P), oS0 = take(16 * P),
                   oS1 = take(16 * P), oS2 = take(16 * P), oS3 = take(4 * P), oSQ0 = take(32 * 4 * P), oV0 = take(4 * P),
                   oSec = take(32 * 2 * P), oSecH = take(16 * 2 * P), oSecR = take(4 * 2 * P), oSecS = take(4 * 2 * P),
                   oT0 = take(16 * 2 * P), oT1 = take(16 * 2 * P), oT2 = take(16 * 2 * P), oSQ1 = take(32 * 4 * P), oV1 = take(4 * P);
    // the depth-2 wave's arrays follow everything else, so the offsets above do not depend on the option
    const bool depth2 = ctx->render_options.max_radiance_ray_depth >= 2;
    const uint64_t oTerQ = take(depth2 ? 32 * 2 * P : 0), oTerH = take(depth2 ? 16 * 2 * P : 0), oTerR = take(depth2 ? 4 * 2 * P : 0),
                   oTerRad = take(depth2 ? 16 * 2 * P : 0), oT3 = take(depth2 ? 8 * 2 * P : 0);
    const bool prevPos = ctx->aov[RT_AOV_PREVIOUS_POSITION] != nullptr;
    const uint64_t oInst = take(prevPos ? 4 * P : 0);
    const uint64_t one = align_up(o, 256);
    if (ctx->ws.bytes < one * parts) {
        if (ctx->ws.base) {
            RT_CUDA(cudaStreamSynchronize(ctx->stream));  // every dispatch joins its helper streams into ctx->stream
            RT_CUDA(cudaFree(ctx->ws.base));
            ctx->ws.base = nullptr;
            ctx->ws.bytes = 0;
        }
        RT_CUDA(cudaMalloc(&ctx->ws.base, one * parts));
        ctx->ws.bytes = one * parts;
    }
    uint8_t *b = static_cast<uint8_t *>(ctx->ws.base) + one * part;
    ws.plane = uint32_t(P);
    ws.hitA = (float4 *)(b + oHitA), ws.hitRec = (uint32_t *)(b + oHitRec), ws.counters = (uint32_t *)(b + oCnt);
    ws.slotInfo = (uint4 *)(b + oSlot), ws.S0 = (float4 *)(b + oS0), ws.S1 = (float4 *)(b + oS1), ws.S2 = (float4 *)(b + oS2);
    ws.S3 = (float *)(b + oS3), ws.shadowQ0 = (rt_ray *)(b + oSQ0), ws.vis0 = b + oV0, ws.secQ = (rt_ray *)(b + oSec);
    ws.secHitA = (float4 *)(b + oSecH), ws.secRec = (uint32_t *)(b + oSecR), ws.secShadow = (uint32_t *)(b + oSecS);
    ws.T0 = (float4 *)(b + oT0), ws.T1 = (float4 *)(b + oT1), ws.T2 = (float4 *)(b + oT2), ws.shadowQ1 = (rt_ray *)(b + oSQ1);
    ws.vis1 = b + oV1;
    ws.terQ = (rt_ray *)(b + oTerQ), ws.terHitA = (float4 *)(b + oTerH), ws.terRec = (uint32_t *)(b + oTerR);
    ws.terRad = (float4 *)(b + oTerRad), ws.T3 = (float2 *)(b + oT3);
    if (inst) *inst = prevPos ? (uint32_t *)(b + oInst) : nullptr;
    return RT_OK;
}

// Persistent kernels run one wave: as many 128-thread blocks as fit on the device at once.
template <int MODE>
int pgrid(rt_context *ctx) {
    static int blocks_per_sm = 0;
    if (blocks_per_sm == 0) {
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, k_trace_persistent<MODE>, 128, 0) != cudaSuccess || blocks_per_sm < 1)
            blocks_per_sm = 4;
    }
    return ctx->num_sms * blocks_per_sm;
}

int upload_records(rt_program *prog) {
    if (!prog->dirty) return RT_OK;
    rt_context *ctx = prog->ctx;
    // RtBindings holds one record per (instance, ray type) (libs/DXRFramework/RtBindings.cpp:131-164): a hole inside the
    // bound range would be shaded through null vertex / index buffers
    for (uint32_t i = 0; i < prog->n_recs; ++i)
        RT_REQUIRE(prog->host_recs[i].vb != nullptr && prog->host_recs[i].ib != nullptr,
                   "unbound hit record inside the bound range (every instance needs a record for every ray type)");
    if (prog->n_recs) {
        RT_CUDA(cudaMemcpyAsync(prog->dev_recs, prog->host_recs, sizeof(rt_hit_record_dev) * prog->n_recs, cudaMemcpyHostToDevice, ctx->stream));
        // host_recs is pageable: the copy is staged before the call returns, so later edits are safe
    }
    prog->dirty = false;
    return RT_OK;
}

}  // namespace

extern "C" {

static int dispatch_band(rt_context *ctx, rt_program *prog, const Launch &L, const WS &ws, uint32_t *inst, cudaStream_t st,
                         cudaStream_t side, cudaEvent_t ev_fork, cudaEvent_t ev_join);

static int dispatch_impl(rt_context *ctx, rt_program *prog, uint32_t width, uint32_t height, uint32_t x0, uint32_t y0, uint32_t x1,
                         uint32_t y1, uint32_t stripShift, uint32_t stripGroups, uint32_t stripGroup) {
    RT_REQUIRE(ctx && prog && prog->ctx == ctx, "context/program");
    RT_REQUIRE(ctx->tlas != nullptr, "no TLAS bound (rt_set_tlas)");
    RT_REQUIRE(ctx->output[0] != nullptr, "no output bound to slot 0 (rt_set_output)");
    RT_REQUIRE(prog->kind != RT_PROGRAM_REALTIME || ctx->output[1] != nullptr, "realtime program needs output slot 1");
    RT_REQUIRE(x0 < x1 && y0 < y1 && x1 <= width && y1 <= height, "pixel rectangle");
    RT_REQUIRE(ctx->pitch[0] >= uint64_t(width) * 16, "output pitch");
    RT_REQUIRE(prog->kind != RT_PROGRAM_REALTIME || ctx->pitch[1] >= uint64_t(width) * 16, "output pitch of slot 1");
    RT_REQUIRE(prog->n_recs > 0, "no hit records bound (rt_bindings_set_hit_record)");
    bool anyAov = false;
    for (uint32_t k = 0; k < RT_AOV_COUNT; ++k) {
        if (!ctx->aov[k]) continue;
        anyAov = true;
        RT_REQUIRE(ctx->aov_pitch[k] >= uint64_t(width) * 16, "AOV output pitch");
    }
    RT_REQUIRE(!anyAov || prog->kind != RT_PROGRAM_REALTIME, "AOV outputs bound for a realtime program (its outputs already are AOVs)");
    RT_REQUIRE(!anyAov || !ctx->frame.options.showAmbientOcclusionOnly, "AOV outputs bound in the ambient-occlusion debug view");
    RT_REQUIRE(!ctx->adaptive_counts || prog->kind != RT_PROGRAM_REALTIME, "adaptive sampling bound for a realtime program");
    RT_CUDA(cudaSetDevice(ctx->device));
    const bool realtime = prog->kind == RT_PROGRAM_REALTIME;
    // RayGen early-out: S/ProgressiveRaytracing.hlsl:13-15
    if (!realtime && ctx->frame.cameraParams.accumCount >= ctx->frame.options.maxIterations) return RT_OK;

    Launch L;
    L.f = ctx->frame;
    L.width = width, L.height = height;
    L.x0 = x0, L.y0 = y0, L.rw = x1 - x0, L.rh = y1 - y0;
    L.v0 = 0, L.stripShift = stripShift, L.stripGroups = stripGroups, L.stripGroup = stripGroup;
    L.jitterScale = realtime ? 10.0f : 30.0f;  // S/ProgressiveRaytracing.hlsl:26, S/RealtimeRaytracing.hlsl:34
    L.realtime = realtime ? 1u : 0u;
    L.shadowsPerHit = (!realtime && L.f.options.showAmbientOcclusionOnly) ? 4u : 2u;
    L.maxDepth = ctx->render_options.max_radiance_ray_depth;
    L.halfTargets = ctx->render_options.half_render_targets;
    int rc = upload_records(prog);
    if (rc) return rc;
    const bool timing = ctx->timing;
    if (timing && !ctx->ev_ready) {
        for (auto &e : ctx->ev) RT_CUDA(cudaEventCreate(&e));
        ctx->ev_ready = true;
    }
    // Pixel bands, each a complete wavefront pipeline on its own stream (forked from and joined back into the
    // context's stream, so the call stays stream-ordered for the caller): whenever one band's kernel runs out of rays —
    // persistent kernels end with 8-20 % of their warps idle, k_primary leaves ~30 % of its warp slots unused — blocks of
    // the other band's kernels move in.  Bands touch disjoint pixels, so the image is bit-identical to the one-band run.
    // Instrumented and stage-timed dispatches, and small regions, run as one band.
    static const uint32_t band_limit = [] {  // RT_BANDS=1: one band per dispatch, for whole-frame kernel profiles (ncu); default RT_DISPATCH_BANDS
        const char *e = getenv("RT_BANDS");
        const int v = e ? atoi(e) : 0;
        return uint32_t(v >= 1 && v <= RT_MAX_BANDS ? v : RT_DISPATCH_BANDS);
    }();
    const uint32_t bands = (!timing && !ctx->collect_stats && !ctx->capture && uint64_t(L.rw) * L.rh >= (1u << 18)) ? std::min<uint32_t>(band_limit, L.rh / 64) : 1u;
    if (bands > 1) {
        if (!ctx->side_stream) {
            RT_CUDA(cudaStreamCreateWithFlags(&ctx->side_stream, cudaStreamNonBlocking));
            RT_CUDA(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
            RT_CUDA(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
        }
        if (!ctx->ev_band_fork) RT_CUDA(cudaEventCreateWithFlags(&ctx->ev_band_fork, cudaEventDisableTiming));
        for (uint32_t k = 1; k < bands; ++k) {
            if (ctx->band_streams[k][0]) continue;
            for (auto &q : ctx->band_streams[k]) RT_CUDA(cudaStreamCreateWithFlags(&q, cudaStreamNonBlocking));
            for (auto &e : ctx->band_events[k]) RT_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        }
        // band boundaries on tile rows
        uint32_t y[RT_MAX_BANDS + 1];
        for (uint32_t k = 0; k <= bands; ++k) y[k] = k == bands ? L.rh : uint32_t((uint64_t(L.rh) * k / bands + 3) / 4 * 4);
        uint64_t Pmax = 0;
        for (uint32_t k = 0; k < bands; ++k) Pmax = std::max<uint64_t>(Pmax, uint64_t(L.rw) * (y[k + 1] - y[k]));
        RT_CUDA(cudaEventRecord(ctx->ev_band_fork, ctx->stream));
        for (uint32_t k = 0; k < bands; ++k) {
            Launch Lk = L;
            Lk.v0 = y[k], Lk.rh = y[k + 1] - y[k];
            WS wk;
            uint32_t *inst;
            rc = ensure_workspace(ctx, Pmax, wk, k, bands, &inst);
            if (rc) return rc;
            if (k == 0) {
                rc = dispatch_band(ctx, prog, Lk, wk, inst, ctx->stream, ctx->side_stream, ctx->ev_fork, ctx->ev_join);
            } else {
                RT_CUDA(cudaStreamWaitEvent(ctx->band_streams[k][0], ctx->ev_band_fork, 0));
                rc = dispatch_band(ctx, prog, Lk, wk, inst, ctx->band_streams[k][0], ctx->band_streams[k][1], ctx->band_events[k][0],
                                   ctx->band_events[k][1]);
                if (rc == RT_OK) RT_CUDA(cudaEventRecord(ctx->band_events[k][2], ctx->band_streams[k][0]));
            }
            if (rc) return rc;
        }
        for (uint32_t k = 1; k < bands; ++k) RT_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->band_events[k][2], 0));
        return RT_OK;
    }
    const uint64_t P = uint64_t(L.rw) * L.rh;
    WS ws;
    uint32_t *inst;
    rc = ensure_workspace(ctx, P, ws, 0, 1, &inst);
    if (rc) return rc;
    if (ctx->capture) ctx->dbg_pixels = P;
    if (!timing && !ctx->collect_stats && !ctx->side_stream) {
        RT_CUDA(cudaStreamCreateWithFlags(&ctx->side_stream, cudaStreamNonBlocking));
        RT_CUDA(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
        RT_CUDA(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
    }
    return dispatch_band(ctx, prog, L, ws, inst, ctx->stream, ctx->side_stream, ctx->ev_fork, ctx->ev_join);
}

// One band of a dispatch: the seven wavefront stages on `st`, the depth-0 shadow wave on `side`.  inst: the band's
// InstanceIndex() array when the previous-position AOV is bound, else nullptr.
static int dispatch_band(rt_context *ctx, rt_program *prog, const Launch &L, const WS &ws, uint32_t *inst, cudaStream_t st,
                         cudaStream_t side, cudaEvent_t ev_fork, cudaEvent_t ev_join) {
    const bool timing = ctx->timing;
    RT_CUDA(cudaMemsetAsync(ws.counters, 0, 256, st));
    const uint32_t tiles = ((L.rw + 7) / 8) * ((L.rh + 3) / 4);
    const int qgrid = ctx->num_sms * 16;
    if (timing) RT_CUDA(cudaEventRecord(ctx->ev[0], st));
    unsigned long long *sPrim = ctx->ray_counts + 8, *sSec = ctx->ray_counts + 16, *sShadow = ctx->ray_counts + 24;
    const bool stats = ctx->collect_stats;
    const uint32_t primBlocks = rt_div_up(tiles, kBlock / 32);
    const Adaptive ad{ctx->adaptive_counts, reinterpret_cast<float2 *>(ctx->adaptive_moments)};
    const bool adaptive = ad.counts != nullptr;
    // one kernel of each family per (stats, inst, adaptive) combination: pick it once, launch it with the same arguments
    void (*prim)(Launch, const void *, WS, uint32_t *, unsigned long long *, const uint32_t *) = k_primary<false, false>;
    void (*primInst)(Launch, const void *, WS, uint32_t *, unsigned long long *, uint32_t *, const uint32_t *) = k_primary_inst<false, false>;
    if (adaptive) prim = stats ? k_primary<true, true> : k_primary<false, true>, primInst = stats ? k_primary_inst<true, true> : k_primary_inst<false, true>;
    else if (stats) prim = k_primary<true, false>, primInst = k_primary_inst<true, false>;
    if (inst) primInst<<<primBlocks, kBlock, 0, st>>>(L, ctx->tlas, ws, ctx->status, sPrim, inst, ad.counts);
    else prim<<<primBlocks, kBlock, 0, st>>>(L, ctx->tlas, ws, ctx->status, sPrim, ad.counts);
    if (timing) RT_CUDA(cudaEventRecord(ctx->ev[1], st));
    const uint32_t shadeTiles = ((L.rw + kShadeTile - 1) / kShadeTile) * ((L.rh + kShadeTile - 1) / kShadeTile);
    AovOut aov{};
    for (int k = 0; k < RT_AOV_COUNT; ++k) {
        aov.ptr[k] = ctx->aov[k], aov.pitch[k] = ctx->aov_pitch[k];
        if (ctx->aov[k]) aov.mask |= 1u << k;
    }
    aov.n_motion = ctx->n_motion;
    aov.motion = reinterpret_cast<const float4 *>(ctx->motion);
    aov.inst = inst;
    aov.deform = ctx->deform;
    aov.n_deform = ctx->n_deform;
    auto shade0 = aov.mask ? (adaptive ? k_shade_primary<true, true> : k_shade_primary<true, false>)
                           : (adaptive ? k_shade_primary<false, true> : k_shade_primary<false, false>);
    shade0<<<shadeTiles, kShadeThreads, 0, st>>>(L, ws, prog->dev_recs, prog->n_recs, prog->env_texels, prog->env_size, ctx->output[0], ctx->pitch[0],
                                                 ctx->output[1], ctx->pitch[1], ctx->ray_counts, ctx->status, aov, ad);
    if (timing) RT_CUDA(cudaEventRecord(ctx->ev[2], st));
    // The depth-0 shadow wave and the secondary-ray chain (trace -> shade -> depth-1 shadow wave) both depend only on
    // k_shade_primary and meet again in k_resolve.  Outside the instrumented / per-stage-timed modes the shadow wave
    // runs on a side stream: its persistent blocks move in as the other kernels' blocks drain, so the tails of the
    // trace kernels (8-20 % of each launch with warps running out of rays, ncu sm__warps_active) overlap.
    const bool overlap = !timing && !stats && side != nullptr;
    if (overlap) {
        RT_CUDA(cudaEventRecord(ev_fork, st));
        RT_CUDA(cudaStreamWaitEvent(side, ev_fork, 0));
    }
    if (stats) k_trace_queue<false, true><<<qgrid, kBlock, 0, st>>>(ctx->tlas, ws.secQ, ws.counters, 2, ws.plane, ws.secHitA, ws.secRec, nullptr, ctx->status, sSec);
    else k_trace_persistent<0><<<pgrid<0>(ctx), 128, 0, st>>>(ctx->tlas, ws.secQ, ws.counters, 2, ws.plane, TraceSink{ws.secHitA, ws.secRec, nullptr, nullptr}, ctx->status, ws.counters + 4, 0, 0xFF);
    if (timing) RT_CUDA(cudaEventRecord(ctx->ev[3], st));
    {
        cudaStream_t s0 = overlap ? side : st;
        if (stats) k_trace_queue<true, true><<<qgrid, kBlock, 0, s0>>>(ctx->tlas, ws.shadowQ0, ws.counters, L.shadowsPerHit, ws.plane, nullptr, nullptr, ws.vis0, ctx->status, sShadow);
        else k_trace_persistent<1><<<pgrid<1>(ctx), 128, 0, s0>>>(ctx->tlas, ws.shadowQ0, ws.counters, L.shadowsPerHit, ws.plane, TraceSink{nullptr, nullptr, ws.vis0, nullptr}, ctx->status, ws.counters + 5, 0, 0xFF);
        if (overlap) RT_CUDA(cudaEventRecord(ev_join, side));
    }
    if (timing) RT_CUDA(cudaEventRecord(ctx->ev[4], st));
    k_shade_secondary<<<qgrid, kBlock, 0, st>>>(L, ws, prog->dev_recs, prog->n_recs, prog->env_texels, prog->env_size, ctx->ray_counts, ctx->status);
    if (timing) RT_CUDA(cudaEventRecord(ctx->ev[5], st));
    if (stats) k_trace_queue<true, true><<<qgrid, kBlock, 0, st>>>(ctx->tlas, ws.shadowQ1, ws.counters + 1, 2, 2 * ws.plane, nullptr, nullptr, ws.vis1, ctx->status, sShadow);
    else k_trace_persistent<1><<<pgrid<1>(ctx), 128, 0, st>>>(ctx->tlas, ws.shadowQ1, ws.counters + 1, 2, 2 * ws.plane, TraceSink{nullptr, nullptr, ws.vis1, nullptr}, ctx->status, ws.counters + 6, 0, 0xFF);
    if (timing) RT_CUDA(cudaEventRecord(ctx->ev[6], st));
    if (L.maxDepth >= 2) {
        // depth-2 wave: the Phong-lobe rays of the secondary hits (incoherent closest-hit rays, counted as secondary rays)
        if (stats) k_trace_queue<false, true><<<qgrid, kBlock, 0, st>>>(ctx->tlas, ws.terQ, ws.counters, 2, ws.plane, ws.terHitA, ws.terRec, nullptr, ctx->status, sSec);
        else k_trace_persistent<0><<<pgrid<0>(ctx), 128, 0, st>>>(ctx->tlas, ws.terQ, ws.counters, 2, ws.plane, TraceSink{ws.terHitA, ws.terRec, nullptr, nullptr}, ctx->status, ws.counters + 7, 0, 0xFF);
        if (timing) RT_CUDA(cudaEventRecord(ctx->ev[7], st));
        k_shade_tertiary<<<qgrid, kBlock, 0, st>>>(L, ws, prog->dev_recs, prog->n_recs, prog->env_texels, prog->env_size, ctx->status);
        ctx->launches += 2;
    }
    if (overlap) RT_CUDA(cudaStreamWaitEvent(st, ev_join, 0));
    auto resolve = aov.mask ? (adaptive ? k_resolve<true, true> : k_resolve<true, false>) : (adaptive ? k_resolve<false, true> : k_resolve<false, false>);
    resolve<<<qgrid, kBlock, 0, st>>>(L, ws, prog->dev_recs, ctx->output[0], ctx->pitch[0], ctx->output[1], ctx->pitch[1], aov, ad);
    ctx->launches += 7;
    RT_LAUNCH_CHECK();
    if (timing) {
        RT_CUDA(cudaEventSynchronize(ctx->ev[6]));
        float ms = 0;
        RT_CUDA(cudaEventElapsedTime(&ms, ctx->ev[0], ctx->ev[1]));
        ctx->t_primary += ms;
        RT_CUDA(cudaEventElapsedTime(&ms, ctx->ev[2], ctx->ev[3]));
        ctx->t_secondary += ms;
        RT_CUDA(cudaEventElapsedTime(&ms, ctx->ev[3], ctx->ev[4]));
        ctx->t_shadow += ms;
        RT_CUDA(cudaEventElapsedTime(&ms, ctx->ev[5], ctx->ev[6]));
        ctx->t_shadow += ms;
        if (L.maxDepth >= 2) {
            RT_CUDA(cudaEventSynchronize(ctx->ev[7]));
            RT_CUDA(cudaEventElapsedTime(&ms, ctx->ev[6], ctx->ev[7]));
            ctx->t_secondary += ms;
        }
    }
    return RT_OK;
}

int rt_dispatch_rays_region(rt_context *ctx, rt_program *prog, uint32_t width, uint32_t height, uint32_t x0, uint32_t y0, uint32_t x1,
                            uint32_t y1) {
    return dispatch_impl(ctx, prog, width, height, x0, y0, x1, y1, 0, 1, 0);
}

int rt_dispatch_rays_interleaved(rt_context *ctx, rt_program *prog, uint32_t width, uint32_t height, uint32_t strip_rows, uint32_t groups,
                                 uint32_t group) {
    RT_REQUIRE(groups >= 1 && group < groups, "strip group");
    RT_REQUIRE(strip_rows >= 4 && (strip_rows & (strip_rows - 1)) == 0, "strip_rows must be a power of two >= 4");
    if (groups == 1) return dispatch_impl(ctx, prog, width, height, 0, 0, width, height, 0, 1, 0);
    uint32_t shift = 0;
    while ((1u << shift) < strip_rows) ++shift;
    // rows of this group: whole strips group, group + groups, ... plus the part of the last strip inside the image
    const uint32_t strips = (height + strip_rows - 1) / strip_rows;
    uint32_t rows = 0;
    for (uint32_t k = group; k < strips; k += groups) rows += std::min(strip_rows, height - k * strip_rows);
    if (rows == 0) return RT_OK;  // more groups than strips: nothing to render for this one
    return dispatch_impl(ctx, prog, width, height, 0, 0, width, rows, shift, groups, group);
}

int rt_dispatch_rays(rt_context *ctx, rt_program *prog, uint32_t width, uint32_t height, uint32_t /*depth*/) {
    // Depth is ignored exactly as the compute fallback does (FL/UberShaderRayTracingProgram.cpp:268-272).
    return rt_dispatch_rays_region(ctx, prog, width, height, 0, 0, width, height);
}

static int trace_common(rt_context *ctx, const void *tlas, const rt_ray *rays, uint64_t n, uint32_t flags, uint32_t mask, rt_hit *hits,
                        rt_trace_stats *stats) {
    RT_REQUIRE(ctx && tlas && (n == 0 || (rays && hits)), "null argument");
    RT_CUDA(cudaSetDevice(ctx->device));
    if (n == 0) return RT_OK;
    if (stats) {
        // instrumented: the one-thread-one-ray BVH2 loop in the reference's visit order (its counters are the roofline's n_int / n_leaf)
        const int grid = int(std::min<uint64_t>(rt_div_up(n, kBlock), uint64_t(ctx->num_sms) * 16));
        k_trace_rays<true><<<grid, kBlock, 0, ctx->stream>>>(tlas, rays, n, flags, mask, hits, reinterpret_cast<unsigned long long *>(stats), ctx->status);
        ctx->launches++;
    } else {
        // production traversal (persistent warps over the 4-wide nodes), in chunks of < 2^31 rays
        uint32_t *counter = ctx->status + 16;
        for (uint64_t done = 0; done < n;) {
            const uint32_t chunk = uint32_t(std::min<uint64_t>(n - done, 1u << 30));
            RT_CUDA(cudaMemsetAsync(counter, 0, 4, ctx->stream));
            k_trace_persistent<2><<<pgrid<2>(ctx), 128, 0, ctx->stream>>>(tlas, rays + done, nullptr, chunk, 0, TraceSink{nullptr, nullptr, nullptr, hits + done},
                                                                         ctx->status, counter, flags, mask);
            ctx->launches++;
            done += chunk;
        }
    }
    RT_LAUNCH_CHECK();
    return RT_OK;
}

int rt_trace_rays_hit_groups(rt_context *ctx, const void *tlas, const rt_ray *rays, uint64_t n, uint32_t flags, uint32_t mask,
                             uint32_t ray_contribution, uint32_t geometry_multiplier, const rt_hit_group_programs *programs,
                             uint32_t n_programs, rt_hit *hits) {
    RT_REQUIRE(ctx && tlas && (n == 0 || (rays && hits)), "null argument");
    RT_REQUIRE(n_programs == 0 || programs != nullptr, "null hit-group program table");
    RT_REQUIRE(n_programs <= 4096, "more than 4096 hit-group records");
    for (uint32_t i = 0; i < n_programs; ++i) {
        // an unknown shader identifier is a std::logic_error in RtBindings (libs/DXRFramework/RtBindings.cpp:77-79)
        RT_REQUIRE(programs[i].any_hit < RT_ANYHIT_COUNT, "unknown any-hit program");
        RT_REQUIRE(programs[i].intersection < RT_INTERSECTION_COUNT, "unknown intersection program");
    }
    RT_CUDA(cudaSetDevice(ctx->device));
    if (n == 0) return RT_OK;
    if (n_programs) {
        if (!ctx->hit_programs) RT_CUDA(cudaMalloc(&ctx->hit_programs, 4096 * sizeof(rt_hit_group_programs)));
        // stream-ordered copy of a pageable host table: staged by the runtime before the call returns
        RT_CUDA(cudaMemcpyAsync(ctx->hit_programs, programs, n_programs * sizeof(rt_hit_group_programs), cudaMemcpyHostToDevice, ctx->stream));
    }
    const HitPrograms hp{n_programs ? ctx->hit_programs : nullptr, n_programs};
    const int grid = int(std::min<uint64_t>(rt_div_up(n, kBlock), uint64_t(ctx->num_sms) * 16));
    if (flags & RT_RAY_FLAG_ACCEPT_FIRST_HIT_AND_END_SEARCH)
        k_trace_rays_hit_groups<true><<<grid, kBlock, 0, ctx->stream>>>(tlas, rays, n, flags, mask, ray_contribution, geometry_multiplier, hp, hits, ctx->status);
    else
        k_trace_rays_hit_groups<false><<<grid, kBlock, 0, ctx->stream>>>(tlas, rays, n, flags, mask, ray_contribution, geometry_multiplier, hp, hits, ctx->status);
    ctx->launches++;
    RT_LAUNCH_CHECK();
    return RT_OK;
}

int rt_trace_rays(rt_context *ctx, const void *tlas, const rt_ray *rays, uint64_t n, uint32_t flags, uint32_t mask, rt_hit *hits) {
    return trace_common(ctx, tlas, rays, n, flags, mask, hits, nullptr);
}
int rt_trace_rays_stats(rt_context *ctx, const void *tlas, const rt_ray *rays, uint64_t n, uint32_t flags, uint32_t mask, rt_hit *hits,
                        rt_trace_stats *stats_dev) {
    RT_REQUIRE(stats_dev != nullptr, "stats");
    return trace_common(ctx, tlas, rays, n, flags, mask, hits, stats_dev);
}

int rt_generate_primary_rays(rt_context *ctx, const rt_per_frame_constants *frame, uint32_t width, uint32_t height, float jitter_scale,
                             rt_ray *rays) {
    RT_REQUIRE(ctx && frame && rays && width && height, "null argument");
    RT_CUDA(cudaSetDevice(ctx->device));
    Launch L{};
    L.f = *frame;
    L.width = width, L.height = height, L.rw = width, L.rh = height;
    L.jitterScale = jitter_scale;
    k_primary_rays<<<rt_div_up(uint64_t(width) * height, kBlock), kBlock, 0, ctx->stream>>>(L, rays);
    ctx->launches++;
    RT_LAUNCH_CHECK();
    return RT_OK;
}

// ---- parity instrumentation: the stage products of the last captured dispatch (SURVEY.md 8b "rt_trace_primary_ids")
int rt_enable_debug_capture(rt_context *ctx, int enable) {
    RT_REQUIRE(ctx != nullptr, "ctx");
    ctx->capture = enable != 0;
    if (!enable) ctx->dbg_pixels = 0;
    return RT_OK;
}

int rt_debug_counts(rt_context *ctx, uint32_t *pixels, uint32_t *hit_slots, uint32_t *shadow1_pairs) {
    RT_REQUIRE(ctx && ctx->dbg_pixels > 0, "no captured dispatch (rt_enable_debug_capture, then dispatch)");
    RT_CUDA(cudaSetDevice(ctx->device));
    WS ws;
    int rc = ensure_workspace(ctx, ctx->dbg_pixels, ws);
    if (rc) return rc;
    uint32_t c[2] = {0, 0};
    RT_CUDA(cudaMemcpyAsync(c, ws.counters, 8, cudaMemcpyDeviceToHost, ctx->stream));
    RT_CUDA(cudaStreamSynchronize(ctx->stream));
    if (pixels) *pixels = uint32_t(ctx->dbg_pixels);
    if (hit_slots) *hit_slots = c[0];
    if (shadow1_pairs) *shadow1_pairs = c[1];
    return RT_OK;
}

int rt_debug_download(rt_context *ctx, int array, uint32_t plane, void *host, uint64_t host_bytes) {
    RT_REQUIRE(ctx && host, "null argument");
    uint32_t P = 0, slots = 0, pairs = 0;
    int rc = rt_debug_counts(ctx, &P, &slots, &pairs);
    if (rc) return rc;
    WS ws;
    rc = ensure_workspace(ctx, P, ws);
    if (rc) return rc;
    const uint8_t *src = nullptr;
    uint64_t elem = 0, count = 0, max_plane = 1;
    switch (array) {
        case RT_DEBUG_PRIMARY_HITS: src = (const uint8_t *)ws.hitA, elem = 16, count = P; break;
        case RT_DEBUG_PRIMARY_RECORDS: src = (const uint8_t *)ws.hitRec, elem = 4, count = P; break;
        case RT_DEBUG_SLOT_INFO: src = (const uint8_t *)ws.slotInfo, elem = 16, count = slots; break;
        case RT_DEBUG_SECONDARY_RAYS: src = (const uint8_t *)(ws.secQ + size_t(plane) * ws.plane), elem = 32, count = slots, max_plane = 2; break;
        case RT_DEBUG_SECONDARY_HITS: src = (const uint8_t *)(ws.secHitA + size_t(plane) * ws.plane), elem = 16, count = slots, max_plane = 2; break;
        case RT_DEBUG_SECONDARY_RECORDS: src = (const uint8_t *)(ws.secRec + size_t(plane) * ws.plane), elem = 4, count = slots, max_plane = 2; break;
        case RT_DEBUG_SHADOW0_RAYS: src = (const uint8_t *)(ws.shadowQ0 + size_t(plane) * ws.plane), elem = 32, count = slots, max_plane = 4; break;
        case RT_DEBUG_SHADOW0_VISIBILITY: src = ws.vis0 + size_t(plane) * ws.plane, elem = 1, count = slots, max_plane = 4; break;
        case RT_DEBUG_SHADOW1_RAYS: src = (const uint8_t *)(ws.shadowQ1 + size_t(plane) * 2 * ws.plane), elem = 32, count = pairs, max_plane = 2; break;
        case RT_DEBUG_SHADOW1_VISIBILITY: src = ws.vis1 + size_t(plane) * 2 * ws.plane, elem = 1, count = pairs, max_plane = 2; break;
        default: RT_REQUIRE(false, "unknown debug array");
    }
    RT_REQUIRE(plane < max_plane, "plane");
    RT_REQUIRE(host_bytes >= elem * count, "host buffer too small (rt_debug_counts gives the element counts)");
    if (count) RT_CUDA(cudaMemcpyAsync(host, src, elem * count, cudaMemcpyDeviceToHost, ctx->stream));
    RT_CUDA(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

int rt_scale_buffer(rt_context *ctx, float *buf, uint64_t count, float scale) {
    RT_REQUIRE(ctx && (buf || count == 0), "null argument");
    RT_CUDA(cudaSetDevice(ctx->device));
    if (count == 0) return RT_OK;
    k_scale<<<ctx->num_sms * 8, 256, 0, ctx->stream>>>(buf, count, scale);
    ctx->launches++;
    RT_LAUNCH_CHECK();
    return RT_OK;
}

}  // extern "C"
