// trace_persistent.cuh — persistent-warp traversal with dynamic ray replacement over 4-wide nodes.
//
// The plain one-thread-one-ray loop (trace.cuh) runs incoherent rays at ~5 of 32 lanes active: rays in a warp
// finish after wildly different numbers of node visits and the warp waits for its longest ray
// (profiles/r1_ncu_trace_baseline.md).  This kernel computes the same hits (same box and triangle arithmetic, same
// acceptance rule t < tCommitted && t > tMin) but schedules the work differently:
//   * persistent warps pull rays from a global counter; when at least kFetchThreshold lanes are idle the warp
//     refills exactly those lanes (Aila & Laine's "dynamic fetch", warp-synchronous via __ballot_sync);
//   * internal-node steps and leaf steps are separate warp-wide phases: a lane that reaches a leaf parks until
//     kLeafThreshold lanes hold one (or nobody can advance), so the triangle test never runs for 1-2 lanes;
//   * an internal step reads ONE 128-byte rt_wide4_node (four 32-byte loads) and tests four boxes, i.e. two BVH2
//     levels per dependent memory round trip — the kernel was latency-bound on the chain of node fetches
//     (profiles/r1_ncu_trace_persistent.md); hits are ordered near-to-far with a 5-exchange network on integer keys;
//   * the ray constants are only recomputed when the instance transform actually changes them.
// MODE 0: closest hit, ray flags 0 (secondary rays of the pipelines)  -> compact hit records
// MODE 1: any hit (shadow rays: ACCEPT_FIRST_HIT | SKIP_CLOSEST_HIT)   -> visibility bytes
// MODE 2: caller-supplied ray flags / instance mask, full rt_hit records (rt_trace_rays)
#pragma once
#include "trace.cuh"

#ifndef RT_FETCH_THRESHOLD
#define RT_FETCH_THRESHOLD 24
#endif
#ifndef RT_LEAF_THRESHOLD
#define RT_LEAF_THRESHOLD 2  // re-tuned once the triangle test lost its branches (pick()): 4 -> 2 is +0 / +3 / +4 % on incoherent rays over
                             // 82 k / 1.3 M / 5.2 M triangles and +0.5 / +3 / +5 % on shadow rays; 1 and 3 are worse
#endif
#ifndef RT_INT_UNROLL
#define RT_INT_UNROLL 2  // internal-node steps per phase selection (A/B on C2 / C1M: 2 = +3.8 / +4.4 % on incoherent rays, +5.3 / +2.9 % on shadow rays; 3 and 4 lose again)
#endif
constexpr int kFetchThreshold = RT_FETCH_THRESHOLD;  // refill when >= this many lanes are idle
constexpr int kLeafThreshold = RT_LEAF_THRESHOLD;    // run a leaf phase when >= this many lanes hold a leaf

// A ray whose origin and direction hold no -0 and no Inf/NaN maps to ITSELF, bit for bit, under an identity
// world->object transform (x*1 + y*0 + z*0 (+0) == x), so its world-space constants stay valid inside the BLAS.
__device__ __forceinline__ bool plain_float(float x) {
    const uint32_t b = __float_as_uint(x);
    return b != 0x80000000u && (b & 0x7f800000u) != 0x7f800000u;
}

struct TraceSink {  // where results go; only the members of the kernel's MODE are used
    float4 *hitA;       // MODE 0: t, u, v, primitive
    uint32_t *hitRec;   // MODE 0: hit-group record index
    uint8_t *vis;       // MODE 1: 1 = unoccluded
    rt_hit *hits;       // MODE 2
};

#ifndef RT_PERSIST_MIN_BLOCKS
#define RT_PERSIST_MIN_BLOCKS 8
#endif
constexpr int kPersistThreads = 128;

// Stack policy of wide4_step (trace.cuh) for the persistent lanes.  It stays in local memory: the kernel is
// issue-bound, and local memory is L1-resident on-chip SRAM already (profiles/r2_trace_ab.md).
struct PersistStack {
    uint32_t lm[RT_STACK_SIZE];
    __device__ __forceinline__ void push(int &sp, uint32_t r, uint32_t) { lm[sp++] = r; }
    __device__ __forceinline__ uint32_t at(int sp) const { return lm[sp]; }
    __device__ __forceinline__ bool room(int sp, int n) const { return sp + n <= RT_STACK_SIZE; }
};

template <int MODE>
__global__ void __launch_bounds__(kPersistThreads, RT_PERSIST_MIN_BLOCKS)
k_trace_persistent(const void *tlas, const rt_ray *rays, const uint32_t *count, uint32_t mult, uint32_t plane, TraceSink sink,
                   uint32_t *status, uint32_t *nextRay, uint32_t userFlags, uint32_t userMask) {
    constexpr bool GENERAL = MODE == 2;
    // Pipeline queues are planar (pipeline.cu): `mult` kinds of `count[0]` rays each, kind k starting at k * plane.
    // Rays are drawn kind-major, so a warp holds one kind.  Standalone launches pass the ray count in `mult`.
    const uint32_t cnt = count ? count[0] : 0u;
    const uint32_t n = count ? cnt * mult : mult;
    const TraceAccel A = resolve_tlas(tlas, status);
    const int lane = threadIdx.x & 31;
    const unsigned ltMask = (1u << lane) - 1u;
    constexpr unsigned FULL = 0xffffffffu;
    const uint32_t rayFlags = GENERAL ? userFlags
                                      : (MODE == 1 ? (RT_RAY_FLAG_ACCEPT_FIRST_HIT_AND_END_SEARCH | RT_RAY_FLAG_SKIP_CLOSEST_HIT_SHADER) : 0u);
    const bool ANY = GENERAL ? (userFlags & RT_RAY_FLAG_ACCEPT_FIRST_HIT_AND_END_SEARCH) != 0 : (MODE == 1);
    const uint32_t instMask = GENERAL ? userMask : 0xFFu;  // InstanceInclusionMask is 0xFF for every ray of the pipelines
    constexpr uint32_t rayContribution = MODE == 1 ? 1u : 0u;  // shadow rays use hit group 1 (S/RaytracingCommon.hlsli:94)

    PersistStack stk;
    // per-lane ray state
    bool alive = false;
    uint32_t rayIdx = 0, ref = RT_SENTINEL;
    int sp = 0, blasBase = -1;
    bool bottom = false;
    bool plain = false;      // the world ray holds no -0 / Inf / NaN component
    bool sameSpace = false;  // inside a BLAS whose instance transform left the ray constants untouched
    float wox = 0, woy = 0, woz = 0, wdx = 0, wdy = 0, wdz = 1, tmin = 0, tCur = 0;
    RayPre cur;
    cur.ox = cur.oy = cur.oz = cur.ix = cur.iy = cur.iz = cur.oix = cur.oiy = cur.oiz = cur.sx = cur.sy = cur.sz = 0;
    cur.kx = 0, cur.ky = 1, cur.kz = 2;
    const rt_wide4_node *const topNodes = A.wide4;
    const rt_wide4_node *nodes = topNodes;
    const rt_packed_tri *tris = nullptr;
    uint32_t instFlags = 0, instOffset = 0;
    int cull = 0;
    float hu = 0, hv = 0;
    uint32_t hprim = RT_NO_HIT, hrec = 0;
    // MODE 2 only: identity of the instance being traversed and of the committed hit
    uint32_t instIndex = 0, instId = 0, hInst = 0, hGeom = 0, hId = 0, hSlot = 0;
    bool noMore = (A.count == 0 && n == 0);

    auto finish = [&]() {  // write the result of a finished ray
        if (MODE == 1) {
            sink.vis[rayIdx] = (hprim != RT_NO_HIT) ? 0 : 1;
        } else if (MODE == 0) {
            sink.hitA[rayIdx] = make_float4(tCur, hu, hv, __uint_as_float(hprim));
            sink.hitRec[rayIdx] = hrec;
        } else {
            uint4 *hp = reinterpret_cast<uint4 *>(sink.hits + rayIdx);
            hp[0] = make_uint4(__float_as_uint(tCur), __float_as_uint(hu), __float_as_uint(hv), hprim);
            hp[1] = make_uint4(hInst, hGeom, hId, hSlot);
        }
        alive = false;
    };

    auto pop = [&]() {  // a lane whose subtree is exhausted takes the next node from its stack (or finishes)
        if (alive && ref == RT_SENTINEL) {
            if (sp == 0) {
                finish();
            } else {
                if (bottom && sp == blasBase) {  // leaving the BLAS: back to the world-space ray (boxes only up there)
                    bottom = false;
                    if (!sameSpace) ray_pre_box<true>(cur, wox, woy, woz, wdx, wdy, wdz);
                    nodes = topNodes;
                    blasBase = -1;
                }
                --sp;
                ref = stk.at(sp);
            }
        }
    };

    for (;;) {
        // ------------------------------------------------------------------ fetch
        const unsigned aliveMask = __ballot_sync(FULL, alive);
        const int idle = 32 - __popc(aliveMask);
        if (!noMore && (idle >= kFetchThreshold)) {
            const unsigned dead = ~aliveMask;
            const int leader = __ffs(dead) - 1;
            uint32_t base = 0;
            if (lane == leader) base = atomicAdd(nextRay, uint32_t(idle));
            base = __shfl_sync(FULL, base, leader);
            noMore = base + uint32_t(idle) >= n;
            if (!alive) {
                const uint32_t drawn = base + __popc(dead & ltMask);
                if (drawn < n) {
                    rayIdx = drawn;
                    if (!GENERAL) {
                        const uint32_t kind = drawn / cnt;
                        rayIdx = kind * plane + (drawn - kind * cnt);
                    }
                    const float4 *rp = reinterpret_cast<const float4 *>(rays + rayIdx);
                    const float4 a = __ldcs(rp), b = __ldcs(rp + 1);
                    wox = a.x, woy = a.y, woz = a.z, tmin = a.w, wdx = b.x, wdy = b.y, wdz = b.z, tCur = b.w;
                    hprim = RT_NO_HIT, hu = hv = 0.0f, hrec = 0;
                    if (GENERAL) hInst = hGeom = hId = hSlot = 0;
                    alive = true;
                    if (b.w < 0.0f || A.count == 0) {  // inactive queue slot / empty scene: a miss
                        if (MODE == 0) hrec = 0xffffffffu;
                        if (MODE == 0 && b.w < 0.0f) tCur = 0.0f;
                        finish();
                    } else {
                        ray_pre_box<true>(cur, wox, woy, woz, wdx, wdy, wdz);  // the TLAS level tests boxes only
                        plain = plain_float(wox) && plain_float(woy) && plain_float(woz) && plain_float(wdx) && plain_float(wdy) &&
                                plain_float(wdz);
                        nodes = topNodes;
                        bottom = false, sameSpace = false, blasBase = -1, sp = 0;
                        float tU;
                        if (ray_box(tU, tCur, cur, A.root_c[0], A.root_c[1], A.root_c[2], A.root_h[0], A.root_h[1], A.root_h[2]))
                            ref = A.root_ref;
                        else
                            finish();
                    }
                }
            }
            continue;  // re-evaluate occupancy (lanes that drew inactive rays refill again)
        }
        if (aliveMask == 0) {
            if (noMore) break;
            continue;
        }
        // ------------------------------------------------------------------ phase selection
        const bool atLeaf = alive && (ref & RT_NODE_LEAF_FLAG);
        const unsigned leafMask = __ballot_sync(FULL, atLeaf);
        const unsigned intMask = aliveMask & ~leafMask;
        if (intMask == 0 || __popc(leafMask) >= kLeafThreshold) {
            // ---------------------------------------------------------------- leaf phase
            if (alive && ref != RT_SENTINEL && (ref & RT_NODE_LEAF_FLAG)) {
                const uint32_t slot = ref & 0x00ffffffu;
                ref = RT_SENTINEL;
                if (!bottom) {
                    // TLAS leaf: TraverseFunction.hlsli:598-634
                    const uint4 *ip = reinterpret_cast<const uint4 *>(A.inst + slot);
                    const uint4 m3 = __ldg(ip + 3);
                    if ((m3.x >> 24) & instMask) {
                        const uint4 m4 = __ldg(ip + 4);
                        instFlags = m3.y >> 24;
                        instOffset = m3.y & 0x00ffffffu;
                        if (GENERAL) instIndex = m3.z, instId = m3.x & 0x00ffffffu;
                        cull = cull_mode(instFlags, rayFlags);
                        sameSpace = plain && (m3.y & RT_PACKED_INSTANCE_IDENTITY);
                        if (sameSpace) {
                            ray_pre_shear(cur, wdx, wdy, wdz);
                        } else {
                            const float4 r0 = __ldg(reinterpret_cast<const float4 *>(ip));
                            const float4 r1 = __ldg(reinterpret_cast<const float4 *>(ip + 1));
                            const float4 r2 = __ldg(reinterpret_cast<const float4 *>(ip + 2));
                            const float m[12] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w, r2.x, r2.y, r2.z, r2.w};
                            const f3 o2 = xform_point(m, mk3(wox, woy, woz));
                            const f3 d2 = xform_vector(m, mk3(wdx, wdy, wdz));
                            cur = make_ray_pre<true>(o2.x, o2.y, o2.z, d2.x, d2.y, d2.z);
                        }
                        nodes = reinterpret_cast<const rt_wide4_node *>(__ldg(reinterpret_cast<const unsigned long long *>(ip + 5)));
                        tris = reinterpret_cast<const rt_packed_tri *>(uintptr_t(uint64_t(m4.z) | (uint64_t(m4.w) << 32)));
                        bottom = true;
                        blasBase = sp;
                        ref = m3.w;  // BLAS root (entered without a box test, as the reference does)
                    }
                } else {
                    // BLAS leaf: TraverseFunction.hlsli:635-735
                    const float4 *tp = reinterpret_cast<const float4 *>(tris + slot);
                    const float4 p0 = __ldg(tp), p1 = __ldg(tp + 1), p2 = __ldg(tp + 2);
                    bool culled = false;
                    if (GENERAL) {  // IsOpaque() and the CULL_(NON_)OPAQUE ray flags (:119-134); the pipelines' rays carry none
                        const bool opaque = is_opaque(__float_as_uint(p2.w), instFlags, rayFlags);
                        culled = (opaque && (rayFlags & RT_RAY_FLAG_CULL_OPAQUE)) || (!opaque && (rayFlags & RT_RAY_FLAG_CULL_NON_OPAQUE));
                    }
                    float t0 = tCur, bu, bv;
                    if (!culled && ray_triangle(t0, bu, bv, cull, cur, p0, p1, p2.x) && t0 < tCur && t0 > tmin) {
                        tCur = t0, hu = bu, hv = bv;
                        hprim = __float_as_uint(p2.y);
                        hrec = rayContribution + instOffset;  // geometry multiplier is 0 in both shader libraries
                        if (GENERAL) hInst = instIndex, hId = instId, hGeom = __float_as_uint(p2.z), hSlot = slot;
                        if (ANY) finish();
                    }
                }
            }
        } else {
            // ---------------------------------------------------------------- internal phase
            // RT_INT_UNROLL > 1: a lane whose step (or the pop after it) ends at another internal node takes the next
            // step right away, before the warp re-evaluates refill and leaf phases: the phase selection (two ballots,
            // counts, branches) is ~25 warp instructions per iteration against ~120 for a step.
#pragma unroll
            for (int u = 0; u < RT_INT_UNROLL; ++u) {
                if (u > 0) pop();
                if (alive && ref != RT_SENTINEL && !(ref & RT_NODE_LEAF_FLAG)) {
                    // one 128-byte node = four child boxes (two BVH2 levels per dependent fetch)
                    ref = wide4_step<false, MODE != 1>(nodes, ref, cur, tCur, stk, sp, status);
                }
            }
        }
        // ------------------------------------------------------------------ pop
        pop();
    }
}
