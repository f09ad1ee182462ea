// trace.cuh — two-level BVH2 traversal for sm_100a (pure SIMT; B200 has no RT cores).
//
// Semantics follow Fallback_TraceRay / Traverse (externals/D3D12RaytracingFallback/src/TraverseShader.hlsli:21-73,
// TraverseFunction.hlsli:520-799): depth-first, children tested when their parent is visited, near child
// first (left on ties), closest hit committed when t < tCommitted && t > tMin, optional
// ACCEPT_FIRST_HIT_AND_END_SEARCH.  What differs is HOW:
//   * nodes carry both child boxes (64 B, four 16-byte loads) so an internal visit is one dependent fetch
//     instead of the reference's three; leaves are referenced directly from their parent, so a leaf visit
//     is three 16-byte loads of a 48-byte triangle that already holds its metadata;
//   * the near child stays in a register instead of being pushed and popped;
//   * the per-thread stack is 64 entries (the reference's 32 overflows silently on deep LBVHs).
// The ray/triangle arithmetic is written with unfused intrinsics so t and barycentrics are bit-identical to
// the CPU restatement; the ray/box test uses fused multiply-adds exactly as the restatement does.
#pragma once
#include "common.cuh"

#ifndef RT_STACK_SIZE
#define RT_STACK_SIZE 64
#endif

// One 256-bit read-only load (LDG.E.256, new with sm_100): half the load instructions of two 16-byte loads for the
// 128-byte nodes.  p must be 32-byte aligned.
__device__ __forceinline__ void ldg256(const void *p, float4 &a, float4 &b) {
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
                 : "l"(p));
}

struct TraceAccel {  // resolved view of a TLAS result buffer
    const rt_wide_node *wide;
    const rt_wide4_node *wide4;
    const rt_packed_instance *inst;
    uint32_t root_ref, count;
    float root_c[3], root_h[3];
};

struct TraceHit {
    float t, u, v;
    uint32_t prim, inst_index, geom_index, inst_id, leaf_slot, record;  // prim == RT_NO_HIT on miss
};

struct TraceCtr {
    uint32_t internal, leaf, inst, max_stack;
};

struct RayPre {  // GetRayData: TraverseFunction.hlsli:438-460
    float ox, oy, oz;
    float ix, iy, iz;     // 1/d
    float oix, oiy, oiz;  // o * (1/d)
    float sx, sy, sz;     // shear
    int kx, ky, kz;
};

// Component k of (x, y, z) as two select instructions.  Written as the nested conditional `k == 0 ? x : (k == 1 ? y : z)`
// nvcc 12.9 emits a BRANCH per pick (BSSY / ISETP / BRA / MOV / BSYNC): ncu attributed 31 % of the closest-hit kernel's warp
// instructions to the nine picks of the watertight triangle test, executed at 7-8 lanes.
__device__ __forceinline__ float pick(float x, float y, float z, int k) {
    float r;
    asm("{\n\t.reg .pred p0, p1;\n\tsetp.eq.s32 p0, %4, 0;\n\tsetp.eq.s32 p1, %4, 1;\n\tselp.f32 %0, %2, %3, p1;\n\tselp.f32 %0, %1, %0, p0;\n\t}"
        : "=f"(r)
        : "f"(x), "f"(y), "f"(z), "r"(k));
    return r;
}

// The part of GetRayData the ray/box test needs: o, 1/d, o*(1/d).
// ROBUST (production kernels): a direction component that is exactly 0 gets the finite "reciprocal" +-2^100 instead
// of +-Inf.  With Inf the reference's slab arithmetic turns into NaN (Inf - Inf) and the slab then passes for EVERY
// box, so an axis-aligned ray (cosine-hemisphere sample with u1 == 0: about one ray per 2^24) walks the whole tree —
// tens of milliseconds on one lane while the GPU waits (tools/dbg_ray.py).  With 2^100 the same fused expression
// evaluates the exact condition |c - o| <= h for that axis, which every box containing a hit point satisfies, so the
// hits are unchanged and only boxes the ray cannot touch are skipped.  The instrumented kernels keep the literal
// arithmetic, so that their visit counts stay those of the reference.
template <bool ROBUST = false>
__device__ __forceinline__ void ray_pre_box(RayPre &r, float ox, float oy, float oz, float dx, float dy, float dz) {
    r.ox = ox, r.oy = oy, r.oz = oz;
    r.ix = div_(1.0f, dx), r.iy = div_(1.0f, dy), r.iz = div_(1.0f, dz);
    if (ROBUST) {
        if (dx == 0.0f) r.ix = copysignf(0x1p100f, dx);
        if (dy == 0.0f) r.iy = copysignf(0x1p100f, dy);
        if (dz == 0.0f) r.iz = copysignf(0x1p100f, dz);
    }
    r.oix = mul_(ox, r.ix), r.oiy = mul_(oy, r.iy), r.oiz = mul_(oz, r.iz);
}

// The part only the ray/triangle test needs: dominant axis and shear constants.  Needs r.ix/iy/iz of the same
// direction: Sz = 1/d[kz] is the very quotient ray_pre_box already formed.
__device__ __forceinline__ void ray_pre_shear(RayPre &r, float dx, float dy, float dz) {
    float ax = fabsf(dx), ay = fabsf(dy), az = fabsf(dz);
    int kz = (ax > ay && ax > az) ? 0 : (ay > az ? 1 : 2);
    int kx = kz == 2 ? 0 : kz + 1, ky = kx == 2 ? 0 : kx + 1;
    float dk = pick(dx, dy, dz, kz);
    if (dk < 0.0f) {
        int t = kx;
        kx = ky;
        ky = t;
    }
    r.kx = kx, r.ky = ky, r.kz = kz;
    r.sx = div_(pick(dx, dy, dz, kx), dk);
    r.sy = div_(pick(dx, dy, dz, ky), dk);
    r.sz = pick(r.ix, r.iy, r.iz, kz);
}

template <bool ROBUST = false>
__device__ __forceinline__ RayPre make_ray_pre(float ox, float oy, float oz, float dx, float dy, float dz) {
    RayPre r;
    ray_pre_box<ROBUST>(r, ox, oy, oz, dx, dy, dz);
    ray_pre_shear(r, dx, dy, dz);
    return r;
}

// RayBoxTest: TraverseFunction.hlsli:173-191 (fused multiply-adds, as pinned in oracle_trace.cpp).
__device__ __forceinline__ bool ray_box(float &tOut, float tClosest, const RayPre &r, float cx, float cy, float cz, float hx,
                                        float hy, float hz) {
    float aix = fabsf(r.ix), aiy = fabsf(r.iy), aiz = fabsf(r.iz);
    float rx = __fmaf_rn(cx, r.ix, -r.oix), ry = __fmaf_rn(cy, r.iy, -r.oiy), rz = __fmaf_rn(cz, r.iz, -r.oiz);
    float maxx = __fmaf_rn(hx, aix, rx), maxy = __fmaf_rn(hy, aiy, ry), maxz = __fmaf_rn(hz, aiz, rz);
    float minx = __fmaf_rn(-hx, aix, rx), miny = __fmaf_rn(-hy, aiy, ry), minz = __fmaf_rn(-hz, aiz, rz);
    float tmin = fmaxf(fmaxf(minx, miny), minz);
    float tmax = fminf(fminf(maxx, maxy), maxz);
    tOut = fmaxf(tmin, 0.0f);
    return tOut < fminf(tmax, tClosest);
}

// RayTriangleIntersect: TraverseFunction.hlsli:200-282 (Woop/Benthin/Wald 2013), unfused arithmetic.
// cull: 0 none, 1 cull back-facing, 2 cull front-facing (already resolved against the instance flags).
__device__ __forceinline__ bool ray_triangle(float &hitT, float &bu, float &bv, int cull, const RayPre &r, const float4 &p0,
                                             const float4 &p1, float v2z) {
    // p0 = (v0.x, v0.y, v0.z, v1.x)  p1 = (v1.y, v1.z, v2.x, v2.y)
    float a0x = sub_(p0.x, r.ox), a0y = sub_(p0.y, r.oy), a0z = sub_(p0.z, r.oz);
    float b0x = sub_(p0.w, r.ox), b0y = sub_(p1.x, r.oy), b0z = sub_(p1.y, r.oz);
    float c0x = sub_(p1.z, r.ox), c0y = sub_(p1.w, r.oy), c0z = sub_(v2z, r.oz);
    float Ax = pick(a0x, a0y, a0z, r.kx), Ay = pick(a0x, a0y, a0z, r.ky), Az = pick(a0x, a0y, a0z, r.kz);
    float Bx = pick(b0x, b0y, b0z, r.kx), By = pick(b0x, b0y, b0z, r.ky), Bz = pick(b0x, b0y, b0z, r.kz);
    float Cx = pick(c0x, c0y, c0z, r.kx), Cy = pick(c0x, c0y, c0z, r.ky), Cz = pick(c0x, c0y, c0z, r.kz);
    Ax = sub_(Ax, mul_(r.sx, Az)), Ay = sub_(Ay, mul_(r.sy, Az));
    Bx = sub_(Bx, mul_(r.sx, Bz)), By = sub_(By, mul_(r.sy, Bz));
    Cx = sub_(Cx, mul_(r.sx, Cz)), Cy = sub_(Cy, mul_(r.sy, Cz));
    float U = sub_(mul_(Cx, By), mul_(Cy, Bx));
    float V = sub_(mul_(Ax, Cy), mul_(Ay, Cx));
    float W = sub_(mul_(Bx, Ay), mul_(By, Ax));
    float det = add_(add_(U, V), W);
    // The reference's early exits (:236-262) as ONE exit: a lane that leaves early only waits for the other lanes of its
    // warp, and every exit costs a convergence barrier.  min / max of (U, V, W) give "some edge function is negative /
    // positive" with the comparisons' own NaN behaviour (fminf / fmaxf return the non-NaN operand).
    const bool anyNeg = fminf(fminf(U, V), W) < 0.0f, anyPos = fmaxf(fmaxf(U, V), W) > 0.0f;
    bool bad = cull == 2 ? anyPos : (cull == 1 ? anyNeg : (anyNeg && anyPos));
    bad = bad || det == 0.0f;
    Az = mul_(r.sz, Az), Bz = mul_(r.sz, Bz), Cz = mul_(r.sz, Cz);
    const float T = add_(add_(mul_(U, Az), mul_(V, Bz)), mul_(W, Cz));
    const float hd = mul_(hitT, det), had = mul_(hitT, fabsf(det));
    float sT = fabsf(T);
    if ((T > 0.0f) != (det > 0.0f)) sT = -sT;
    const bool bad2 = T > 0.0f || T < hd, bad1 = T < 0.0f || T > hd, bad0 = sT < 0.0f || sT > had;
    bad = bad || (cull == 2 ? bad2 : (cull == 1 ? bad1 : bad0));
    if (bad) return false;
    float rcpDet = div_(1.0f, det);
    bu = mul_(V, rcpDet);
    bv = mul_(W, rcpDet);
    hitT = mul_(T, rcpDet);
    return true;
}

// The `cull` argument of ray_triangle for a ray entering an instance: TraverseFunction.hlsli:215-220.
__device__ __forceinline__ int cull_mode(uint32_t instFlags, uint32_t rayFlags) {
    const bool useCulling = !(instFlags & RT_INSTANCE_FLAG_TRIANGLE_CULL_DISABLE);
    const bool flip = (instFlags & RT_INSTANCE_FLAG_TRIANGLE_FRONT_COUNTERCLOCKWISE) != 0;
    const uint32_t backFlag = flip ? RT_RAY_FLAG_CULL_FRONT_FACING_TRIANGLES : RT_RAY_FLAG_CULL_BACK_FACING_TRIANGLES;
    const uint32_t frontFlag = flip ? RT_RAY_FLAG_CULL_BACK_FACING_TRIANGLES : RT_RAY_FLAG_CULL_FRONT_FACING_TRIANGLES;
    return (useCulling && (rayFlags & frontFlag)) ? 2 : ((useCulling && (rayFlags & backFlag)) ? 1 : 0);
}

// IsOpaque(): TraverseFunction.hlsli:119-134.  The geometry flag, overridden by the instance's FORCE_(NON_)OPAQUE,
// overridden by the ray's.
__device__ __forceinline__ bool is_opaque(uint32_t geomFlags, uint32_t instFlags, uint32_t rayFlags) {
    bool opaque = (geomFlags & RT_GEOMETRY_FLAG_OPAQUE) != 0;
    if (instFlags & RT_INSTANCE_FLAG_FORCE_OPAQUE) opaque = true;
    else if (instFlags & RT_INSTANCE_FLAG_FORCE_NON_OPAQUE) opaque = false;
    if (rayFlags & RT_RAY_FLAG_FORCE_OPAQUE) opaque = true;
    else if (rayFlags & RT_RAY_FLAG_FORCE_NON_OPAQUE) opaque = false;
    return opaque;
}

// `status` != nullptr: the caller's kernels know triangles only (hit groups of type TRIANGLES).  A TLAS that reaches
// procedural primitives is then a hit-group type mismatch: status bit 1 is raised (rt_get_status -> RT_ERR_UNSUPPORTED)
// and every ray misses.  rt_trace_rays_hit_groups is the entry point that runs intersection programs.
__device__ __forceinline__ TraceAccel resolve_tlas(const void *tlas_result, uint32_t *status = nullptr) {
    const uint8_t *base = static_cast<const uint8_t *>(tlas_result);
    const rt_bvh_offsets *off = reinterpret_cast<const rt_bvh_offsets *>(base);
    const rt_ext_header *e = reinterpret_cast<const rt_ext_header *>(base + align_up(off->totalSize, 64));
    TraceAccel a;
    a.wide = reinterpret_cast<const rt_wide_node *>(base + e->off_wide);
    a.wide4 = reinterpret_cast<const rt_wide4_node *>(base + e->off_wide4);
    a.inst = reinterpret_cast<const rt_packed_instance *>(base + e->off_leaf);
    a.root_ref = e->root_ref;
    a.count = e->count;
    if (status != nullptr && e->has_procedural) {
        if (threadIdx.x == 0) atomicOr(status, 2u);
        a.count = 0;
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) a.root_c[k] = e->root_center[k], a.root_h[k] = e->root_half[k];
    return a;
}

#define RT_SENTINEL 0x7fffffffu  // never a valid internal index (indices are < 2^24)

// Sorting key of a child hit: the entry distance (>= 0, so its bits order like the float) with the slot number in
// the two lowest mantissa bits; a miss sorts last.
__device__ __forceinline__ uint32_t hit_key(bool hit, float t, uint32_t slot) {
    return hit ? ((__float_as_uint(t) & 0x7ffffffcu) | slot) : 0xffffffffu;
}
__device__ __forceinline__ void key_cas(uint32_t &a, uint32_t &b) {
    const uint32_t lo = min(a, b), hi = max(a, b);
    a = lo, b = hi;
}
// a ? x : y as ONE select instruction (nvcc turns some of these conditionals into branches, see pick())
__device__ __forceinline__ uint32_t select_u32(uint32_t cond, uint32_t x, uint32_t y) {
    uint32_t r;
    asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %3, 0;\n\tselp.u32 %0, %1, %2, p;\n\t}" : "=r"(r) : "r"(x), "r"(y), "r"(cond));
    return r;
}
__device__ __forceinline__ uint32_t ref_of(uint32_t key, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3) {
    const uint32_t lo = select_u32(key & 1u, r1, r0), hi = select_u32(key & 1u, r3, r2);
    return select_u32(key & 2u, hi, lo);
}

// One internal step over a 4-wide node: test the four child boxes (RayBoxTest arithmetic unchanged), order the
// hits near-to-far with a 5-exchange network on integer keys, return the nearest and push the others farthest
// first.  WITH_T: also record each pushed node's entry distance so that it can be dropped at pop time.
// The traversal stack is a policy type S with  bool room(sp, n)  and  void push(sp, ref, key):
//   LocalStack   — 64 entries (+ entry distances) in local memory: the one-thread-one-ray loop (k_primary)
//   PersistStack — 64 entries, no distances: the persistent kernels (trace_persistent.cuh)
struct LocalStack {
    uint32_t ref[RT_STACK_SIZE], key[RT_STACK_SIZE];
    __device__ __forceinline__ bool room(int sp, int n) const { return sp + n <= RT_STACK_SIZE; }
    __device__ __forceinline__ void push(int &sp, uint32_t r, uint32_t k) { ref[sp] = r, key[sp] = k, ++sp; }
};

template <bool WITH_T, bool SORTED = true, class S>
__device__ __forceinline__ uint32_t wide4_step(const rt_wide4_node *nodes, uint32_t ref, const RayPre &cur, float tCur, S &stk, int &sp,
                                               uint32_t *status) {
    const float4 *np = reinterpret_cast<const float4 *>(nodes + ref);
    float4 c0, h0, c1, h1, c2, h2, c3, h3;
    ldg256(np, c0, h0), ldg256(np + 2, c1, h1), ldg256(np + 4, c2, h2), ldg256(np + 6, c3, h3);
    float t0, t1, t2, t3;
    const bool b0 = ray_box(t0, tCur, cur, c0.x, c0.y, c0.z, h0.x, h0.y, h0.z);
    const bool b1 = ray_box(t1, tCur, cur, c1.x, c1.y, c1.z, h1.x, h1.y, h1.z);
    const bool b2 = ray_box(t2, tCur, cur, c2.x, c2.y, c2.z, h2.x, h2.y, h2.z);
    const bool b3 = ray_box(t3, tCur, cur, c3.x, c3.y, c3.z, h3.x, h3.y, h3.z);
    const uint32_t r0 = __float_as_uint(c0.w), r1 = __float_as_uint(c1.w), r2 = __float_as_uint(c2.w), r3 = __float_as_uint(c3.w);
    if (!SORTED) {
        // any-hit rays: visibility does not depend on the visiting order, so the children are taken in slot order
        uint32_t first = RT_SENTINEL;
        const bool v[4] = {b0, b1, b2 && r2 != RT_WIDE4_EMPTY, b3 && r3 != RT_WIDE4_EMPTY};
        const uint32_t r[4] = {r0, r1, r2, r3};
#pragma unroll
        for (int k = 3; k >= 0; --k) {
            if (v[k]) {
                if (first != RT_SENTINEL) {
                    if (stk.room(sp, 1)) stk.push(sp, first, 0u);
                    else atomicOr(status, 1u);
                }
                first = r[k];
            }
        }
        return first;
    }
    // slots 2 and 3 may be empty; their half = -1 box fails the slab test of every ray except one whose slabs are all
    // NaN (a zero direction passes every box, in the reference too), hence the explicit check
    uint32_t k0 = hit_key(b0, t0, 0), k1 = hit_key(b1, t1, 1), k2 = hit_key(b2 && r2 != RT_WIDE4_EMPTY, t2, 2),
             k3 = hit_key(b3 && r3 != RT_WIDE4_EMPTY, t3, 3);
    key_cas(k0, k1), key_cas(k2, k3), key_cas(k0, k2), key_cas(k1, k3), key_cas(k1, k2);
    if (k0 == 0xffffffffu) return RT_SENTINEL;
    if (k1 != 0xffffffffu) {  // push the other hits, farthest first
        if (!stk.room(sp, 3)) {
            atomicOr(status, 1u);
        } else {
            if (k3 != 0xffffffffu) stk.push(sp, ref_of(k3, r0, r1, r2, r3), k3);
            if (k2 != 0xffffffffu) stk.push(sp, ref_of(k2, r0, r1, r2, r3), k2);
            stk.push(sp, ref_of(k1, r0, r1, r2, r3), k1);
        }
    }
    return ref_of(k0, r0, r1, r2, r3);
}

// Closest-hit traversal of ONE ray over the 4-wide nodes, for coherent rays (one thread per pixel): the same
// hits as trace_ray (same box / triangle arithmetic and acceptance rule) in a different visiting order.  No
// any-hit / opaque-flag handling: the caller's rays carry only cull flags (RayGen: CULL_BACK_FACING_TRIANGLES).
__device__ __forceinline__ bool trace_ray4(const TraceAccel &A, float ox, float oy, float oz, float tmin, float dx, float dy, float dz,
                                           float tmax, uint32_t rayFlags, uint32_t mask, uint32_t rayContribution, TraceHit &hit,
                                           uint32_t *status) {
    hit.prim = RT_NO_HIT;
    hit.t = tmax;
    hit.u = hit.v = 0.0f;
    hit.inst_index = hit.geom_index = hit.inst_id = hit.leaf_slot = hit.record = 0;
    if (A.count == 0) return false;
    LocalStack stk;
    int sp = 0, blasBase = -1;
    float tCur = tmax;
    RayPre cur;
    ray_pre_box<true>(cur, ox, oy, oz, dx, dy, dz);
    float tUnused;
    if (!ray_box(tUnused, tCur, cur, A.root_c[0], A.root_c[1], A.root_c[2], A.root_h[0], A.root_h[1], A.root_h[2])) return false;
    const bool plain = [&] {
        const float v[6] = {ox, oy, oz, dx, dy, dz};
        bool p = true;
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            const uint32_t b = __float_as_uint(v[k]);
            p = p && b != 0x80000000u && (b & 0x7f800000u) != 0x7f800000u;
        }
        return p;
    }();
    const rt_wide4_node *nodes = A.wide4;
    const rt_packed_tri *tris = nullptr;
    bool bottom = false, sameSpace = false;
    uint32_t instIndex = 0, instOffset = 0, instId = 0;
    int cull = 0;
    uint32_t ref = A.root_ref;
    while (true) {
        if (ref & RT_NODE_LEAF_FLAG) {
            const uint32_t slot = ref & 0x00ffffffu;
            ref = RT_SENTINEL;
            if (!bottom) {
                const uint4 *ip = reinterpret_cast<const uint4 *>(A.inst + slot);
                const uint4 m3 = __ldg(ip + 3);
                if ((m3.x >> 24) & mask) {
                    const uint4 m4 = __ldg(ip + 4);
                    instIndex = m3.z, instOffset = m3.y & 0x00ffffffu, instId = m3.x & 0x00ffffffu;
                    cull = cull_mode(m3.y >> 24, rayFlags);
                    sameSpace = plain && (m3.y & RT_PACKED_INSTANCE_IDENTITY);
                    if (sameSpace) {
                        ray_pre_shear(cur, dx, dy, dz);
                    } else {
                        const float4 r0 = __ldg(reinterpret_cast<const float4 *>(ip));
                        const float4 r1 = __ldg(reinterpret_cast<const float4 *>(ip + 1));
                        const float4 r2 = __ldg(reinterpret_cast<const float4 *>(ip + 2));
                        const float m[12] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w, r2.x, r2.y, r2.z, r2.w};
                        const f3 o2 = xform_point(m, mk3(ox, oy, oz));
                        const f3 d2 = xform_vector(m, mk3(dx, dy, dz));
                        cur = make_ray_pre<true>(o2.x, o2.y, o2.z, d2.x, d2.y, d2.z);
                    }
                    nodes = reinterpret_cast<const rt_wide4_node *>(__ldg(reinterpret_cast<const unsigned long long *>(ip + 5)));
                    tris = reinterpret_cast<const rt_packed_tri *>(uintptr_t(uint64_t(m4.z) | (uint64_t(m4.w) << 32)));
                    bottom = true;
                    blasBase = sp;
                    ref = m3.w;
                }
            } else {
                const float4 *tp = reinterpret_cast<const float4 *>(tris + slot);
                const float4 p0 = __ldg(tp), p1 = __ldg(tp + 1), p2 = __ldg(tp + 2);
                float t0 = tCur, bu, bv;
                if (ray_triangle(t0, bu, bv, cull, cur, p0, p1, p2.x) && t0 < tCur && t0 > tmin) {
                    tCur = t0;
                    hit.t = t0, hit.u = bu, hit.v = bv;
                    hit.prim = __float_as_uint(p2.y);
                    hit.geom_index = __float_as_uint(p2.z);
                    hit.inst_index = instIndex, hit.inst_id = instId, hit.leaf_slot = slot;
                    hit.record = rayContribution + instOffset;
                }
            }
        } else {
            ref = wide4_step<true>(nodes, ref, cur, tCur, stk, sp, status);
        }
        if (ref == RT_SENTINEL) {
            bool done = false;
            for (;;) {
                if (sp == 0) {
                    done = true;
                    break;
                }
                if (bottom && sp == blasBase) {
                    bottom = false;
                    if (!sameSpace) ray_pre_box<true>(cur, ox, oy, oz, dx, dy, dz);
                    nodes = A.wide4;
                    blasBase = -1;
                }
                --sp;
                if ((stk.key[sp] & 0x7ffffffcu) >= __float_as_uint(tCur)) continue;
                ref = stk.ref[sp];
                break;
            }
            if (done) break;
        }
    }
    return hit.prim != RT_NO_HIT;
}

// Fallback_TraceRay without shader call-outs.  ANY = RAY_FLAG_ACCEPT_FIRST_HIT_AND_END_SEARCH.
// rayContribution / geomMultiplier feed the hit-group record index exactly as TraverseFunction.hlsli:684-687.
// ---------------------------------------------------------------------------------------------------------------
// Compiled-in any-hit / intersection programs (rt_types.h RT_ANYHIT_*, RT_INTERSECTION_*) and the machinery the
// reference runs around application shaders: InvokeAnyHit / IgnoreHit / AcceptHitAndEndSearch
// (FL/TraverseFunction.hlsli:102-117) and Fallback_ReportHit (:136-158).  Same arithmetic, operation for operation,
// as the CPU restatement the parity tests check it against (the library is built with -fmad=false).
struct HitPrograms {
    const rt_hit_group_programs *table;  // one entry per hit-group record; nullptr = no any-hit / intersection programs
    uint32_t count;
};
#define RT_AH_END_SEARCH (-1)
#define RT_AH_IGNORE 0
#define RT_AH_ACCEPT 1

__device__ __forceinline__ int run_any_hit(uint32_t program, float ax, float ay) {
    switch (program) {
        case RT_ANYHIT_IGNORE: return RT_AH_IGNORE;
        case RT_ANYHIT_END_SEARCH: return RT_AH_END_SEARCH;
        case RT_ANYHIT_CUTOUT: return ((int(floorf(8.0f * ax)) + int(floorf(8.0f * ay))) & 1) ? RT_AH_IGNORE : RT_AH_ACCEPT;
        default: return RT_AH_ACCEPT;
    }
}

struct ReportCtx {
    float tmin, tCur;
    uint32_t rayFlags, anyHit;
    int anyHitResult;
    bool committed;
    float t, ax, ay;
    uint32_t kind;
};

__device__ __forceinline__ int report_hit(ReportCtx &c, float tHit, uint32_t hitKind, float ax, float ay) {
    if (tHit < c.tmin || c.tCur <= tHit) return 0;
    int ret = RT_AH_ACCEPT;
    bool opaque = true;  // "geomOpaque = true; // TODO" and instance flags 0 in the reference (:147-149)
    if (c.rayFlags & RT_RAY_FLAG_FORCE_OPAQUE) opaque = true;
    else if (c.rayFlags & RT_RAY_FLAG_FORCE_NON_OPAQUE) opaque = false;
    if (c.anyHit > 0 && !opaque) ret = c.anyHitResult = run_any_hit(c.anyHit, ax, ay);
    if (ret != RT_AH_IGNORE) {
        c.tCur = tHit;
        c.committed = true;
        c.t = tHit, c.ax = ax, c.ay = ay, c.kind = hitKind;
        if (c.rayFlags & RT_RAY_FLAG_ACCEPT_FIRST_HIT_AND_END_SEARCH) ret = RT_AH_END_SEARCH;
    }
    return ret;
}

__device__ __forceinline__ float dot3_(f3 a, f3 b) { return (a.x * b.x + a.y * b.y) + a.z * b.z; }

__device__ __forceinline__ void intersect_box(ReportCtx &c, f3 o, f3 d, f3 mn, f3 mx) {
    const f3 t0 = mk3((mn.x - o.x) / d.x, (mn.y - o.y) / d.y, (mn.z - o.z) / d.z);
    const f3 t1 = mk3((mx.x - o.x) / d.x, (mx.y - o.y) / d.y, (mx.z - o.z) / d.z);
    const float tNear = fmaxf(fmaxf(fminf(t0.x, t1.x), fminf(t0.y, t1.y)), fminf(t0.z, t1.z));
    const float tFar = fminf(fminf(fmaxf(t0.x, t1.x), fmaxf(t0.y, t1.y)), fmaxf(t0.z, t1.z));
    if (!(tNear <= tFar)) return;
    if (report_hit(c, tNear, RT_HIT_KIND_BOX_ENTER, 0.0f, 0.0f) == 0) report_hit(c, tFar, RT_HIT_KIND_BOX_EXIT, 0.0f, 0.0f);
}

__device__ __forceinline__ void intersect_sphere(ReportCtx &c, f3 o, f3 d, f3 mn, f3 mx) {
    const f3 ctr = mk3((mn.x + mx.x) * 0.5f, (mn.y + mx.y) * 0.5f, (mn.z + mx.z) * 0.5f);
    const f3 h = mk3(mx.x - ctr.x, mx.y - ctr.y, mx.z - ctr.z);
    const float r = fminf(fminf(h.x, h.y), h.z);
    if (!(r > 0.0f)) return;
    const f3 oc = mk3(o.x - ctr.x, o.y - ctr.y, o.z - ctr.z);
    const float a = dot3_(d, d), b = dot3_(oc, d), cc = dot3_(oc, oc) - r * r;
    const float disc = b * b - a * cc;
    if (!(disc >= 0.0f) || !(a > 0.0f)) return;
    const float s = sqrtf(disc);
    const float tA = (-b - s) / a, tB = (-b + s) / a;
    const float nAx = (oc.x + d.x * tA) / r, nAy = (oc.y + d.y * tA) / r;
    const float nBx = (oc.x + d.x * tB) / r, nBy = (oc.y + d.y * tB) / r;
    if (report_hit(c, tA, RT_HIT_KIND_SPHERE_ENTER, nAx, nAy) == 0) report_hit(c, tB, RT_HIT_KIND_SPHERE_EXIT, nBx, nBy);
}

// HOOKS = true: hit groups may carry any-hit / intersection programs and the BLAS may hold procedural primitives
// (rt_trace_rays_hit_groups); hit.leaf_slot then carries HitKind() in bits 31:24.  HOOKS = false is the application's
// case — all-triangle geometry and, at most, a no-op any-hit shader — and compiles to exactly the loop it was.
template <bool ANY, bool STATS, bool HOOKS = false>
__device__ __forceinline__ bool trace_ray(const TraceAccel &A, float ox, float oy, float oz, float tmin, float dx, float dy,
                                          float dz, float tmax, uint32_t rayFlags, uint32_t mask, uint32_t rayContribution,
                                          uint32_t geomMultiplier, TraceHit &hit, TraceCtr *ctr, uint32_t *status,
                                          HitPrograms programs = HitPrograms{nullptr, 0}) {
    hit.prim = RT_NO_HIT;
    hit.t = tmax;
    hit.u = hit.v = 0.0f;
    hit.inst_index = hit.geom_index = hit.inst_id = hit.leaf_slot = hit.record = 0;
    if (A.count == 0) return false;

    uint32_t stack[RT_STACK_SIZE];
    int sp = 0;
    float tCur = tmax;

    RayPre world = make_ray_pre<!STATS>(ox, oy, oz, dx, dy, dz);
    RayPre cur = world;
    const rt_wide_node *nodes = A.wide;
    const rt_packed_tri *tris = nullptr;
    bool bottom = false;
    int blasBase = -1;  // stack height at which the current BLAS was entered
    uint32_t instIndex = 0, instFlags = 0, instOffset = 0, instId = 0;
    int cull = 0;
    f3 objO = mk3(ox, oy, oz), objD = mk3(dx, dy, dz);  // ObjectRayOrigin() / ObjectRayDirection() (HOOKS only)

    float tUnused;
    if (!ray_box(tUnused, tCur, world, A.root_c[0], A.root_c[1], A.root_c[2], A.root_h[0], A.root_h[1], A.root_h[2])) return false;

    uint32_t ref = A.root_ref;
    while (true) {
        if (ref & RT_NODE_LEAF_FLAG) {
            const uint32_t slot = ref & 0x00ffffffu;
            if (!bottom) {
                // TLAS leaf: TraverseFunction.hlsli:598-634
                if (STATS) ctr->inst++;
                const uint4 *ip = reinterpret_cast<const uint4 *>(A.inst + slot);
                const uint4 m3 = __ldg(ip + 3);  // id|mask, hitgroup|flags, instance index, blas root ref
                instIndex = m3.z;
                instOffset = m3.y & 0x00ffffffu;
                instId = m3.x & 0x00ffffffu;
                ref = RT_SENTINEL;
                if ((m3.x >> 24) & mask) {
                    const float4 r0 = __ldg(reinterpret_cast<const float4 *>(ip));
                    const float4 r1 = __ldg(reinterpret_cast<const float4 *>(ip + 1));
                    const float4 r2 = __ldg(reinterpret_cast<const float4 *>(ip + 2));
                    const uint4 m4 = __ldg(ip + 4);
                    instFlags = m3.y >> 24;
                    cull = cull_mode(instFlags, rayFlags);
                    const float m[12] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w, r2.x, r2.y, r2.z, r2.w};
                    f3 o2 = xform_point(m, mk3(ox, oy, oz));
                    f3 d2 = xform_vector(m, mk3(dx, dy, dz));
                    cur = make_ray_pre<!STATS>(o2.x, o2.y, o2.z, d2.x, d2.y, d2.z);
                    if (HOOKS) objO = o2, objD = d2;
                    nodes = reinterpret_cast<const rt_wide_node *>(uintptr_t(uint64_t(m4.x) | (uint64_t(m4.y) << 32)));
                    tris = reinterpret_cast<const rt_packed_tri *>(uintptr_t(uint64_t(m4.z) | (uint64_t(m4.w) << 32)));
                    bottom = true;
                    blasBase = sp;
                    ref = m3.w;  // BLAS root (pushed without a box test, as the reference does)
                }
            } else {
                // BLAS leaf: TraverseFunction.hlsli:635-735
                if (STATS) ctr->leaf++;
                const float4 *tp = reinterpret_cast<const float4 *>(tris + slot);
                const float4 p0 = __ldg(tp), p1 = __ldg(tp + 1), p2 = __ldg(tp + 2);
                const uint32_t gflags = __float_as_uint(p2.w);
                const bool opaque = is_opaque(gflags, instFlags, rayFlags);
                const bool culled = (opaque && (rayFlags & RT_RAY_FLAG_CULL_OPAQUE)) || (!opaque && (rayFlags & RT_RAY_FLAG_CULL_NON_OPAQUE));
                ref = RT_SENTINEL;
                if (HOOKS) {
                    const uint32_t geomIndex = __float_as_uint(p2.z);
                    const uint32_t record = rayContribution + geomIndex * geomMultiplier + instOffset;
                    rt_hit_group_programs prog{RT_ANYHIT_NONE, RT_INTERSECTION_NONE};
                    if (programs.table != nullptr && record < programs.count) prog = programs.table[record];
                    bool endSearch = false, commit = false;
                    float ct = 0.0f, cu = 0.0f, cv = 0.0f;
                    uint32_t kind = 0;
                    if (!culled && (gflags & RT_PACKED_PROCEDURAL)) {
                        // :656-671
                        ReportCtx rc{tmin, tCur, rayFlags, prog.any_hit, RT_AH_ACCEPT, false, 0.0f, 0.0f, 0.0f, 0u};
                        if (prog.intersection == RT_INTERSECTION_BOX)
                            intersect_box(rc, objO, objD, mk3(p0.x, p0.y, p0.z), mk3(p0.w, p1.x, p1.y));
                        else if (prog.intersection == RT_INTERSECTION_SPHERE)
                            intersect_sphere(rc, objO, objD, mk3(p0.x, p0.y, p0.z), mk3(p0.w, p1.x, p1.y));
                        commit = rc.committed, ct = rc.t, cu = rc.ax, cv = rc.ay, kind = rc.kind;
                        endSearch = rc.anyHitResult == RT_AH_END_SEARCH;
                    } else if (!culled) {
                        float t0 = tCur, bu, bv;
                        if (ray_triangle(t0, bu, bv, cull, cur, p0, p1, p2.x) && t0 < tCur && t0 > tmin) {
                            // :699-722 (under ACCEPT_FIRST_HIT an ignored candidate still ends the search, :721)
                            int ret = RT_AH_ACCEPT;
                            if (!opaque && prog.any_hit) ret = run_any_hit(prog.any_hit, bu, bv);
                            commit = ret != RT_AH_IGNORE, ct = t0, cu = bu, cv = bv, kind = RT_HIT_KIND_TRIANGLE_FRONT_FACE;
                            endSearch = ret == RT_AH_END_SEARCH || ANY;
                        }
                    }
                    if (commit) {
                        tCur = ct;
                        hit.t = ct, hit.u = cu, hit.v = cv;
                        hit.prim = __float_as_uint(p2.y);
                        hit.geom_index = geomIndex;
                        hit.inst_index = instIndex;
                        hit.inst_id = instId;
                        hit.leaf_slot = slot | (kind << 24);
                        hit.record = record;
                    }
                    if (endSearch) return hit.prim != RT_NO_HIT;
                } else if (!culled) {
                    float t0 = tCur, bu, bv;
                    if (ray_triangle(t0, bu, bv, cull, cur, p0, p1, p2.x) && t0 < tCur && t0 > tmin) {
                        tCur = t0;
                        hit.t = t0, hit.u = bu, hit.v = bv;
                        hit.prim = __float_as_uint(p2.y);
                        hit.geom_index = __float_as_uint(p2.z);
                        hit.inst_index = instIndex;
                        hit.inst_id = instId;
                        hit.leaf_slot = slot;
                        hit.record = rayContribution + hit.geom_index * geomMultiplier + instOffset;
                        if (ANY) return true;
                    }
                }
            }
        } else {
            // internal node: TraverseFunction.hlsli:737-786 with both child boxes in the node
            if (STATS) ctr->internal++;
            const float4 *np = reinterpret_cast<const float4 *>(nodes + ref);
            const float4 n0 = __ldg(np), n1 = __ldg(np + 1), n2 = __ldg(np + 2), n3 = __ldg(np + 3);
            float lt, rt;
            const bool lh = ray_box(lt, tCur, cur, n0.x, n0.y, n0.z, n1.x, n1.y, n1.z);
            const bool rh = ray_box(rt, tCur, cur, n2.x, n2.y, n2.z, n3.x, n3.y, n3.z);
            const uint32_t l = __float_as_uint(n0.w), r = __float_as_uint(n1.w);
            if (lh && rh) {
                const bool rightFirst = rt < lt;  // ties: left first
                if (sp < RT_STACK_SIZE) stack[sp++] = rightFirst ? l : r;
                else atomicOr(status, 1u);
                if (STATS) ctr->max_stack = max(ctr->max_stack, uint32_t(sp) + 1);
                ref = rightFirst ? r : l;
            } else if (lh || rh) {
                ref = rh ? r : l;
            } else {
                ref = RT_SENTINEL;
            }
        }
        if (ref == RT_SENTINEL) {
            // pop; leaving a BLAS restores the world-space ray (TraverseFunction.hlsli:788-791)
            if (bottom && sp == blasBase) {
                bottom = false;
                cur = world;
                if (HOOKS) objO = mk3(ox, oy, oz), objD = mk3(dx, dy, dz);
                nodes = A.wide;
                blasBase = -1;
            }
            if (sp == 0) break;
            ref = stack[--sp];
        }
    }
    return hit.prim != RT_NO_HIT;
}
