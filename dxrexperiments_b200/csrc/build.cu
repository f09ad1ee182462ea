// build.cu — LBVH acceleration-structure build for sm_100a.
//
// B200-native replacement of the Fallback Layer's GpuBvh2Builder pass chain
// (externals/D3D12RaytracingFallback/src/GpuBVH2Builder.cpp:137-328): load -> scene AABB -> 30-bit Morton
// codes -> sort -> rearrange -> Karras hierarchy -> bottom-up AABB fit, for BLAS (triangles) and TLAS
// (instances).  Differences in HOW (results are bit-identical to the CPU restatement):
//   * scene AABB is one fused pass (block reduce + ordered-int atomics) instead of ceil(log8 N) dispatches;
//   * the O(log^2 N)-pass bitonic sort becomes a 4-pass stable LSD radix sort, which yields exactly the
//     order BitonicSortCommon.hlsli:37-47 defines (ascending key, ties by ascending index);
//   * the fit pass also emits this library's traversal section (64-byte nodes with both child boxes, 128-byte
//     4-wide nodes, 48-byte triangles) so no separate packing pass re-reads the tree;
//   * a plain LBVH build (PREFER_FAST_BUILD: no treelet pass) emits the Karras hierarchy and fits the boxes in ONE
//     bottom-up kernel (k_lbvh_fit / k_lbvh_exits): no binary searches, no hierarchy array.
// This file is compiled with -fmad=false: every float op below is the IEEE operation written.
#include <algorithm>
#include <cfloat>
#include <cstdio>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "treelet.cuh"

namespace {

constexpr int kThreads = 256;

// ------------------------------------------------------------------------------------------ utilities
__device__ __forceinline__ uint32_t enc_f32(float f) {  // monotonic float -> uint
    uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float dec_f32(uint32_t e) {
    uint32_t b = (e & 0x80000000u) ? (e & 0x7fffffffu) : ~e;
    return __uint_as_float(b);
}

struct Aabb3 {
    float mn[3], mx[3];
};

// Warp shuffles, then one shared-memory exchange, then ONE set of six atomics per block (a per-warp version sent
// 1.9 M atomics to the same six words for a 10 M-triangle build and made the load pass atomics-bound).
__device__ __forceinline__ void block_reduce_aabb(float mn[3], float mx[3], uint32_t *enc /* 6 words */) {
    __shared__ float s_red[32][6];
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mn[k] = fminf(mn[k], __shfl_xor_sync(0xffffffffu, mn[k], o));
            mx[k] = fmaxf(mx[k], __shfl_xor_sync(0xffffffffu, mx[k], o));
        }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 3; ++k) s_red[warp][k] = mn[k], s_red[warp][3 + k] = mx[k];
    }
    __syncthreads();
    if (warp == 0) {
        float v[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) v[k] = lane < nwarps ? s_red[lane][k] : (k < 3 ? FLT_MAX : -FLT_MAX);
#pragma unroll
        for (int k = 0; k < 6; ++k)
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float t = __shfl_xor_sync(0xffffffffu, v[k], o);
                v[k] = k < 3 ? fminf(v[k], t) : fmaxf(v[k], t);
            }
        if (lane == 0) {
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                atomicMin(&enc[k], enc_f32(v[k]));
                atomicMax(&enc[3 + k], enc_f32(v[3 + k]));
            }
        }
    }
}

__global__ void k_init_aabb(uint32_t *enc) {
    if (threadIdx.x < 3) enc[threadIdx.x] = enc_f32(FLT_MAX);
    else if (threadIdx.x < 6) enc[threadIdx.x] = enc_f32(-FLT_MAX);
    else if (threadIdx.x < 8) enc[threadIdx.x] = 0;  // spare words of the 32-byte slot (k_lbvh_fit's exit-list length)
}
__global__ void k_decode_aabb(const uint32_t *enc, float *out) {
    // + 0.0f canonicalises -0 to +0 (fminf(-0,+0) is unspecified on the CPU side).
    if (threadIdx.x < 6) out[threadIdx.x] = dec_f32(enc[threadIdx.x]) + 0.0f;
}

// ------------------------------------------------------------------------------------------ load triangles
// FL/BottomLevelLoadTriangles.hlsli:88-126 + LoadPrimitivesBindings.h:72-79, fused with the scene AABB
// (FL/CalculateSceneAABBFromPrimitives.hlsl:16-40).
struct LoadGeom {
    const uint8_t *vb;
    const void *ib;
    uint32_t stride, index_format, num_tris, prim_offset, geom_index, flags, has_xf, procedural;
    float xf[12];
};

// The load-order scratch record is the 48-byte rt_packed_tri (9 floats + PrimitiveMetaData): three aligned 16-byte
// stores here, three aligned 16-byte gathers in k_rearrange_tris (gathering the reference's unaligned 40 + 12 byte
// records instead cost 2.6 GB of DRAM reads per 10 M triangles).
__global__ void __launch_bounds__(kThreads) k_load_triangles(LoadGeom g, rt_packed_tri *recs, uint32_t *aabb_enc) {
    float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < g.num_tris; t += gridDim.x * blockDim.x) {
        if (g.procedural) {
            // FL/LoadProceduralGeometry.hlsl:16-42: the AABB is copied verbatim; scene AABB from min and max
            // (CalculateSceneAABBFromPrimitives.hlsl:32-37)
            const float *p = reinterpret_cast<const float *>(g.vb + size_t(t) * g.stride);
            const float b[6] = {p[0], p[1], p[2], p[3], p[4], p[5]};
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                mn[k] = fminf(fminf(mn[k], b[k]), b[3 + k]);
                mx[k] = fmaxf(fmaxf(mx[k], b[k]), b[3 + k]);
            }
            float4 *dst = reinterpret_cast<float4 *>(recs + g.prim_offset + t);
            dst[0] = make_float4(b[0], b[1], b[2], b[3]);
            dst[1] = make_float4(b[4], b[5], 0.0f, 0.0f);
            dst[2] = make_float4(0.0f, __uint_as_float(t), __uint_as_float(g.geom_index), __uint_as_float(g.flags | RT_PACKED_PROCEDURAL));
            continue;
        }
        uint32_t idx[3];
        if (g.index_format == 32) {
            const uint32_t *ib = static_cast<const uint32_t *>(g.ib);
            idx[0] = ib[3 * size_t(t)], idx[1] = ib[3 * size_t(t) + 1], idx[2] = ib[3 * size_t(t) + 2];
        } else if (g.index_format == 16) {
            const uint16_t *ib = static_cast<const uint16_t *>(g.ib);
            idx[0] = ib[3 * size_t(t)], idx[1] = ib[3 * size_t(t) + 1], idx[2] = ib[3 * size_t(t) + 2];
        } else {
            idx[0] = 3 * t, idx[1] = 3 * t + 1, idx[2] = 3 * t + 2;
        }
        float w[9];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float *p = reinterpret_cast<const float *>(g.vb + size_t(idx[k]) * g.stride);
            f3 v = mk3(p[0], p[1], p[2]);
            if (g.has_xf) v = xform_point(g.xf, v);
            w[3 * k] = v.x, w[3 * k + 1] = v.y, w[3 * k + 2] = v.z;
            mn[0] = fminf(mn[0], v.x), mn[1] = fminf(mn[1], v.y), mn[2] = fminf(mn[2], v.z);
            mx[0] = fmaxf(mx[0], v.x), mx[1] = fmaxf(mx[1], v.y), mx[2] = fmaxf(mx[2], v.z);
        }
        float4 *dst = reinterpret_cast<float4 *>(recs + g.prim_offset + t);
        dst[0] = make_float4(w[0], w[1], w[2], w[3]);
        dst[1] = make_float4(w[4], w[5], w[6], w[7]);
        dst[2] = make_float4(w[8], __uint_as_float(t), __uint_as_float(g.geom_index), __uint_as_float(g.flags));
    }
    block_reduce_aabb(mn, mx, aabb_enc);
}

// ------------------------------------------------------------------------------------------ Morton codes
// FL/CalculateMortonCodes.hlsli:73-118 (non-scaled variant).
__device__ __forceinline__ uint32_t expand10(uint32_t v) {  // bit b -> bit 3b
    v &= 0x3ffu;
    v = (v | (v << 16)) & 0x030000ffu;
    v = (v | (v << 8)) & 0x0300f00fu;
    v = (v | (v << 4)) & 0x030c30c3u;
    v = (v | (v << 2)) & 0x09249249u;
    return v;
}
__device__ __forceinline__ uint32_t morton_from_centroid(f3 c, const float *aabb) {
    const float eps = 0.00001f;
    float dx = fmaxf(aabb[3] - aabb[0], eps), dy = fmaxf(aabb[4] - aabb[1], eps), dz = fmaxf(aabb[5] - aabb[2], eps);
    float ux = (c.x - aabb[0]) / dx, uy = (c.y - aabb[1]) / dy, uz = (c.z - aabb[2]) / dz;
    float ax = fminf(fmaxf(ux * 1024.0f, 0.0f), 1023.0f), ay = fminf(fmaxf(uy * 1024.0f, 0.0f), 1023.0f),
          az = fminf(fmaxf(uz * 1024.0f, 0.0f), 1023.0f);
    uint32_t qx = uint32_t(ax), qy = uint32_t(ay), qz = uint32_t(az);
    // axis order (y, x, z): bit 3b+0 <- y, 3b+1 <- x, 3b+2 <- z
    return expand10(qy) | (expand10(qx) << 1) | (expand10(qz) << 2);
}

__global__ void __launch_bounds__(kThreads) k_morton_prims(const rt_packed_tri *recs, uint32_t n, const float *aabb,
                                                           uint32_t *codes) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 *q = reinterpret_cast<const float4 *>(recs + i);
    const float4 q0 = q[0], q1 = q[1], q2 = q[2];
    const float v[9] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x};
    // (v0 + v1 + v2) / 3.0  (CalculateMortonCodesForPrimitives.hlsl:22-25); procedural: (min + max) / 2.0 (:26-30)
    f3 c = (__float_as_uint(q2.w) & RT_PACKED_PROCEDURAL)
               ? mk3((v[0] + v[3]) / 2.0f, (v[1] + v[4]) / 2.0f, (v[2] + v[5]) / 2.0f)
               : mk3(((v[0] + v[3]) + v[6]) / 3.0f, ((v[1] + v[4]) + v[7]) / 3.0f, ((v[2] + v[5]) + v[8]) / 3.0f);
    codes[i] = morton_from_centroid(c, aabb);
}

__global__ void __launch_bounds__(kThreads) k_morton_boxes(const rt_aabb_node *boxes, uint32_t n, const float *aabb,
                                                           uint32_t *codes) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    codes[i] = morton_from_centroid(mk3(boxes[i].center[0], boxes[i].center[1], boxes[i].center[2]), aabb);
}

// ------------------------------------------------------------------------------------------ radix sort
// Stable LSD radix sort of (key, value) pairs, 8-bit digits.  Each block owns a contiguous range of tiles,
// so the digit-major scan is over a fixed 256 x gridDim array whatever N is.
constexpr int kRadixBits = 8, kRadix = 1 << kRadixBits, kSortThreads = 256, kSortItems = 8;
constexpr int kSortTile = kSortThreads * kSortItems;
constexpr int kSortWarps = kSortThreads / 32;

__global__ void __launch_bounds__(kSortThreads) k_radix_hist(const uint32_t *keys, uint32_t n, int shift,
                                                             uint32_t tiles_per_block, uint32_t *hist /* [256][grid] */) {
    __shared__ uint32_t s[kRadix];
    s[threadIdx.x] = 0;
    __syncthreads();
    uint64_t begin = uint64_t(blockIdx.x) * tiles_per_block * kSortTile;
    uint64_t end = min(uint64_t(n), begin + uint64_t(tiles_per_block) * kSortTile);
    for (uint64_t i = begin + threadIdx.x; i < end; i += kSortThreads) atomicAdd(&s[(keys[i] >> shift) & (kRadix - 1)], 1u);
    __syncthreads();
    hist[threadIdx.x * gridDim.x + blockIdx.x] = s[threadIdx.x];
}

// Exclusive scan of the digit-major histogram hist[256][G] in flattened order, split in two: block d scans row d
// (G <= 4 x SMs entries) and leaves the row total in row_total[d]; the 256 row totals are scanned by every scatter
// block for itself (k_radix_scatter).  One 1024-thread block doing the whole table took 50 us per pass.
__device__ __forceinline__ uint32_t block_exclusive_scan_256(uint32_t v, uint32_t *s_warp /* [8] */, uint32_t &total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint32_t base = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < kSortWarps; ++w) {
        const uint32_t c = s_warp[w];
        if (w < warp) base += c;
        tot += c;
    }
    total = tot;
    __syncthreads();
    return base + incl - v;
}

__global__ void __launch_bounds__(kSortThreads) k_scan_rows(uint32_t *hist, uint32_t G, uint32_t *row_total) {
    __shared__ uint32_t s_warp[kSortWarps];
    uint32_t *p = hist + size_t(blockIdx.x) * G;
    const uint32_t per = (G + kSortThreads - 1) / kSortThreads;  // consecutive entries per thread
    const uint32_t c0 = threadIdx.x * per;
    uint32_t sum = 0;
    for (uint32_t k = 0; k < per; ++k) sum += (c0 + k < G) ? p[c0 + k] : 0u;
    uint32_t total;
    uint32_t run = block_exclusive_scan_256(sum, s_warp, total);
    for (uint32_t k = 0; k < per; ++k)
        if (c0 + k < G) {
            const uint32_t v = p[c0 + k];
            p[c0 + k] = run;
            run += v;
        }
    if (threadIdx.x == 0) row_total[blockIdx.x] = total;
}

// One pass of the LSD sort over this block's tiles.  Five block barriers per tile (a first version had nine, and four
// resident blocks per SM do not hide them): the digit counters are cleared and the keys loaded before barrier A, the
// running bases take the previous tile's counts right after it, the values are fetched once the ranks are known so that
// their latency falls into the scan phases.  (Staging the next tile's keys and values in shared memory with cp.async was
// measured and changed nothing: 2.867 vs 2.853 ms for the 10 M-triangle build.)
template <bool IOTA>
__global__ void __launch_bounds__(kSortThreads, 4) k_radix_scatter(const uint32_t *keys_in, const uint32_t *vals_in, uint32_t n,
                                                                   int shift, uint32_t tiles_per_block, const uint32_t *offsets,
                                                                   const uint32_t *row_total, uint32_t *keys_out, uint32_t *vals_out) {
    __shared__ uint32_t warp_count[kSortWarps][kRadix];
    __shared__ uint32_t base[kRadix], tile_start[kRadix], tile_count[kRadix];
    __shared__ uint32_t s_warp[kSortWarps];
    __shared__ uint32_t s_key[kSortTile], s_val[kSortTile];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // n < 2^24 elements (rt_blas_build / rt_tlas_build) and tiles are whole: 32-bit element indices never wrap
    const uint32_t block_begin = blockIdx.x * tiles_per_block * kSortTile;
    {
        uint32_t unused;
        const uint32_t row_base = block_exclusive_scan_256(row_total[threadIdx.x], s_warp, unused);
        base[threadIdx.x] = row_base + offsets[threadIdx.x * gridDim.x + blockIdx.x];
        tile_count[threadIdx.x] = 0;
    }
    for (uint32_t tile = 0; tile < tiles_per_block; ++tile) {
        const uint32_t tile_begin = block_begin + tile * kSortTile;
        if (tile_begin >= n) break;
        const uint32_t tile_valid = min(uint32_t(kSortTile), n - tile_begin);
        uint32_t key[kSortItems], prev[kSortItems], info[kSortItems];
        // all of the tile's key loads are in flight before the first rank is computed
#pragma unroll
        for (int r = 0; r < kSortItems; ++r) {
            const uint32_t e = warp * 32 * kSortItems + r * 32 + lane;
            key[r] = e < tile_valid ? __ldcs(keys_in + tile_begin + e) : 0xffffffffu;
        }
#pragma unroll
        for (int w = 0; w < kSortWarps; ++w) warp_count[w][threadIdx.x] = 0;
        __syncthreads();  // A: counters are clear; every warp has left the previous tile (its reads of base / tile_start / s_key / s_val)
        base[threadIdx.x] += tile_count[threadIdx.x];  // the previous tile's digit counts (0 before the first tile)
#pragma unroll
        for (int r = 0; r < kSortItems; ++r) {
            const uint32_t e = warp * 32 * kSortItems + r * 32 + lane;
            const bool valid = e < tile_valid;
            const uint32_t d = (key[r] >> shift) & (kRadix - 1);
            // lanes holding the same digit, from one ballot per digit bit: MATCH.ANY resolves one distinct value at a
            // time (~30 per warp here) and eight warps queue for it per scheduler — it was the kernel's bottleneck
            unsigned peers = __ballot_sync(0xffffffffu, valid);
#pragma unroll
            for (int b = 0; b < kRadixBits; ++b) {
                // all ones where this lane's digit has bit b: peers &= bit ? m : ~m becomes ONE three-input logic op
                const uint32_t sel = uint32_t(int32_t(d << (31 - b)) >> 31);
                const unsigned m = __ballot_sync(0xffffffffu, sel != 0u);
                peers &= ~(m ^ sel);
            }
            // The group's first lane bumps the warp's counter with ONE shared-memory atomic.  Its result is not used
            // before the loop ends, so the eight items' ballots and atomics pipeline (a load -> store -> shuffle chain
            // per item was a fifth of the stall samples).  Only this warp touches warp_count[warp]; __syncwarp orders
            // the items' updates of one counter.
            const uint32_t leader = uint32_t(__ffs(peers) - 1) & 31u;
            prev[r] = 0;
            if (valid && uint32_t(lane) == leader) prev[r] = atomicAdd(&warp_count[warp][d], uint32_t(__popc(peers)));
            info[r] = uint32_t(__popc(peers & ((1u << lane) - 1))) | (leader << 8);
            __syncwarp();
        }
#pragma unroll
        for (int r = 0; r < kSortItems; ++r)  // rank inside the warp's part of the tile: group base + position in the group
            info[r] = __shfl_sync(0xffffffffu, prev[r], int(info[r] >> 8)) + (info[r] & 0xffu);
        // the values are not needed before the tile is laid out by digit: their latency falls into the scan phases
        uint32_t val[kSortItems];
#pragma unroll
        for (int r = 0; r < kSortItems; ++r) {
            const uint32_t e = warp * 32 * kSortItems + r * 32 + lane;
            val[r] = IOTA ? tile_begin + e : (e < tile_valid ? __ldcs(vals_in + tile_begin + e) : 0u);
        }
        __syncthreads();  // B: every warp's digit counts are final
        {   // per-digit exclusive prefix over the warps of this tile, then where digit d's run starts inside the sorted tile
            const int d = threadIdx.x;
            uint32_t off = 0;
#pragma unroll
            for (int w = 0; w < kSortWarps; ++w) {
                uint32_t c = warp_count[w][d];
                warp_count[w][d] = off;
                off += c;
            }
            uint32_t incl = off;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            if (lane == 31) s_warp[warp] = incl;
            tile_count[d] = off;
            __syncthreads();  // C
            uint32_t wbase = 0;
#pragma unroll
            for (int w = 0; w < kSortWarps; ++w) wbase += w < warp ? s_warp[w] : 0u;
            tile_start[d] = wbase + incl - off;
        }
        __syncthreads();  // D
        // The tile is first sorted by digit in shared memory, then written out position by position: neighbouring
        // threads hold neighbours of one digit run, so each run leaves as contiguous, sector-filling stores.  Scattering
        // straight from the ranking registers issued 4-byte writes to ~32 different sectors per warp instruction.
#pragma unroll
        for (int r = 0; r < kSortItems; ++r) {
            const uint32_t e = warp * 32 * kSortItems + r * 32 + lane;
            if (e < tile_valid) {
                const uint32_t dd = (key[r] >> shift) & (kRadix - 1);
                const uint32_t local = tile_start[dd] + warp_count[warp][dd] + info[r];
                s_key[local] = key[r];
                s_val[local] = val[r];
            }
        }
        __syncthreads();  // E
#pragma unroll
        for (int r = 0; r < kSortItems; ++r) {
            const uint32_t idx = r * kSortThreads + threadIdx.x;
            if (idx < tile_valid) {
                const uint32_t k = s_key[idx];
                const uint32_t dd = (k >> shift) & (kRadix - 1);
                const uint32_t pos = base[dd] + (idx - tile_start[dd]);
                keys_out[pos] = k;
                vals_out[pos] = s_val[idx];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------ Karras hierarchy
// FL/BuildBVHSplits.hlsli:35-143
struct KarrasDev {
    const uint32_t *codes;
    int n;
    __device__ __forceinline__ int lcp(int a, int b) const {
        if (a < 0 || b < 0 || a >= n || b >= n) return -1;
        uint32_t ca = codes[a], cb = codes[b];
        if (ca != cb) return __clz(int(ca ^ cb));
        return __clz(a ^ b) + 31;
    }
};

// `local` (may be null): local[i] = 1 when every leaf under internal node i lies in one kFitBlock-aligned block of
// sorted slots — such a node's whole subtree is fitted inside one thread block's shared memory by k_fit_local.
#ifndef RT_FIT_BLOCK
#define RT_FIT_BLOCK 256
#endif
constexpr int kFitBlock = RT_FIT_BLOCK;
__global__ void __launch_bounds__(kThreads) k_hierarchy(const uint32_t *codes, uint32_t n, rt_hierarchy_node *nodes, uint8_t *local) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= int(n) - 1) return;
    KarrasDev k{codes, int(n)};
    int d = k.lcp(idx, idx + 1) - k.lcp(idx, idx - 1);
    d = min(max(d, -1), 1);
    int minPrefix = k.lcp(idx, idx - d);
    // 32-bit is enough: n < 2^24 (rt_blas_build), and the search leaves the range — and stops — before maxLength
    // passes 2^27, so idx +- maxLength never wraps
    int maxLength = 2;
    while (true) {
        const int j = idx + maxLength * d;
        const int p = k.lcp(idx, j);  // -1 outside [0, n)
        if (!(p > minPrefix)) break;
        maxLength *= 4;
    }
    int length = 0;
    for (int t = maxLength / 2; t > 0; t /= 2) {
        const int j = idx + (length + t) * d;
        const int p = k.lcp(idx, j);
        if (p > minPrefix) length += t;
    }
    int j = idx + length * d;
    int first = min(idx, j), last = max(idx, j);
    // FindSplit
    int commonPrefix = k.lcp(first, last);
    int split = first, step = last - first;
    do {
        step = (step + 1) >> 1;
        int ns = split + step;
        if (ns < last && k.lcp(first, ns) > commonPrefix) split = ns;
    } while (step > 1);
    uint32_t leafOffset = n - 1;
    uint32_t a = (split == first) ? leafOffset + split : split;
    uint32_t b = (split + 1 == last) ? leafOffset + split + 1 : split + 1;
    nodes[idx].left = a;
    nodes[idx].right = b;
    nodes[a].parent = idx;
    nodes[b].parent = idx;
    if (local) local[idx] = (first / kFitBlock == last / kFitBlock) ? 1 : 0;
}

// ------------------------------------------------------------------------------------------ rearrange
// The 48-byte records are gathered in random order: L2::64B caps the L2 prefetch of each load at 64 bytes.
__device__ __forceinline__ uint4 ld_gather16(const uint4 *p) {
    uint4 v;
    asm volatile("ld.global.L2::64B.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
// FL/RearrangeTriangles.hlsl:18-36: out[dst] = in[perm[dst]]; also emits the packed 48-byte triangle.
__global__ void __launch_bounds__(kThreads) k_rearrange_tris(const rt_packed_tri *recs, const uint32_t *perm, uint32_t n,
                                                             rt_primitive *out_prims, rt_primitive_meta *out_meta, rt_packed_tri *packed) {
    // The block's kThreads gathered records are staged in shared memory and written out as three contiguous runs
    // (packed 48 B, Primitive 40 B, PrimitiveMetaData 12 B per element) with coalesced stores; one thread writing its
    // own 40 + 12 + 48 bytes word by word kept the load/store unit saturated (ncu: lg_throttle) at 4 TB/s.
    __shared__ uint4 s_rec[kThreads * 3];
    const uint32_t b0 = blockIdx.x * kThreads;
    const uint32_t cnt = min(uint32_t(kThreads), n - b0);
    if (threadIdx.x < cnt) {
        const uint32_t src = perm[b0 + threadIdx.x];
        const uint4 *q = reinterpret_cast<const uint4 *>(recs + src);
        // each record is read exactly once
        s_rec[3 * threadIdx.x] = ld_gather16(q), s_rec[3 * threadIdx.x + 1] = ld_gather16(q + 1), s_rec[3 * threadIdx.x + 2] = ld_gather16(q + 2);
    }
    __syncthreads();
    const uint32_t *sw = reinterpret_cast<const uint32_t *>(s_rec);  // 12 words per element
    {   // packed: 3 x 16 bytes per element, 16-byte aligned
        uint4 *dst = reinterpret_cast<uint4 *>(packed + b0);
        for (uint32_t i = threadIdx.x; i < 3 * cnt; i += kThreads) dst[i] = s_rec[i];
    }
    {   // Primitive: {type, 9 floats}; the array starts 16-byte aligned and a full block is 640 x 16 bytes
        uint4 *dst = reinterpret_cast<uint4 *>(reinterpret_cast<uint32_t *>(out_prims) + size_t(b0) * 10);
        const uint32_t words = 10 * cnt;
        auto word = [&](uint32_t w) -> uint32_t {
            const uint32_t e = w / 10, f = w - 10 * e;
            return f == 0 ? ((sw[12 * e + 11] & RT_PACKED_PROCEDURAL) ? RT_PRIMITIVE_TYPE_PROCEDURAL : RT_PRIMITIVE_TYPE_TRIANGLE) : sw[12 * e + f - 1];
        };
        for (uint32_t i = threadIdx.x; 4 * i < words; i += kThreads) {
            const uint32_t w = 4 * i;
            if (w + 4 <= words) {
                dst[i] = make_uint4(word(w), word(w + 1), word(w + 2), word(w + 3));
            } else {
                uint32_t *d = reinterpret_cast<uint32_t *>(dst + i);
                for (uint32_t k = 0; w + k < words; ++k) d[k] = word(w + k);
            }
        }
    }
    {   // PrimitiveMetaData: {geometryContributionToHitGroupIndex, primitiveIndex, geometryFlags}, 4-byte aligned
        uint32_t *dst = reinterpret_cast<uint32_t *>(out_meta) + size_t(b0) * 3;
        for (uint32_t w = threadIdx.x; w < 3 * cnt; w += kThreads) {
            const uint32_t e = w / 3, f = w - 3 * e;
            dst[w] = f == 0 ? sw[12 * e + 10] : (f == 1 ? sw[12 * e + 9] : (sw[12 * e + 11] & ~RT_PACKED_PROCEDURAL));
        }
    }
}

// ------------------------------------------------------------------------------------------ bottom-up fit
// The node rules, written once and used by every fit kernel: leaf box, child-box merge, root record, fitted parent
// (child order, reference node, wide node, 4-wide node) and the 4-wide collapse.
struct Box {
    float c[3], h[3];
};
// AABBtoBoundingBox: FL/RayTracingHelper.hlsli:251-257
__device__ __forceinline__ Box aabb_to_box(const float mn[3], const float mx[3]) {
    Box b;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        b.c[k] = (mn[k] + mx[k]) * 0.5f;
        b.h[k] = mx[k] - b.c[k];
    }
    return b;
}
__device__ __forceinline__ void store_node(rt_aabb_node *nodes, uint32_t i, const Box &b, uint32_t flags, uint32_t right) {
    float4 *p = reinterpret_cast<float4 *>(nodes + i);
    __stcg(p, make_float4(b.c[0], b.c[1], b.c[2], __uint_as_float(flags)));
    __stcg(p + 1, make_float4(b.h[0], b.h[1], b.h[2], __uint_as_float(right)));
}
__device__ __forceinline__ Box load_node_box(const rt_aabb_node *nodes, uint32_t i) {
    const float4 *p = reinterpret_cast<const float4 *>(nodes + i);
    float4 a = __ldcg(p), b = __ldcg(p + 1);
    Box r;
    r.c[0] = a.x, r.c[1] = a.y, r.c[2] = a.z, r.h[0] = b.x, r.h[1] = b.y, r.h[2] = b.z;
    return r;
}

// Leaf box of a sorted primitive from its nine floats: GetBoxDataFromTriangle (RayTracingHelper.hlsli:273-285) with
// AABB_Min_Padding, or for a procedural primitive the AABB {min, max} as given (ComputeLeafAABB, procedural branch,
// FL/BottomLevelComputeAABBs.hlsl:32-40).
__device__ __forceinline__ Box leaf_box(const float *v, bool procedural) {
    float mn[3], mx[3];
    if (procedural) {
#pragma unroll
        for (int k = 0; k < 3; ++k) mn[k] = v[k], mx[k] = v[3 + k];
    } else {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            mn[k] = fminf(fminf(v[k], v[3 + k]), v[6 + k]);
            mx[k] = fmaxf(fmaxf(v[k], v[3 + k]), v[6 + k]);
            mn[k] = fminf(mn[k], mx[k] - 0.001f);  // AABB_Min_Padding
        }
    }
    return aabb_to_box(mn, mx);
}

// GetBoxFromChildBoxes: FL/RayTracingHelper.hlsli:297-307.  `bl` is the child stored on the left: the reference's
// operand order of min / max.
__device__ __forceinline__ Box merge_boxes(const Box &bl, const Box &br) {
    float mn[3], mx[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        mn[k] = fminf(bl.c[k] - bl.h[k], br.c[k] - br.h[k]);
        mx[k] = fmaxf(bl.c[k] + bl.h[k], br.c[k] + br.h[k]);
    }
    return aabb_to_box(mn, mx);
}

__device__ __forceinline__ void store_root(rt_ext_header *ext, const Box &b) {
    ext->root_center[0] = b.c[0], ext->root_center[1] = b.c[1], ext->root_center[2] = b.c[2];
    ext->root_half[0] = b.h[0], ext->root_half[1] = b.h[1], ext->root_half[2] = b.h[2];
}

// A child reference of the traversal section: internal node i is i, leaf node nInternal + slot is LEAF_FLAG | slot.
__device__ __forceinline__ uint32_t node_ref(uint32_t node, uint32_t nInternal) {
    return node >= nInternal ? (RT_NODE_LEAF_FLAG | (node - nInternal)) : node;
}

// The two halves of an empty 4-wide slot: {0, 0, 0, RT_WIDE4_EMPTY}, {-1, -1, -1, 0}.
__device__ __forceinline__ float4 wide4_empty(bool half) {
    return half ? make_float4(-1.0f, -1.0f, -1.0f, 0.0f) : make_float4(0.0f, 0.0f, 0.0f, __uint_as_float(RT_WIDE4_EMPTY));
}

// BVH2 -> BVH4 for the traversal kernels.  A node's 4-wide node starts from its two (ordered) children and opens, twice,
// the internal child with the largest surface area (half-extent product sum); strict >, so the lower slot wins a tie.
// The opened child's left child takes its slot and its right child is appended.  `src` supplies the children: a
// Src::Slot is one child, src.ref / src.half give its reference and half extents, and src.open(s, l, r) the two
// children of the internal child s.  Returns the number of filled slots (2 to 4).
template <class Src>
__device__ __forceinline__ int collapse4(const Src &src, typename Src::Slot s[4]) {
    int cnt = 2;
#pragma unroll
    for (int it = 0; it < 2; ++it) {
        int best = -1;
        float bestArea = -1.0f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (k < cnt && !(src.ref(s[k]) & RT_NODE_LEAF_FLAG)) {
                const float3 h = src.half(s[k]);
                const float a = h.x * h.y + h.y * h.z + h.z * h.x;
                if (a > bestArea) bestArea = a, best = k;
            }
        }
        if (best < 0) break;
        typename Src::Slot opened = s[0], l, r;
#pragma unroll
        for (int k = 1; k < 4; ++k)
            if (k == best) opened = s[k];
        src.open(opened, l, r);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (k == best) s[k] = l;
            if (k == cnt) s[k] = r;
        }
        cnt++;
    }
    return cnt;
}

// collapse4's children from the finished BVH2 wide nodes in global memory.  Loads go through L2: the wide nodes were
// written in the same kernel and published with a fence before the counter that let us fit the parent.
struct WideChildren {
    struct Slot {
        float4 c, h;  // {center, ref}, {half, -}
    };
    const rt_wide_node *wide;
    __device__ __forceinline__ uint32_t ref(const Slot &s) const { return __float_as_uint(s.c.w); }
    __device__ __forceinline__ float3 half(const Slot &s) const { return make_float3(s.h.x, s.h.y, s.h.z); }
    __device__ __forceinline__ void open(const Slot &s, Slot &l, Slot &r) const {
        const float4 *w = reinterpret_cast<const float4 *>(wide + ref(s));
        const float4 w0 = __ldcg(w), w1 = __ldcg(w + 1), w2 = __ldcg(w + 2), w3 = __ldcg(w + 3);
        l.c = w0, l.h = w1;
        r.c = make_float4(w2.x, w2.y, w2.z, w1.w), r.h = w3;
    }
};

// The fit of one parent from its children l, r (Karras order) with subtree sizes lc, rc and boxes bl, br: the child
// order, the reference node, the BVH2 wide node (both child boxes live in the parent), the 4-wide node when WIDE4 and,
// for the root, the root record.  REORDER: smaller subtree on the left, ties keep the Karras order (on equal counts the
// reference is arrival-order dependent, pinned here).  A refit (PERFORM_UPDATE) passes false: the topology and the child
// order are those of the build it updates.  Every subtree below `parent` is complete and published (fence + counter).
// Returns the parent's box.
template <bool REORDER, bool WIDE4>
__device__ __forceinline__ Box fit_parent(uint32_t parent, uint32_t l, uint32_t r, uint32_t lc, uint32_t rc, Box bl, Box br,
                                          uint32_t nInternal, rt_aabb_node *nodes, rt_wide_node *wide, rt_wide4_node *wide4,
                                          rt_ext_header *ext) {
    if (REORDER && rc < lc) {
        uint32_t t = l; l = r; r = t;
        Box tb = bl; bl = br; br = tb;
    }
    const Box box = merge_boxes(bl, br);
    store_node(nodes, parent, box, l & 0x00ffffffu, r);
    const uint32_t lref = node_ref(l, nInternal), rref = node_ref(r, nInternal);
    float4 *w = reinterpret_cast<float4 *>(wide + parent);
    w[0] = make_float4(bl.c[0], bl.c[1], bl.c[2], __uint_as_float(lref));
    w[1] = make_float4(bl.h[0], bl.h[1], bl.h[2], __uint_as_float(rref));
    w[2] = make_float4(br.c[0], br.c[1], br.c[2], 0.0f);
    w[3] = make_float4(br.h[0], br.h[1], br.h[2], 0.0f);
    if (WIDE4) {
        WideChildren::Slot s[4];
        s[0].c = make_float4(bl.c[0], bl.c[1], bl.c[2], __uint_as_float(lref)), s[0].h = make_float4(bl.h[0], bl.h[1], bl.h[2], 0.0f);
        s[1].c = make_float4(br.c[0], br.c[1], br.c[2], __uint_as_float(rref)), s[1].h = make_float4(br.h[0], br.h[1], br.h[2], 0.0f);
        const int cnt = collapse4(WideChildren{wide}, s);
        float4 *o = reinterpret_cast<float4 *>(wide4 + parent);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            o[2 * k] = k < cnt ? s[k].c : wide4_empty(false);
            o[2 * k + 1] = k < cnt ? make_float4(s[k].h.x, s[k].h.y, s[k].h.z, 0.0f) : wide4_empty(true);
        }
    }
    if (parent == 0) store_root(ext, box);
    return box;
}

// FL/ComputeAABBs.hlsli:69-175, through global memory: one thread carries a fitted node (its box and subtree size) up
// the tree; the second child to arrive at a parent (atomic counter carrying subtree sizes) fits the parent.
// UPDATE (PERFORM_UPDATE, ComputeAABBs.hlsli:38-67): the topology is the one already in `nodes` — children from each
// node's {flags, right} words, parents from the cached parent array — and only the boxes are re-fitted.
// WIDE4: write the 4-wide node of every parent fitted (k_fit_exits); k_fit leaves them to k_collapse4.
template <bool UPDATE, bool WIDE4>
__device__ __forceinline__ void climb(uint32_t node, uint32_t count, Box box, uint32_t nInternal, const rt_hierarchy_node *hier,
                                      const uint32_t *parents, uint32_t *counters, rt_aabb_node *nodes, rt_wide_node *wide,
                                      rt_wide4_node *wide4, rt_ext_header *ext) {
    const uint32_t *hw = reinterpret_cast<const uint32_t *>(hier);
    while (true) {
        uint32_t parent, l = 0, r = 0;
        if (UPDATE) {
            parent = parents[node];
        } else {
            parent = __ldg(hw + 3 * size_t(node)) & ~treelet::kCollapseBit;
            l = __ldg(hw + 3 * size_t(parent) + 1), r = __ldg(hw + 3 * size_t(parent) + 2);
        }
        __threadfence();
        const uint32_t other = atomicAdd(&counters[parent], count);
        if (other == 0) return;  // first to arrive: the sibling will fit the parent
        __threadfence();
        if (UPDATE) l = nodes[parent].flags & 0x00ffffffu, r = nodes[parent].right;
        const bool isLeft = (l == node);
        const Box sb = load_node_box(nodes, isLeft ? r : l);
        box = fit_parent<!UPDATE, WIDE4>(parent, l, r, isLeft ? count : other, isLeft ? other : count, isLeft ? box : sb, isLeft ? sb : box,
                                         nInternal, nodes, wide, wide4, ext);
        if (parent == 0) return;
        count += other;
        node = parent;
    }
}

// One thread per leaf: the leaf box, then the global climb.  TLAS builds and updates, and PERFORM_UPDATE refits of a BLAS;
// their 4-wide nodes are written afterwards by k_collapse4.
// TOP = false: leaf box from the sorted primitive.  TOP = true: leaf box = load-order instance box permuted by `perm`.
template <bool TOP, bool UPDATE>
__global__ void __launch_bounds__(kThreads) k_fit(uint32_t n, const rt_hierarchy_node *hier, uint32_t *counters,
                                                  rt_aabb_node *nodes, const rt_primitive *sorted_prims,
                                                  const rt_aabb_node *inst_boxes, const uint32_t *perm,
                                                  rt_wide_node *wide, rt_ext_header *ext, const uint32_t *parents) {
    uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= n) return;
    const uint32_t nInternal = n - 1;
    Box box;
    uint32_t leafFlags = slot | RT_NODE_LEAF_FLAG;
    if (TOP) {
        const rt_aabb_node &s = inst_boxes[perm[slot]];
        box.c[0] = s.center[0], box.c[1] = s.center[1], box.c[2] = s.center[2];
        box.h[0] = s.halfDim[0], box.h[1] = s.halfDim[1], box.h[2] = s.halfDim[2];
    } else {
        const bool procedural = *reinterpret_cast<const uint32_t *>(sorted_prims + slot) == RT_PRIMITIVE_TYPE_PROCEDURAL;
        box = leaf_box(sorted_prims[slot].v, procedural);
        if (procedural) leafFlags |= RT_NODE_PROCEDURAL_FLAG;
    }
    store_node(nodes, nInternal + slot, box, leafFlags, 1u);
    if (n == 1) store_root(ext, box);
    else climb<UPDATE, false>(nInternal + slot, 1u, box, nInternal, hier, parents, counters, nodes, wide, nullptr, ext);
}

// BVH2 -> BVH4 after k_fit: thread i collapses node i, reading the child boxes straight from the finished BVH2 wide nodes.
__global__ void __launch_bounds__(kThreads) k_collapse4(const rt_wide_node *wide, uint32_t n_internal, rt_wide4_node *wide4) {
    // the block's kThreads x 128-byte nodes leave through shared memory as one contiguous run of 16-byte stores; slot
    // k of thread t sits at t * 8 + (k ^ (t & 7)) so that neither side has bank conflicts
    __shared__ float4 s_out[kThreads * 8];
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_internal) {
        const float4 *w = reinterpret_cast<const float4 *>(wide + i);
        const float4 w0 = w[0], w1 = w[1], w2 = w[2], w3 = w[3];
        WideChildren::Slot s[4];
        s[0].c = w0, s[0].h = w1;
        s[1].c = make_float4(w2.x, w2.y, w2.z, w1.w), s[1].h = w3;
        const int cnt = collapse4(WideChildren{wide}, s);
        float4 *o = s_out + threadIdx.x * 8;
        const int sw = threadIdx.x & 7;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            o[(2 * k) ^ sw] = k < cnt ? s[k].c : wide4_empty(false);
            o[(2 * k + 1) ^ sw] = k < cnt ? make_float4(s[k].h.x, s[k].h.y, s[k].h.z, 0.0f) : wide4_empty(true);
        }
    }
    __syncthreads();
    const uint32_t b0 = blockIdx.x * blockDim.x;
    const uint32_t valid = 8 * min(uint32_t(kThreads), n_internal - b0);
    float4 *dst = reinterpret_cast<float4 *>(wide4 + b0);
    for (uint32_t g = threadIdx.x; g < valid; g += kThreads) {
        const uint32_t t = g >> 3, e = g & 7;
        dst[g] = s_out[t * 8 + (e ^ (t & 7))];
    }
}

// ------------------------------------------------------------------------------------------ block fit
// A full bottom-level build fits the lower levels of the tree inside the thread block.  A block owns kFitBlock
// consecutive sorted slots and works in rounds over a shared-memory ready queue: a node enters the queue when its second
// child has been fitted, and the nodes of a round are handed to consecutive threads, so the warps stay dense where the
// one-thread-per-leaf climb runs at 6-7 of 32 lanes (ncu) and pays a global atomic plus two device-wide fences per
// level.  Child boxes and subtree sizes are exchanged through shared memory.  Nodes whose parent lies outside the block
// leave through an exit list and finish with a global climb.  Results (reference nodes, wide nodes, 4-wide nodes, child
// order) are those of the global climb, bit for bit: the child order depends only on the subtree sizes and the Karras
// order, never on who arrives first.  Two kernels share this structure and differ in where the topology comes from:
// k_fit_local reads the hierarchy array, k_lbvh_fit grows the Karras hierarchy from the Morton codes as it goes.
//
// Shared index of a node: leaf -> slot - b0 in [0, B); internal node i -> B + i - b0 in [B, 2B).
constexpr size_t kFitLocalDynSmem = sizeof(float) * 6 * 2 * kFitBlock + sizeof(uint32_t) * 4 * kFitBlock;
__device__ __forceinline__ uint32_t shared_index(uint32_t node, uint32_t nInternal, uint32_t b0) {
    return node >= nInternal ? node - nInternal - b0 : kFitBlock + node - b0;
}
__device__ __forceinline__ Box shared_box(const float (*s_box)[6], uint32_t si) {
    Box b;
#pragma unroll
    for (int k = 0; k < 3; ++k) b.c[k] = s_box[si][k], b.h[k] = s_box[si][3 + k];
    return b;
}
__device__ __forceinline__ void put_shared_box(float (*s_box)[6], uint32_t si, const Box &b) {
#pragma unroll
    for (int k = 0; k < 3; ++k) s_box[si][k] = b.c[k], s_box[si][3 + k] = b.h[k];
}

// This thread's leaf into shared memory: the box from the 48-byte packed record k_rearrange_tris wrote next to the
// reference-format Primitive (same nine floats through three aligned 16-byte loads instead of ten 4-byte loads at
// stride 40), and whether it is procedural.  Returns the box.
__device__ __forceinline__ Box stage_leaf(float4 q0, float4 q1, float4 q2, float (*s_box)[6], uint8_t *s_proc) {
    const float v[9] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x};
    const bool procedural = (__float_as_uint(q2.w) & RT_PACKED_PROCEDURAL) != 0;
    const Box box = leaf_box(v, procedural);
    put_shared_box(s_box, threadIdx.x, box);
    s_proc[threadIdx.x] = procedural ? 1 : 0;
    return box;
}

// Rounds.  fit_ready(entry, next) fits one ready entry of s_queue[cur] and queues what it readies in s_queue[next].  The
// number of ready nodes never grows (a node fitted in one round readies at most its one parent), so once a round fits in
// a warp the rest of the chain is run by warp 0 alone with warp barriers ...
template <class Entry, class FitReady>
__device__ __forceinline__ void block_fit_rounds(uint32_t *s_qn, Entry (*s_queue)[kFitBlock], const FitReady &fit_ready, const float (*s_box)[6],
                                                 const uint8_t *s_proc, uint32_t b0, uint32_t nInternal, uint32_t cntLeaf, rt_aabb_node *nodes) {
    int cur = 0;
    for (; s_qn[cur] > 32; cur ^= 1) {  // block-uniform: s_qn[cur] is stable between the two barriers
        if (threadIdx.x < s_qn[cur]) fit_ready(s_queue[cur][threadIdx.x], cur ^ 1);
        __syncthreads();
        if (threadIdx.x == 0) s_qn[cur] = 0;
        __syncthreads();
    }
    __syncthreads();  // every warp has read the exit condition before warp 0 starts rewriting the queue counters
    if (threadIdx.x < 32) {
        for (;; cur ^= 1) {
            const uint32_t q = s_qn[cur];
            if (q == 0) break;
            if (threadIdx.x < q) fit_ready(s_queue[cur][threadIdx.x], cur ^ 1);
            __syncwarp();
            if (threadIdx.x == 0) s_qn[cur] = 0;
            __syncwarp();
        }
    } else {
        // ... while the other warps write the leaf nodes {center, slot | flags}, {halfDim, 1}, which no round touches
        // (a third of k_fit_local's stall samples were warps waiting at the barrier below for warp 0's tail)
        float4 *dst = reinterpret_cast<float4 *>(nodes + nInternal + b0);
        for (uint32_t g = threadIdx.x - 32; g < 2 * cntLeaf; g += kFitBlock - 32) {
            const uint32_t e = g >> 1;
            const float *bx = s_box[e];
            if (g & 1) dst[g] = make_float4(bx[3], bx[4], bx[5], __uint_as_float(1u));
            else dst[g] = make_float4(bx[0], bx[1], bx[2], __uint_as_float((b0 + e) | RT_NODE_LEAF_FLAG | (s_proc[e] ? RT_NODE_PROCEDURAL_FLAG : 0u)));
        }
    }
    __syncthreads();
}

// collapse4's children from the block's shared memory: the boxes in s_box, the children of a node the block fitted
// from `children` (see block_write_out).
template <class Children>
struct SharedChildren {
    struct Slot {
        uint32_t ref, si;  // traversal-section reference, shared index
    };
    const float (*s_box)[6];
    Children children;
    uint32_t nInternal, b0;
    __device__ __forceinline__ uint32_t ref(const Slot &s) const { return s.ref; }
    __device__ __forceinline__ float3 half(const Slot &s) const { return make_float3(s_box[s.si][3], s_box[s.si][4], s_box[s.si][5]); }
    __device__ __forceinline__ Slot slot(uint32_t node) const { return {node_ref(node, nInternal), shared_index(node, nInternal, b0)}; }
    __device__ __forceinline__ void open(const Slot &s, Slot &l, Slot &r) const {
        uint32_t a, b;
        children(s.ref - b0, a, b);
        l = slot(a), r = slot(b);
    }
};

// Write-out.  Everything the block fitted is described by shared memory (boxes, children), so the reference nodes, the
// wide nodes and the 4-wide nodes leave as contiguous runs of 16-byte stores — the rounds issued none.  (One thread
// storing its own node's 32 + 64 bytes touched 32 sectors per warp instruction.)  fitted(e): the block fitted internal
// node b0 + e; children(e, l, r): that node's children, in their final order.  s_w4 receives the 4-wide child lists.
template <class Fitted, class Children>
__device__ __forceinline__ void block_write_out(uint32_t b0, uint32_t nInternal, uint32_t cntInt, const float (*s_box)[6], uint32_t (*s_w4)[4],
                                                const Fitted &fitted, const Children &children, rt_aabb_node *nodes, rt_wide_node *wide,
                                                rt_wide4_node *wide4, rt_ext_header *ext) {
    {   // internal reference nodes: {center, left}, {halfDim, right}
        float4 *dst = reinterpret_cast<float4 *>(nodes + b0);
        for (uint32_t g = threadIdx.x; g < 2 * cntInt; g += kFitBlock) {
            const uint32_t e = g >> 1;
            if (!fitted(e)) continue;
            uint32_t l, r;
            children(e, l, r);
            const float *bx = s_box[kFitBlock + e];
            if (g & 1) dst[g] = make_float4(bx[3], bx[4], bx[5], __uint_as_float(r));
            else dst[g] = make_float4(bx[0], bx[1], bx[2], __uint_as_float(l & 0x00ffffffu));
        }
    }
    {   // wide nodes: both child boxes and child references
        float4 *dst = reinterpret_cast<float4 *>(wide + b0);
        for (uint32_t g = threadIdx.x; g < 4 * cntInt; g += kFitBlock) {
            const uint32_t e = g >> 2, part = g & 3;
            if (!fitted(e)) continue;
            uint32_t l, r;
            children(e, l, r);
            const float *bx = s_box[shared_index(part < 2 ? l : r, nInternal, b0)];
            const uint32_t w = part == 0 ? node_ref(l, nInternal) : (part == 1 ? node_ref(r, nInternal) : 0u);
            if (part & 1) dst[g] = make_float4(bx[3], bx[4], bx[5], __uint_as_float(w));
            else dst[g] = make_float4(bx[0], bx[1], bx[2], __uint_as_float(w));
        }
    }
    // 4-wide nodes, straight from shared memory: the child lists first ...
    if (threadIdx.x < cntInt && fitted(threadIdx.x)) {
        const SharedChildren<Children> src{s_box, children, nInternal, b0};
        typename SharedChildren<Children>::Slot s[4];
        uint32_t l, r;
        children(threadIdx.x, l, r);
        s[0] = src.slot(l), s[1] = src.slot(r);
        const int cnt = collapse4(src, s);
#pragma unroll
        for (int k = 0; k < 4; ++k) s_w4[threadIdx.x][k] = k < cnt ? s[k].ref : RT_WIDE4_EMPTY;
    }
    __syncthreads();
    {   // ... then the 128-byte nodes as one contiguous run
        float4 *dst = reinterpret_cast<float4 *>(wide4 + b0);
        for (uint32_t g = threadIdx.x; g < 8 * cntInt; g += kFitBlock) {
            const uint32_t e = g >> 3, part = g & 7;
            if (!fitted(e)) continue;
            const uint32_t ref = s_w4[e][part >> 1];
            if (ref == RT_WIDE4_EMPTY) {
                dst[g] = wide4_empty(part & 1);
            } else {
                const float *bx = s_box[(ref & RT_NODE_LEAF_FLAG) ? (ref & 0x00ffffffu) - b0 : kFitBlock + ref - b0];
                dst[g] = (part & 1) ? make_float4(bx[3], bx[4], bx[5], 0.0f) : make_float4(bx[0], bx[1], bx[2], __uint_as_float(ref));
            }
        }
    }
    if (b0 == 0 && nInternal > 0 && threadIdx.x == 0 && fitted(0)) store_root(ext, shared_box(s_box, kFitBlock));  // the whole tree was local
}

// The block fit driven by the hierarchy array: a parent flagged `local` (k_hierarchy; kept valid by k_treelet_reorder)
// has its whole subtree among the block's slots.  Full BLAS builds with treelet passes or ALLOW_UPDATE.
__global__ void __launch_bounds__(kFitBlock) k_fit_local(uint32_t n, const rt_hierarchy_node *hier, uint32_t *counters, rt_aabb_node *nodes,
                                                         const rt_packed_tri *packed, rt_wide_node *wide, rt_wide4_node *wide4,
                                                         rt_ext_header *ext, const uint8_t *local, uint32_t *exit_nodes,
                                                         uint16_t *exit_sizes) {
    extern __shared__ __align__(16) uint8_t s_dyn[];  // kFitLocalDynSmem bytes: the boxes and the 4-wide child lists
    float(*s_box)[6] = reinterpret_cast<float(*)[6]>(s_dyn);
    uint32_t(*s_w4)[4] = reinterpret_cast<uint32_t(*)[4]>(s_dyn + sizeof(float) * 6 * 2 * kFitBlock);
    __shared__ uint32_t s_size[2 * kFitBlock];
    __shared__ uint32_t s_arrive[kFitBlock];     // children fitted so far; 2 = this node was fitted by this block
    __shared__ uint32_t s_queue[2][kFitBlock];  // ready internal nodes of this / the next round
    __shared__ uint32_t s_exit[kFitBlock];       // fitted nodes whose parent is not local (roots of disjoint subtrees)
    __shared__ uint32_t s_qn[2], s_en, s_base;
    // the hierarchy records and flags of this block's internal nodes (a local node's index lies in [b0, b0 + B)),
    // fetched once and coalesced: the rounds below run out of shared memory alone
    __shared__ uint32_t s_hier[3 * kFitBlock];
    __shared__ uint8_t s_local[kFitBlock], s_proc[kFitBlock];
    const uint32_t b0 = blockIdx.x * kFitBlock;
    const uint32_t nInternal = n - 1;
    const uint32_t *hw = reinterpret_cast<const uint32_t *>(hier);
    s_arrive[threadIdx.x] = 0;
    if (threadIdx.x < 2) s_qn[threadIdx.x] = 0;
    if (threadIdx.x == 2) s_en = 0;
    // every global load of the block is issued before the first barrier: one DRAM latency, not two
    const uint32_t slot = b0 + threadIdx.x;
    const uint32_t cntLeaf = min(uint32_t(kFitBlock), n - b0);
    const uint32_t cntInt = b0 < nInternal ? min(uint32_t(kFitBlock), nInternal - b0) : 0u;
    float4 q0 = make_float4(0, 0, 0, 0), q1 = q0, q2 = q0;
    uint32_t leafParent = 0;
    if (slot < n) {
        const float4 *q = reinterpret_cast<const float4 *>(packed + slot);
        q0 = q[0], q1 = q[1], q2 = q[2];
        if (n > 1) leafParent = __ldg(hw + 3 * size_t(nInternal + slot)) & ~treelet::kCollapseBit;
    }
    for (uint32_t i = threadIdx.x; i < 3 * cntInt; i += kFitBlock) s_hier[i] = __ldg(hw + 3 * size_t(b0) + i);
    s_local[threadIdx.x] = threadIdx.x < cntInt ? __ldg(local + b0 + threadIdx.x) : uint8_t(0);
    __syncthreads();
    // a fitted node reports to its parent: the second arrival makes the parent ready
    auto report = [&](uint32_t node, uint32_t parent, int next) {
        if (parent - b0 < uint32_t(kFitBlock) && s_local[parent - b0]) {
            if (atomicAdd(&s_arrive[parent - b0], 1u) == 1u) s_queue[next][atomicAdd(&s_qn[next], 1u)] = parent;
        } else {
            s_exit[atomicAdd(&s_en, 1u)] = node;
        }
    };
    if (slot < n) {
        const Box box = stage_leaf(q0, q1, q2, s_box, s_proc);
        s_size[threadIdx.x] = 1;
        if (n == 1) store_root(ext, box);
        else report(nInternal + slot, leafParent, 0);
    }
    __syncthreads();
    // One ready node: its box from its children's shared boxes, published in shared memory; nothing is stored to
    // global memory here.
    auto fit_ready = [&](uint32_t p, int next) {
        const uint32_t *rec = s_hier + 3 * (p - b0);
        const uint32_t up = rec[0] & ~treelet::kCollapseBit;
        uint32_t li = shared_index(rec[1], nInternal, b0), ri = shared_index(rec[2], nInternal, b0);
        if (s_size[ri] < s_size[li]) {  // smaller subtree on the left; ties keep the Karras order
            const uint32_t t = li; li = ri; ri = t;
        }
        const uint32_t pi = kFitBlock + p - b0;
        put_shared_box(s_box, pi, merge_boxes(shared_box(s_box, li), shared_box(s_box, ri)));
        s_size[pi] = s_size[li] + s_size[ri];
        if (p != 0) report(p, up, next);
    };
    block_fit_rounds(s_qn, s_queue, fit_ready, s_box, s_proc, b0, nInternal, cntLeaf, nodes);
    const uint32_t en = s_en;
    if (threadIdx.x == 0 && en) s_base = atomicAdd(&counters[nInternal], en);  // counters[n-1] is no node's counter
    // The child order of a fitted node is applied once, in place, to the shared copy of the hierarchy records, so that
    // the write-out (which visits a node once per 16-byte store) just reads {left, right}.
    if (threadIdx.x < cntInt && s_arrive[threadIdx.x] == 2) {
        const uint32_t l = s_hier[3 * threadIdx.x + 1], r = s_hier[3 * threadIdx.x + 2];
        if (s_size[shared_index(r, nInternal, b0)] < s_size[shared_index(l, nInternal, b0)]) s_hier[3 * threadIdx.x + 1] = r, s_hier[3 * threadIdx.x + 2] = l;
    }
    __syncthreads();
    block_write_out(
        b0, nInternal, cntInt, s_box, s_w4, [&](uint32_t e) { return s_arrive[e] == 2; },
        [&](uint32_t e, uint32_t &l, uint32_t &r) { l = s_hier[3 * e + 1], r = s_hier[3 * e + 2]; }, nodes, wide, wide4, ext);
    __syncthreads();
    // the nodes whose parent's subtree crosses the block boundary continue in k_fit_exits
    if (threadIdx.x < en) {
        const uint32_t node = s_exit[threadIdx.x];
        exit_nodes[s_base + threadIdx.x] = node;
        exit_sizes[s_base + threadIdx.x] = uint16_t(s_size[shared_index(node, nInternal, b0)]);
    }
}

// Second half of k_fit_local: one thread per exit-list entry climbs through global memory.
__global__ void __launch_bounds__(kThreads) k_fit_exits(uint32_t n, const rt_hierarchy_node *hier, uint32_t *counters, rt_aabb_node *nodes,
                                                        rt_wide_node *wide, rt_wide4_node *wide4, rt_ext_header *ext,
                                                        const uint32_t *exit_nodes, const uint16_t *exit_sizes) {
    const uint32_t nInternal = n - 1;
    const uint32_t entries = __ldcg(&counters[nInternal]);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < entries; i += gridDim.x * blockDim.x) {  // grid: see k_lbvh_exits
        const uint32_t node = exit_nodes[i];
        climb<false, true>(node, exit_sizes[i], load_node_box(nodes, node), nInternal, hier, nullptr, counters, nodes, wide, wide4, ext);
    }
}

// ------------------------------------------------------------------------------------------ hierarchy + fit in one pass
// PREFER_FAST_BUILD (no treelet pass, no update caches): FL/BuildBVHSplits.hlsli:35-143 and FL/ComputeAABBs.hlsli:69-175
// as ONE bottom-up sweep.  The reference's hierarchy is the binary radix tree of the sorted keys under its delta
// (common prefix of the Morton codes, ties by `clz(i ^ j) + 31`); that tree is unique, and it can be grown from the leaves
// (Apetrei 2014): a finished node covering the sorted slots [lo, hi] is the LEFT child of the node that splits at hi when
// delta(hi, hi+1) > delta(lo-1, lo) — it shares the longer prefix with its right neighbour — and otherwise the RIGHT child
// of the node that splits at lo-1 (delta = -1 outside [0, n), so the range [0, n-1] is the root; the two deltas are never
// equal for distinct keys).  Karras' numbering follows from the same decision: a left child is internal node `hi`, a right
// child internal node `lo`, the root node 0 (BuildBVHSplits.hlsli:128-141: children of a split at s are s and s+1).
// So there is no search (k_hierarchy runs ~20 divergent binary-search steps per node), no hierarchy array and no memset
// of it.  Subtree size = hi - lo + 1.  The block structure is k_fit_local's: a block owns kFitBlock sorted slots, meets
// its children in shared memory at the SPLIT position (both neighbours of a split inside the block), fits round by
// round, writes reference nodes, wide nodes and 4-wide nodes once and coalesced.  Nodes whose parent's split is on a
// block boundary, or whose sibling reaches out of the block, leave through an exit list and finish in k_lbvh_exits.
__device__ __forceinline__ int lbvh_delta(const uint32_t *codes, uint32_t n, uint32_t i) {  // delta(i, i+1); i = 0xffffffff is "-1"
    if (i >= n - 1) return -1;
    const uint32_t a = __ldg(codes + i), b = __ldg(codes + i + 1);
    return a != b ? __clz(int(a ^ b)) : __clz(int(i ^ (i + 1))) + 31;
}

constexpr uint32_t kNoKid = 0xffffffffu;
__global__ void __launch_bounds__(kFitBlock) k_lbvh_fit(uint32_t n, const uint32_t *codes, rt_aabb_node *nodes,
                                                        const rt_packed_tri *packed, rt_wide_node *wide, rt_wide4_node *wide4,
                                                        rt_ext_header *ext, uint32_t *exit_count, uint32_t *exit_nodes, uint32_t *exit_lo,
                                                        uint32_t *exit_hi) {
    constexpr int B = kFitBlock;
    extern __shared__ __align__(16) uint8_t s_dyn[];  // kFitLocalDynSmem bytes: the boxes and the 4-wide child lists
    float(*s_box)[6] = reinterpret_cast<float(*)[6]>(s_dyn);
    uint32_t(*s_w4)[4] = reinterpret_cast<uint32_t(*)[4]>(s_dyn + sizeof(float) * 6 * 2 * B);
    __shared__ uint32_t s_kid[2][B];     // by split - b0: the node that arrived from the left / from the right
    __shared__ uint16_t s_bound[2][B];   // by split - b0: lo - b0 of the left arrival / hi - b0 of the right arrival
    __shared__ uint32_t s_arrive[B];     // by split - b0: arrivals
    __shared__ uint32_t s_left[B], s_right[B];  // by id - b0: children of a node fitted here, smaller subtree first
    __shared__ uint32_t s_range[B];      // by id - b0: (lo - b0) | (hi - b0) << 16
    __shared__ uint8_t s_fitted[B], s_proc[B];
    __shared__ int8_t s_delta[B + 1];    // s_delta[k] = delta(b0 - 1 + k, b0 + k)
    __shared__ uint16_t s_queue[2][B];   // ready splits (minus b0) of this / the next round
    __shared__ uint32_t s_exit[B];       // finished nodes that continue through global memory
    __shared__ uint32_t s_qn[2], s_en, s_base;
    const uint32_t b0 = blockIdx.x * B;
    const uint32_t nInternal = n - 1;
    const uint32_t slot = b0 + threadIdx.x;
    const uint32_t cntLeaf = min(uint32_t(B), n - b0);
    const uint32_t cntInt = b0 < nInternal ? min(uint32_t(B), nInternal - b0) : 0u;
    s_arrive[threadIdx.x] = 0;
    s_kid[0][threadIdx.x] = kNoKid, s_kid[1][threadIdx.x] = kNoKid;
    s_fitted[threadIdx.x] = 0;
    if (threadIdx.x < 2) s_qn[threadIdx.x] = 0;
    if (threadIdx.x == 2) s_en = 0;
    float4 q0 = make_float4(0, 0, 0, 0), q1 = q0, q2 = q0;
    if (slot < n) {
        const float4 *q = reinterpret_cast<const float4 *>(packed + slot);
        q0 = q[0], q1 = q[1], q2 = q[2];
        s_delta[threadIdx.x + 1] = int8_t(lbvh_delta(codes, n, slot));
        if (threadIdx.x == 0) s_delta[0] = int8_t(lbvh_delta(codes, n, slot - 1));  // slot 0: index "-1"
    }
    // a finished node [lo, hi] (global slots, inside this block) reports to the split it hangs on
    auto report = [&](uint32_t node, uint32_t lo, uint32_t hi, int next) {
        const bool goRight = s_delta[hi - b0 + 1] > s_delta[lo - b0];
        const uint32_t g = (goRight ? hi : lo - 1) - b0;  // lo - 1 - b0 wraps for a split left of the block
        if (g < uint32_t(B - 1)) {                        // slots g and g + 1 both belong to this block
            const int side = goRight ? 0 : 1;
            s_kid[side][g] = node;
            s_bound[side][g] = uint16_t((goRight ? lo : hi) - b0);
            if (atomicAdd(&s_arrive[g], 1u) == 1u) s_queue[next][atomicAdd(&s_qn[next], 1u)] = uint16_t(g);
        } else {
            s_exit[atomicAdd(&s_en, 1u)] = node;
        }
    };
    if (slot < n) {
        const Box box = stage_leaf(q0, q1, q2, s_box, s_proc);
        if (n == 1) store_root(ext, box);
    }
    __syncthreads();  // s_delta, the cleared slots
    if (slot < n && n > 1) report(nInternal + slot, slot, slot, 0);
    __syncthreads();
    // One ready split: both children are in shared memory.
    auto fit_ready = [&](uint32_t g, int next) {
        const uint32_t lo = b0 + s_bound[0][g], hi = b0 + s_bound[1][g], split = b0 + g;
        uint32_t a = s_kid[0][g], b = s_kid[1][g];
        if (hi - split < split - lo + 1) {  // smaller subtree on the left; ties keep the Karras order
            const uint32_t t = a; a = b; b = t;
        }
        const Box box = merge_boxes(shared_box(s_box, shared_index(a, nInternal, b0)), shared_box(s_box, shared_index(b, nInternal, b0)));
        const bool root = lo == 0 && hi == n - 1;
        const uint32_t id = root ? 0u : (s_delta[hi - b0 + 1] > s_delta[lo - b0] ? hi : lo);
        const uint32_t e = id - b0;
        put_shared_box(s_box, B + e, box);
        s_left[e] = a, s_right[e] = b;
        s_range[e] = (lo - b0) | ((hi - b0) << 16);
        s_fitted[e] = 1;
        if (!root) report(id, lo, hi, next);
    };
    block_fit_rounds(s_qn, s_queue, fit_ready, s_box, s_proc, b0, nInternal, cntLeaf, nodes);
    // a node still waiting at a split is one whose sibling reaches out of the block
    if (s_arrive[threadIdx.x] == 1u) {
        const uint32_t l = s_kid[0][threadIdx.x];
        s_exit[atomicAdd(&s_en, 1u)] = l != kNoKid ? l : s_kid[1][threadIdx.x];
    }
    __syncthreads();
    const uint32_t en = s_en;
    block_write_out(
        b0, nInternal, cntInt, s_box, s_w4, [&](uint32_t e) { return s_fitted[e] != 0; },
        [&](uint32_t e, uint32_t &l, uint32_t &r) { l = s_left[e], r = s_right[e]; }, nodes, wide, wide4, ext);
    // the nodes that leave the block continue in k_lbvh_exits: {node, lo, hi}
    if (threadIdx.x == 0 && en) s_base = atomicAdd(exit_count, en);
    __syncthreads();
    if (threadIdx.x < en) {
        const uint32_t node = s_exit[threadIdx.x];
        uint32_t lo, hi;
        if (node >= nInternal) {
            lo = hi = node - nInternal;
        } else {
            const uint32_t rg = s_range[node - b0];
            lo = b0 + (rg & 0xffffu), hi = b0 + (rg >> 16);
        }
        exit_nodes[s_base + threadIdx.x] = node;
        exit_lo[s_base + threadIdx.x] = lo;
        exit_hi[s_base + threadIdx.x] = hi;
    }
}

// Second half of k_lbvh_fit: one thread per exit-list entry climbs through global memory.  A node [lo, hi] meets its
// sibling at g_slot[split]: one 64-bit exchange carries {node + 1, far end of the range}; the second arrival fits the
// parent (its Karras index and its own parent's split follow from the two deltas at the ends of the merged range).
// Kept out of k_lbvh_fit on purpose: with the climb inside, a block stays resident until its longest chain of
// dependent atomics ends (tens of microseconds against ~10 for the block's own work) and the kernel took 1.63 ms
// instead of 0.7 + 0.2 (10 M triangles).
__global__ void __launch_bounds__(kThreads) k_lbvh_exits(uint32_t n, const uint32_t *codes, unsigned long long *g_slot, rt_aabb_node *nodes,
                                                         rt_wide_node *wide, rt_wide4_node *wide4, rt_ext_header *ext,
                                                         const uint32_t *exit_count, const uint32_t *exit_nodes, const uint32_t *exit_lo,
                                                         const uint32_t *exit_hi) {
    const uint32_t nInternal = n - 1;
    // The list holds a few entries per fit block (~8 of 256 slots); the grid is sized for one entry per 8 leaves and strides
    // over longer lists.  (One thread per LEAF meant 39 000 blocks at 10 M triangles of which 1 200 had work.)
    const uint32_t count = __ldcg(exit_count);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    uint32_t node = exit_nodes[i], lo = exit_lo[i], hi = exit_hi[i];
    Box box = load_node_box(nodes, node);
    bool goRight = lbvh_delta(codes, n, hi) > lbvh_delta(codes, n, lo - 1);
    while (true) {
        const uint32_t split = goRight ? hi : lo - 1;
        const unsigned long long mine = (static_cast<unsigned long long>(goRight ? lo : hi) << 32) | (node + 1u);
        __threadfence();
        const unsigned long long other = atomicExch(g_slot + split, mine);
        if (other == 0ull) break;  // first to arrive: the sibling will fit the parent
        __threadfence();
        const uint32_t sib = uint32_t(other) - 1u, far = uint32_t(other >> 32);
        const Box sb = load_node_box(nodes, sib);
        const uint32_t nlo = goRight ? lo : far, nhi = goRight ? far : hi;
        const bool root = nlo == 0 && nhi == n - 1;
        bool up = false;
        uint32_t id = 0;
        if (!root) {
            up = lbvh_delta(codes, n, nhi) > lbvh_delta(codes, n, nlo - 1);
            id = up ? nhi : nlo;
        }
        // Karras order: the child on the lower slots is "left"; fit_parent applies the size rule
        box = fit_parent<true, true>(id, goRight ? node : sib, goRight ? sib : node, split - nlo + 1, nhi - split, goRight ? box : sb,
                                     goRight ? sb : box, nInternal, nodes, wide, wide4, ext);
        if (root) break;
        node = id, lo = nlo, hi = nhi, goRight = up;
    }
    }
}

// ALLOW_UPDATE: what FL/RearrangeTriangles.hlsl:25-28 (load order -> sorted slot) and FL/ComputeAABBs.hlsli:160-164
// (parent of every node) leave behind for a later PERFORM_UPDATE.  The root's entry is 0.
__global__ void __launch_bounds__(kThreads) k_save_update_cache(const uint32_t *perm, const rt_hierarchy_node *hier, uint32_t n,
                                                                uint32_t *sort_cache, uint32_t *parents) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) sort_cache[perm[i]] = i;
    if (i < 2 * n - 1) parents[i] = i == 0 ? 0u : (hier[i].parent & ~treelet::kCollapseBit);
}
// PERFORM_UPDATE: sorted slot -> load-order element, so that the rearrange kernels of the full build are reused.
__global__ void __launch_bounds__(kThreads) k_invert_cache(const uint32_t *sort_cache, uint32_t n, uint32_t *perm) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) perm[sort_cache[i]] = i;
}

__global__ void k_write_headers(uint8_t *result, rt_bvh_offsets off, rt_ext_header ext, uint64_t ext_offset) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        *reinterpret_cast<rt_bvh_offsets *>(result) = off;
        rt_ext_header *e = reinterpret_cast<rt_ext_header *>(result + ext_offset);
        e->magic = ext.magic, e->count = ext.count, e->root_ref = ext.root_ref, e->top_level = ext.top_level;
        e->off_wide = ext.off_wide, e->off_leaf = ext.off_leaf, e->off_wide4 = ext.off_wide4;
        e->off_sort_cache = ext.off_sort_cache, e->off_parents = ext.off_parents, e->build_flags = ext.build_flags;
        e->total_bytes = ext.total_bytes, e->compacted_bytes = ext.compacted_bytes;
        e->has_procedural = ext.has_procedural;
        e->_pad0 = e->_pad1 = 0;
        e->_pad2[0] = e->_pad2[1] = 0;
        if (ext.count == 0) {
            // empty TLAS: node 0 is a zero box with zero flags (FL/TopLevelPrepareForComputeAABBs.hlsl:40-48)
            float4 *p = reinterpret_cast<float4 *>(result + 16);
            p[0] = make_float4(0, 0, 0, 0);
            p[1] = make_float4(0, 0, 0, 0);
            for (int k = 0; k < 3; ++k) e->root_center[k] = 0.0f, e->root_half[k] = 0.0f;
        }
    }
}

// ------------------------------------------------------------------------------------------ TLAS load
// FL/RayTracingHelper.hlsli:309-338 (terms multiplied by literal 0 dropped, see the oracle).
__device__ void invert_affine(const float *t, float *o) {
#define T(r, c) t[(r)*4 + (c)]
    float det = T(0, 0) * T(1, 1) * T(2, 2) - T(0, 0) * T(2, 1) * T(1, 2) - T(1, 0) * T(0, 1) * T(2, 2) +
                T(1, 0) * T(2, 1) * T(0, 2) + T(2, 0) * T(0, 1) * T(1, 2) - T(2, 0) * T(1, 1) * T(0, 2);
    float invDet = 1.0f / det;
    o[0] = invDet * (T(1, 1) * T(2, 2) + T(2, 1) * (0.0f - T(1, 2)));
    o[4] = invDet * (T(1, 2) * T(2, 0) + T(2, 2) * (0.0f - T(1, 0)));
    o[8] = invDet * (T(1, 0) * T(2, 1) - T(2, 0) * T(1, 1));
    o[1] = invDet * (T(2, 1) * T(0, 2) + T(0, 1) * (0.0f - T(2, 2)));
    o[5] = invDet * (T(2, 2) * T(0, 0) + T(0, 2) * (0.0f - T(2, 0)));
    o[9] = invDet * (T(2, 0) * T(0, 1) - T(0, 0) * T(2, 1));
    o[2] = invDet * (T(0, 1) * T(1, 2) + T(1, 1) * (0.0f - T(0, 2)));
    o[6] = invDet * (T(0, 2) * T(1, 0) + T(1, 2) * (0.0f - T(0, 0)));
    o[10] = invDet * (T(0, 0) * T(1, 1) - T(1, 0) * T(0, 1));
    o[3] = invDet * (T(0, 1) * (T(2, 2) * T(1, 3) - T(1, 2) * T(2, 3)) + T(1, 1) * (T(0, 2) * T(2, 3) - T(2, 2) * T(0, 3)) +
                     T(2, 1) * (T(1, 2) * T(0, 3) - T(0, 2) * T(1, 3)));
    o[7] = invDet * (T(0, 2) * (T(2, 0) * T(1, 3) - T(1, 0) * T(2, 3)) + T(1, 2) * (T(0, 0) * T(2, 3) - T(2, 0) * T(0, 3)) +
                     T(2, 2) * (T(1, 0) * T(0, 3) - T(0, 0) * T(1, 3)));
    o[11] = invDet * (T(0, 3) * (T(2, 0) * T(1, 1) - T(1, 0) * T(2, 1)) + T(1, 3) * (T(0, 0) * T(2, 1) - T(2, 0) * T(0, 1)) +
                      T(2, 3) * (T(1, 0) * T(0, 1) - T(0, 0) * T(1, 1)));
#undef T
}

// FL/TopLevelLoadAABBs.hlsli:58-100 fused with FL/CalculateSceneAABBFromBVHs.hlsl:16-40.
// `ptrs` != nullptr: D3D12_ELEMENTS_LAYOUT_ARRAY_OF_POINTERS — element i is *ptrs[i] (FL/TopLevelLoadAABBs.hlsli:38-49).
__device__ __forceinline__ bool blas_is_valid(const uint8_t *blas) {
    if (blas == nullptr || (uintptr_t(blas) & 63) != 0) return false;
    const rt_bvh_offsets *bo = reinterpret_cast<const rt_bvh_offsets *>(blas);
    if (bo->offsetToBoxes != 16 || bo->totalSize < 48 || bo->totalSize > (1ull << 33)) return false;
    const rt_ext_header *be = reinterpret_cast<const rt_ext_header *>(blas + align_up(bo->totalSize, 64));
    return be->magic == RT_EXT_MAGIC && be->top_level == 0;
}

__global__ void __launch_bounds__(kThreads) k_load_instances(const rt_instance_desc *descs, const rt_instance_desc *const *ptrs, uint32_t n,
                                                             rt_aabb_node *boxes, rt_bvh_metadata *md, uint32_t *aabb_enc,
                                                             rt_ext_header *tlas_ext, uint32_t *status) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    float smn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, smx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    if (i < n) {
        rt_instance_desc d = ptrs ? *ptrs[i] : descs[i];
        const uint8_t *blas = reinterpret_cast<const uint8_t *>(uintptr_t(d.blas));
        // A null BLAS address, or one that does not point at a finished rt_core bottom-level build, makes the instance
        // inactive (empty box, mask 0) and raises status bit 2 (rt_get_status -> RT_ERR_INVALID_ARG) instead of faulting.
        const bool valid = blas_is_valid(blas);
        if (!valid) {
            atomicOr(status, 4u);
            d.instance_id_and_mask &= 0x00ffffffu;
            d.blas = 0;
        }
        const rt_aabb_node *root = reinterpret_cast<const rt_aabb_node *>(blas + 16);
        // a TLAS over a BLAS with procedural primitives needs hit groups with intersection programs (rt_trace_rays_hit_groups)
        if (valid) {
            const rt_ext_header *be = reinterpret_cast<const rt_ext_header *>(blas + align_up(reinterpret_cast<const rt_bvh_offsets *>(blas)->totalSize, 64));
            if (be->has_procedural) atomicOr(&tlas_ext->has_procedural, 1u);
        }
        float bmn[3], bmx[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {  // BoundingBoxToAABB
            bmn[k] = valid ? root->center[k] - root->halfDim[k] : FLT_MAX;
            bmx[k] = valid ? root->center[k] + root->halfDim[k] : -FLT_MAX;
        }
        // TransformAABB: FL/RayTracingHelper.hlsli:340-366
        float mn[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, mx[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            f3 v = xform_point(d.transform, mk3((c & 4) ? bmx[0] : bmn[0], (c & 2) ? bmx[1] : bmn[1], (c & 1) ? bmx[2] : bmn[2]));
            mn[0] = fminf(mn[0], v.x), mn[1] = fminf(mn[1], v.y), mn[2] = fminf(mn[2], v.z);
            mx[0] = fmaxf(mx[0], v.x), mx[1] = fmaxf(mx[1], v.y), mx[2] = fmaxf(mx[2], v.z);
        }
        Box b = aabb_to_box(mn, mx);
        if (!valid) {  // an empty box: the union with it leaves every ancestor unchanged and no ray passes its slab test
#pragma unroll
            for (int k = 0; k < 3; ++k) b.c[k] = 0.0f, b.h[k] = -FLT_MAX;
        }
        rt_aabb_node nb;
#pragma unroll
        for (int k = 0; k < 3; ++k) nb.center[k] = b.c[k], nb.halfDim[k] = b.h[k];
        nb.flags = RT_NODE_LEAF_FLAG | i;
        nb.right = RT_NODE_LEAF_FLAG | i;
        boxes[i] = nb;
        // BVHMetadata (116 B): world->object transform, ids, BLAS address, object->world, instance index
        uint32_t w[29];
        float inv[12];
        invert_affine(d.transform, inv);
#pragma unroll
        for (int k = 0; k < 12; ++k) w[k] = __float_as_uint(inv[k]);
        w[12] = d.instance_id_and_mask;
        w[13] = d.hit_group_and_flags;
        w[14] = uint32_t(d.blas);
        w[15] = uint32_t(d.blas >> 32);
#pragma unroll
        for (int k = 0; k < 12; ++k) w[16 + k] = __float_as_uint(d.transform[k]);
        w[28] = i;
        uint32_t *dst = reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(md) + size_t(i) * 116);
#pragma unroll
        for (int k = 0; k < 29; ++k) dst[k] = w[k];
        if (valid) {
#pragma unroll
            for (int k = 0; k < 3; ++k) {  // scene AABB from the re-derived corners of the stored box
                smn[k] = b.c[k] - b.h[k];
                smx[k] = b.c[k] + b.h[k];
            }
        }
    }
    block_reduce_aabb(smn, smx, aabb_enc);
}

// FL/RearrangeBVHs.hlsl:50-58 (metadata only; leaf boxes are re-fitted by k_fit<true>) + packed instances.
__global__ void __launch_bounds__(kThreads) k_rearrange_instances(const rt_bvh_metadata *md, const uint32_t *perm, uint32_t n,
                                                                  rt_bvh_metadata *out_md, rt_packed_instance *packed) {
    uint32_t dst = blockIdx.x * blockDim.x + threadIdx.x;
    if (dst >= n) return;
    uint32_t src = perm[dst];
    const uint32_t *s = reinterpret_cast<const uint32_t *>(reinterpret_cast<const uint8_t *>(md) + size_t(src) * 116);
    uint32_t w[29];
#pragma unroll
    for (int k = 0; k < 29; ++k) w[k] = s[k];
    uint32_t *d = reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(out_md) + size_t(dst) * 116);
#pragma unroll
    for (int k = 0; k < 29; ++k) d[k] = w[k];
    rt_packed_instance pi;
#pragma unroll
    for (int k = 0; k < 12; ++k) pi.w2o[k] = __uint_as_float(w[k]);
    pi.instance_id_and_mask = w[12];
    // rt_core-private marker (bit 7 of the flags byte, unused by D3D12): world->object is the identity, so the
    // traversal kernels may keep the world-space ray constants (trace_persistent.cuh).  -0 compares equal to 0.
    bool ident = true;
#pragma unroll
    for (int k = 0; k < 12; ++k) ident = ident && (pi.w2o[k] == ((k == 0 || k == 5 || k == 10) ? 1.0f : 0.0f));
    pi.hit_group_and_flags = (w[13] & ~RT_PACKED_INSTANCE_IDENTITY) | (ident ? RT_PACKED_INSTANCE_IDENTITY : 0u);
    pi.instance_index = w[28];
    const uint8_t *blas = reinterpret_cast<const uint8_t *>(uintptr_t(uint64_t(w[14]) | (uint64_t(w[15]) << 32)));
    if (blas != nullptr) {
        const rt_bvh_offsets *bo = reinterpret_cast<const rt_bvh_offsets *>(blas);
        const rt_ext_header *be = reinterpret_cast<const rt_ext_header *>(blas + align_up(bo->totalSize, 64));
        pi.blas_root_ref = be->root_ref;
        pi.blas_wide = reinterpret_cast<const rt_wide_node *>(blas + be->off_wide);
        pi.blas_tris = reinterpret_cast<const rt_packed_tri *>(blas + be->off_leaf);
        pi.blas_wide4 = reinterpret_cast<const rt_wide4_node *>(blas + be->off_wide4);
    } else {  // inactive instance (k_load_instances cleared its mask and address)
        pi.blas_root_ref = RT_NODE_LEAF_FLAG;
        pi.blas_wide = nullptr, pi.blas_tris = nullptr, pi.blas_wide4 = nullptr;
    }
    pi._pad = 0;
    packed[dst] = pi;
}

// ------------------------------------------------------------------------------------------ host side
struct SortPlan {
    uint32_t blocks, tiles_per_block;
};
constexpr uint32_t kSortHistRows = 148 * 8;  // rows of kRadix counters in the scratch buffer (a public prebuild size: device independent)
SortPlan plan_sort(uint32_t n, int num_sms) {
    uint32_t tiles = (n + kSortTile - 1) / kSortTile;
    // the scratch layout (make_layout, sized without a context) reserves kSortHistRows histogram rows: blocks + the row totals
    uint32_t max_blocks = std::min<uint32_t>(uint32_t(num_sms) * 4, kSortHistRows - 1);
    SortPlan p;
    p.blocks = std::max(1u, std::min(tiles, max_blocks));
    p.tiles_per_block = (tiles + p.blocks - 1) / p.blocks;
    p.blocks = std::max(1u, (tiles + p.tiles_per_block - 1) / std::max(1u, p.tiles_per_block));
    return p;
}

struct Layout {
    uint64_t aabb_enc, aabb, codes, keysB, valsB, keysC, valsC, hier, counters, hist, elems, meta, tl_aabb, tl_base, total;
};
Layout make_layout(uint32_t n, bool top) {
    Layout L{};
    uint64_t o = 0;
    auto take = [&](uint64_t bytes) {
        uint64_t r = o;
        o = align_up(o + bytes, 256);
        return r;
    };
    const uint64_t nn = std::max(n, 1u);
    L.aabb_enc = take(32);
    L.aabb = take(32);
    L.codes = take(4 * nn);
    L.keysB = take(4 * nn);
    L.valsB = take(4 * nn);
    L.keysC = take(4 * nn);
    L.valsC = take(4 * nn);
    L.hier = take(12 * (2 * nn - 1));
    L.counters = take(4 * nn);
    L.hist = take(4ull * kRadix * kSortHistRows);
    L.elems = take((top ? 32 : 48) * nn);  // BLAS: rt_packed_tri records in load order; TLAS: instance boxes
    L.meta = take((top ? 116 : 0) * nn);
    // treelet pass (bottom level only): one 24-byte box per node, the base-treelet list (FL/GpuBVH2Builder.cpp:376-408)
    L.tl_aabb = take(top ? 0 : 24 * (2 * nn - 1));
    L.tl_base = take(top ? 0 : 4 * (nn / treelet::kFull + 2));
    L.total = o;
    return L;
}

struct ResultLayout {
    rt_bvh_offsets off;
    uint64_t ext, wide, leaf, wide4, sort_cache, parents, total;
};
ResultLayout make_result_layout(uint32_t n, bool top, bool allow_update = false) {
    ResultLayout R{};
    const uint32_t nodes = n == 0 ? 1 : 2 * n - 1;
    R.off.offsetToBoxes = 16;
    R.off.offsetToVertices = 16 + 32 * nodes;
    if (top) {
        R.off.offsetToPrimitiveMetaData = 0;
        R.off.totalSize = R.off.offsetToVertices + 116 * n;
    } else {
        R.off.offsetToPrimitiveMetaData = R.off.offsetToVertices + 40 * n;
        R.off.totalSize = R.off.offsetToPrimitiveMetaData + 12 * n;
    }
    R.ext = align_up(R.off.totalSize, 64);
    R.wide = R.ext + sizeof(rt_ext_header);
    R.leaf = R.wide + 64ull * std::max(1u, n > 0 ? n - 1 : 0u);
    R.wide4 = align_up(R.leaf + (top ? 96ull : 48ull) * std::max(n, 1u), 128);
    R.total = R.wide4 + 128ull * std::max(1u, n > 0 ? n - 1 : 0u);
    if (allow_update && n > 0) {
        // The reference appends exactly these 4n + 4(2n-1) bytes to ResultDataMaxSizeInBytes (FL/GpuBVH2Builder.cpp:444-448,
        // asserted by UT:1054-1087); here they follow the traversal section (they are private to the builder).
        R.sort_cache = R.total;
        R.parents = R.sort_cache + 4ull * n;
        R.total = R.parents + 4ull * (2ull * n - 1);
    }
    return R;
}

int sort_pairs(rt_context *ctx, uint8_t *scratch, const Layout &L, uint32_t n) {
    // 30-bit keys -> 4 passes of 8 bits.  codes -> B -> C -> B -> C
    SortPlan sp = plan_sort(n, ctx->num_sms);
    uint32_t *codes = reinterpret_cast<uint32_t *>(scratch + L.codes);
    uint32_t *kB = reinterpret_cast<uint32_t *>(scratch + L.keysB), *vB = reinterpret_cast<uint32_t *>(scratch + L.valsB);
    uint32_t *kC = reinterpret_cast<uint32_t *>(scratch + L.keysC), *vC = reinterpret_cast<uint32_t *>(scratch + L.valsC);
    uint32_t *hist = reinterpret_cast<uint32_t *>(scratch + L.hist);
    const uint32_t *kin = codes, *vin = nullptr;
    uint32_t *kout = kB, *vout = vB;
    for (int pass = 0; pass < 4; ++pass) {
        const int shift = pass * kRadixBits;
        k_radix_hist<<<sp.blocks, kSortThreads, 0, ctx->stream>>>(kin, n, shift, sp.tiles_per_block, hist);
        uint32_t *row_total = hist + size_t(kRadix) * sp.blocks;
        k_scan_rows<<<kRadix, kSortThreads, 0, ctx->stream>>>(hist, sp.blocks, row_total);
        if (pass == 0)
            k_radix_scatter<true><<<sp.blocks, kSortThreads, 0, ctx->stream>>>(kin, vin, n, shift, sp.tiles_per_block, hist, row_total, kout, vout);
        else
            k_radix_scatter<false><<<sp.blocks, kSortThreads, 0, ctx->stream>>>(kin, vin, n, shift, sp.tiles_per_block, hist, row_total, kout, vout);
        ctx->launches += 3;
        kin = kout, vin = vout;
        if (kout == kB) kout = kC, vout = vC; else kout = kB, vout = vB;
    }
    RT_LAUNCH_CHECK();
    return RT_OK;  // sorted pairs are in (kC, vC)
}

}  // namespace

extern "C" {

uint64_t rt_blob_bytes(uint32_t n, int top_level) { return make_result_layout(n, top_level != 0).off.totalSize; }

int rt_build_scratch_layout(uint32_t n, int top_level, rt_scratch_layout *out) {
    RT_REQUIRE(out != nullptr, "layout");
    Layout L = make_layout(n, top_level != 0);
    out->scene_aabb = L.aabb;
    out->morton_codes = L.codes;
    out->sorted_codes = L.keysC;
    out->sorted_indices = L.valsC;
    out->hierarchy = L.hier;
    out->primitives = L.elems;
    out->metadata = top_level ? L.meta : L.elems;
    out->total = L.total;
    return RT_OK;
}

static inline bool is_procedural(const rt_geometry_desc &d) { return d.type == RT_GEOMETRY_TYPE_PROCEDURAL_AABBS; }
static inline uint32_t geom_prims(const rt_geometry_desc &d) {  // FL/LoadPrimitivesPass.cpp:87-88,136
    return is_procedural(d) ? d.vertex_count : (d.index_format == 0 ? d.vertex_count : d.index_count) / 3;
}
static uint32_t count_prims(const rt_geometry_desc *geoms, uint32_t n_geoms) {
    uint64_t n = 0;
    for (uint32_t g = 0; g < n_geoms; ++g) n += geom_prims(geoms[g]);
    return uint32_t(std::min<uint64_t>(n, 0xffffffffull));
}

static inline bool allows_update(uint32_t f) { return (f & RT_BUILD_FLAG_ALLOW_UPDATE) != 0; }
static inline bool performs_update(uint32_t f) { return (f & RT_BUILD_FLAG_PERFORM_UPDATE) != 0; }
// FL/TreeletReorder.cpp:66-80
static inline uint32_t treelet_passes(uint32_t f) {
    return (f & RT_BUILD_FLAG_PREFER_FAST_BUILD) ? 0u : ((f & RT_BUILD_FLAG_PREFER_FAST_TRACE) ? 3u : 1u);
}

int rt_blas_prebuild(rt_context *ctx, const rt_geometry_desc *geoms, uint32_t n_geoms, uint32_t flags, rt_prebuild_info *info) {
    RT_REQUIRE(ctx && info && (geoms || n_geoms == 0), "null argument");
    uint32_t n = count_prims(geoms, n_geoms);
    RT_REQUIRE(n < (1u << 24), "more than 2^24-1 primitives (node indices are 24 bit: RayTracingHelper.hlsli:112-118)");
    info->result_bytes = make_result_layout(n, false, allows_update(flags)).total;
    info->scratch_bytes = make_layout(n, false).total;  // the same with and without ALLOW_UPDATE (UT:1085)
    info->update_scratch_bytes = allows_update(flags) ? info->scratch_bytes : 0;
    return RT_OK;
}

int rt_tlas_prebuild(rt_context *ctx, uint32_t n, uint32_t flags, rt_prebuild_info *info) {
    RT_REQUIRE(ctx && info, "null argument");
    RT_REQUIRE(n < (1u << 24), "more than 2^24-1 instances");
    info->result_bytes = make_result_layout(n, true, allows_update(flags)).total;
    info->scratch_bytes = make_layout(n, true).total;
    info->update_scratch_bytes = allows_update(flags) ? info->scratch_bytes : 0;
    return RT_OK;
}

int rt_update_cache_layout(uint32_t n, int top_level, uint64_t *sort_cache_offset, uint64_t *parents_offset) {
    RT_REQUIRE(sort_cache_offset && parents_offset, "null argument");
    ResultLayout R = make_result_layout(n, top_level != 0, true);
    *sort_cache_offset = R.sort_cache;
    *parents_offset = R.parents;
    return RT_OK;
}

// PERFORM_UPDATE is only defined on a buffer that an ALLOW_UPDATE build of the same element count produced
// (the reference does not check and reads garbage; here it is E_INVALIDARG).  One 128-byte read back.
static int check_updatable(rt_context *ctx, const uint8_t *result, const ResultLayout &R, uint32_t n, bool top) {
    rt_ext_header e{};
    RT_CUDA(cudaMemcpyAsync(&e, result + R.ext, sizeof(e), cudaMemcpyDeviceToHost, ctx->stream));
    RT_CUDA(cudaStreamSynchronize(ctx->stream));
    RT_REQUIRE(e.magic == RT_EXT_MAGIC && e.count == n && e.top_level == (top ? 1u : 0u) && allows_update(e.build_flags) &&
                   e.off_sort_cache == R.sort_cache && e.off_parents == R.parents,
               "PERFORM_UPDATE: the result buffer does not hold an ALLOW_UPDATE build of the same element count");
    return RT_OK;
}

static int build_common(rt_context *ctx, uint32_t n, bool top, uint32_t flags, uint8_t *scratch, uint8_t *result, const Layout &L,
                        const ResultLayout &R) {
    cudaStream_t st = ctx->stream;
    const bool update = performs_update(flags);
    const int grid = rt_div_up(n, kThreads);
    uint32_t *perm = reinterpret_cast<uint32_t *>(scratch + L.valsC);
    rt_hierarchy_node *hier = reinterpret_cast<rt_hierarchy_node *>(scratch + L.hier);
    uint32_t *sort_cache = reinterpret_cast<uint32_t *>(result + R.sort_cache);
    uint32_t *parents = reinterpret_cast<uint32_t *>(result + R.parents);
    // one byte per internal node in the sort's dead ping-pong buffer (the sorted pairs end up in keysC / valsC)
    uint8_t *fit_local = !top ? scratch + L.keysB : nullptr;
    // full bottom-level build without treelet passes or update caches: hierarchy emission and fit are one kernel (k_lbvh_fit)
    const bool fused = !top && !update && treelet_passes(flags) == 0 && !allows_update(flags);
    if (update) {
        k_invert_cache<<<grid, kThreads, 0, st>>>(sort_cache, n, perm);
        ctx->launches++;
    } else {
        float *aabb = reinterpret_cast<float *>(scratch + L.aabb);
        uint32_t *codes = reinterpret_cast<uint32_t *>(scratch + L.codes);
        k_decode_aabb<<<1, 32, 0, st>>>(reinterpret_cast<uint32_t *>(scratch + L.aabb_enc), aabb);
        if (top)
            k_morton_boxes<<<grid, kThreads, 0, st>>>(reinterpret_cast<rt_aabb_node *>(scratch + L.elems), n, aabb, codes);
        else
            k_morton_prims<<<grid, kThreads, 0, st>>>(reinterpret_cast<rt_packed_tri *>(scratch + L.elems), n, aabb, codes);
        ctx->launches += 2;
        int rc = sort_pairs(ctx, scratch, L, n);
        if (rc) return rc;
        const uint32_t *sorted_codes = reinterpret_cast<uint32_t *>(scratch + L.keysC);
        if (fused) {
            if (n > 1) RT_CUDA(cudaMemsetAsync(hier, 0, 8ull * (n - 1), st));  // g_slot: one 64-bit meeting word per split
        } else {
            RT_CUDA(cudaMemsetAsync(hier, 0, 12ull * (2ull * n - 1), st));
        }
        if (n > 1 && !fused) {
            k_hierarchy<<<rt_div_up(n - 1, kThreads), kThreads, 0, st>>>(sorted_codes, n, hier, fit_local);
            ctx->launches++;
        }
    }
    rt_aabb_node *nodes = reinterpret_cast<rt_aabb_node *>(result + 16);
    rt_wide_node *wide = reinterpret_cast<rt_wide_node *>(result + R.wide);
    rt_ext_header *ext = reinterpret_cast<rt_ext_header *>(result + R.ext);
    uint32_t *counters = reinterpret_cast<uint32_t *>(scratch + L.counters);
    const rt_aabb_node *boxes = reinterpret_cast<rt_aabb_node *>(scratch + L.elems);
    rt_primitive *sp = reinterpret_cast<rt_primitive *>(result + R.off.offsetToVertices);
    rt_packed_tri *packed = reinterpret_cast<rt_packed_tri *>(result + R.leaf);
    if (top)
        k_rearrange_instances<<<grid, kThreads, 0, st>>>(reinterpret_cast<rt_bvh_metadata *>(scratch + L.meta), perm, n,
                                                         reinterpret_cast<rt_bvh_metadata *>(result + R.off.offsetToVertices),
                                                         reinterpret_cast<rt_packed_instance *>(result + R.leaf));
    else
        k_rearrange_tris<<<grid, kThreads, 0, st>>>(reinterpret_cast<rt_packed_tri *>(scratch + L.elems), perm, n, sp,
                                                    reinterpret_cast<rt_primitive_meta *>(result + R.off.offsetToPrimitiveMetaData), packed);
    ctx->launches++;
    if (!update) {
        if (!top) {
            // FL/TreeletReorder.cpp:38-109: 0 / 1 / 3 optimisation passes, MinTrianglesPerTreelet 7, 14, 28
            uint32_t min_tris = treelet::kFull;
            float *tl_aabb = reinterpret_cast<float *>(scratch + L.tl_aabb);
            uint32_t *tl_base = reinterpret_cast<uint32_t *>(scratch + L.tl_base);
            for (uint32_t pass = 0; pass < treelet_passes(flags) && min_tris <= n; ++pass, min_tris *= 2) {
                RT_CUDA(cudaMemsetAsync(counters, 0, 4ull * n, st));  // ClearBuffers.hlsl
                RT_CUDA(cudaMemsetAsync(tl_base, 0, 4, st));
                treelet::k_find_treelets<<<grid, kThreads, 0, st>>>(n, hier, packed, counters, tl_aabb, tl_base, min_tris);
                treelet::k_treelet_reorder<<<rt_div_up(n / min_tris, treelet::kWarps), 32 * treelet::kWarps, 0, st>>>(n, hier, counters,
                                                                                                                    tl_aabb, tl_base, fit_local);
                ctx->launches += 2;
            }
        }
        if (allows_update(flags)) {
            k_save_update_cache<<<rt_div_up(2ull * n - 1, kThreads), kThreads, 0, st>>>(perm, hier, n, sort_cache, parents);
            ctx->launches++;
        }
    }
    if (!fused) RT_CUDA(cudaMemsetAsync(counters, 0, 4ull * n, st));
    rt_wide4_node *wide4 = reinterpret_cast<rt_wide4_node *>(result + R.wide4);
    if (fused) {
        RT_CUDA(cudaFuncSetAttribute(k_lbvh_fit, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kFitLocalDynSmem)));  // per device
        // exit list {node, lo, hi} in buffers this path leaves unused (the sort's ping-pong pair, the arrival counters);
        // its length in the spare word behind the encoded scene AABB (zeroed by k_init_aabb)
        uint32_t *exit_count = reinterpret_cast<uint32_t *>(scratch + L.aabb_enc) + 7;
        uint32_t *exit_nodes = reinterpret_cast<uint32_t *>(scratch + L.valsB), *exit_lo = reinterpret_cast<uint32_t *>(scratch + L.keysB);
        const uint32_t *codes_sorted = reinterpret_cast<uint32_t *>(scratch + L.keysC);
        unsigned long long *g_slot = reinterpret_cast<unsigned long long *>(hier);
        k_lbvh_fit<<<rt_div_up(n, kFitBlock), kFitBlock, kFitLocalDynSmem, st>>>(n, codes_sorted, nodes, packed, wide, wide4, ext,
                                                                                 exit_count, exit_nodes, exit_lo, counters);
        if (n > kFitBlock) {  // a build of one block leaves no exits
            k_lbvh_exits<<<std::max(1, rt_div_up(n / 8, kThreads)), kThreads, 0, st>>>(n, codes_sorted, g_slot, nodes, wide, wide4, ext, exit_count, exit_nodes, exit_lo, counters);
            ctx->launches++;
        }
    } else if (top) {
        if (update)
            k_fit<true, true><<<grid, kThreads, 0, st>>>(n, hier, counters, nodes, nullptr, boxes, perm, wide, ext, parents);
        else
            k_fit<true, false><<<grid, kThreads, 0, st>>>(n, hier, counters, nodes, nullptr, boxes, perm, wide, ext, parents);
    } else {
        if (update)
            k_fit<false, true><<<grid, kThreads, 0, st>>>(n, hier, counters, nodes, sp, nullptr, perm, wide, ext, parents);
        else {
            // exit list in the sort's dead ping-pong buffers: node ids in valsB, subtree sizes (<= kFitBlock) behind the flags.
            // keysB holds 4n bytes; flags take n, the sizes 2 x (exit entries <= n) after a 256-byte round-up, and a build of
            // n <= kFitBlock primitives fits in one block and leaves no entries — so the 3n + 255 bytes used fit for every n
            uint32_t *exit_nodes = reinterpret_cast<uint32_t *>(scratch + L.valsB);
            uint16_t *exit_sizes = reinterpret_cast<uint16_t *>(scratch + L.keysB + align_up(n, 256));
            RT_CUDA(cudaFuncSetAttribute(k_fit_local, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kFitLocalDynSmem)));  // per device
            k_fit_local<<<rt_div_up(n, kFitBlock), kFitBlock, kFitLocalDynSmem, st>>>(n, hier, counters, nodes, packed, wide, wide4, ext,
                                                                                      fit_local, exit_nodes, exit_sizes);
            if (n > 1) {
                // every block leaves at least one and on average ~log2(kFitBlock) entries; n bounds it
                k_fit_exits<<<std::max(1, rt_div_up(n / 4, kThreads)), kThreads, 0, st>>>(n, hier, counters, nodes, wide, wide4, ext,
                                                                                            exit_nodes, exit_sizes);
                ctx->launches++;
            }
        }
    }
    ctx->launches++;
    if (n > 1 && (top || update)) {  // k_fit leaves the 4-wide nodes to k_collapse4
        k_collapse4<<<rt_div_up(n - 1, kThreads), kThreads, 0, st>>>(wide, n - 1, wide4);
        ctx->launches++;
    }
    RT_LAUNCH_CHECK();
    return RT_OK;
}

static int write_headers(rt_context *ctx, uint32_t n, bool top, uint32_t flags, uint8_t *result, const ResultLayout &R,
                         bool has_procedural = false) {
    rt_ext_header e{};
    e.has_procedural = has_procedural ? 1u : 0u;
    e.magic = RT_EXT_MAGIC;
    e.count = n;
    e.root_ref = (n == 1) ? RT_NODE_LEAF_FLAG : 0u;
    e.top_level = top ? 1u : 0u;
    e.off_wide = R.wide;
    e.off_leaf = R.leaf;
    e.off_wide4 = R.wide4;
    e.off_sort_cache = R.sort_cache;
    e.off_parents = R.parents;
    e.build_flags = flags & ~uint32_t(RT_BUILD_FLAG_PERFORM_UPDATE);
    e.total_bytes = R.total;
    e.compacted_bytes = R.sort_cache ? R.sort_cache : R.total;
    k_write_headers<<<1, 32, 0, ctx->stream>>>(result, R.off, e, R.ext);
    ctx->launches++;
    RT_LAUNCH_CHECK();
    return RT_OK;
}

int rt_blas_build(rt_context *ctx, const rt_geometry_desc *geoms, uint32_t n_geoms, uint32_t build_flags, void *scratch_,
                  uint64_t scratch_bytes, void *result_, uint64_t result_bytes) {
    RT_REQUIRE(ctx && scratch_ && result_, "null argument");  // E_INVALIDARG: FL/GpuBVH2Builder.cpp:145-148
    RT_REQUIRE((uintptr_t(result_) & 63) == 0 && (uintptr_t(scratch_) & 63) == 0, "buffers must be 64-byte aligned");
    RT_REQUIRE(!performs_update(build_flags) || allows_update(build_flags), "PERFORM_UPDATE without ALLOW_UPDATE");
    uint32_t n = count_prims(geoms, n_geoms);
    RT_REQUIRE(n > 0, "bottom-level build with zero primitives");
    RT_REQUIRE(n < (1u << 24), "more than 2^24-1 primitives");
    Layout L = make_layout(n, false);
    ResultLayout R = make_result_layout(n, false, allows_update(build_flags));
    if (scratch_bytes < L.total || result_bytes < R.total) {
        rt_set_error("buffer too small: scratch %llu < %llu or result %llu < %llu", (unsigned long long)scratch_bytes,
                     (unsigned long long)L.total, (unsigned long long)result_bytes, (unsigned long long)R.total);
        return RT_ERR_TOO_SMALL;
    }
    RT_CUDA(cudaSetDevice(ctx->device));
    uint8_t *scratch = static_cast<uint8_t *>(scratch_), *result = static_cast<uint8_t *>(result_);
    cudaStream_t st = ctx->stream;
    bool any_procedural = false;
    for (uint32_t g = 0; g < n_geoms; ++g) {
        RT_REQUIRE(geoms[g].type == RT_GEOMETRY_TYPE_TRIANGLES || is_procedural(geoms[g]), "unrecognized geometry type");  // LoadPrimitivesPass.cpp:124-127
        any_procedural |= is_procedural(geoms[g]);
    }
    int rc = performs_update(build_flags) ? check_updatable(ctx, result, R, n, false)
                                          : write_headers(ctx, n, false, build_flags, result, R, any_procedural);
    if (rc) return rc;
    uint32_t *aabb_enc = reinterpret_cast<uint32_t *>(scratch + L.aabb_enc);
    k_init_aabb<<<1, 32, 0, st>>>(aabb_enc);
    ctx->launches++;
    uint32_t offset = 0;
    for (uint32_t g = 0; g < n_geoms; ++g) {  // one launch per geometry, like FL/LoadPrimitivesPass.cpp:60-170
        const rt_geometry_desc &d = geoms[g];
        LoadGeom lg{};
        lg.vb = static_cast<const uint8_t *>(d.vertex_buffer);
        lg.ib = d.index_buffer;
        lg.stride = d.vertex_stride_bytes;
        lg.index_format = d.index_format;
        lg.num_tris = geom_prims(d);
        lg.procedural = is_procedural(d);
        RT_REQUIRE(d.vertex_buffer != nullptr || lg.num_tris == 0,
                   lg.procedural ? "non-zero AABBCount provided with a null AABB buffer" : "null vertex buffer");  // LoadPrimitivesPass.cpp:130-133
        if (lg.procedural) {
            RT_REQUIRE(d.vertex_stride_bytes >= 24 && d.vertex_stride_bytes % 4 == 0, "AABB stride");
        } else {
            RT_REQUIRE(d.index_format == 0 || d.index_format == 16 || d.index_format == 32, "index_format must be 0, 16 or 32");
            RT_REQUIRE(d.index_format == 0 || d.index_buffer != nullptr, "null index buffer");
            RT_REQUIRE(d.vertex_stride_bytes >= 12 && d.vertex_stride_bytes % 4 == 0, "vertex stride");
        }
        lg.prim_offset = offset;
        lg.geom_index = g;
        lg.flags = d.flags;
        lg.has_xf = !lg.procedural && d.transform3x4 != nullptr;
        if (lg.has_xf) {
            RT_CUDA(cudaMemcpyAsync(lg.xf, d.transform3x4, 48, cudaMemcpyDefault, st));
            RT_CUDA(cudaStreamSynchronize(st));
        }
        if (lg.num_tris) {
            k_load_triangles<<<std::min(rt_div_up(lg.num_tris, kThreads), ctx->num_sms * 16), kThreads, 0, st>>>(
                lg, reinterpret_cast<rt_packed_tri *>(scratch + L.elems), aabb_enc);
            ctx->launches++;
        }
        offset += lg.num_tris;
    }
    RT_LAUNCH_CHECK();
    return build_common(ctx, n, false, build_flags, scratch, result, L, R);
}

static int tlas_build_impl(rt_context *ctx, const rt_instance_desc *descs, const rt_instance_desc *const *ptrs, uint32_t n,
                           uint32_t build_flags, void *scratch_, uint64_t scratch_bytes, void *result_, uint64_t result_bytes);

int rt_tlas_build(rt_context *ctx, const rt_instance_desc *descs, uint32_t n, uint32_t build_flags, void *scratch_,
                  uint64_t scratch_bytes, void *result_, uint64_t result_bytes) {
    return tlas_build_impl(ctx, descs, nullptr, n, build_flags, scratch_, scratch_bytes, result_, result_bytes);
}

int rt_tlas_build_ptrs(rt_context *ctx, const rt_instance_desc *const *desc_ptrs, uint32_t n, uint32_t build_flags, void *scratch_,
                       uint64_t scratch_bytes, void *result_, uint64_t result_bytes) {
    return tlas_build_impl(ctx, nullptr, desc_ptrs, n, build_flags, scratch_, scratch_bytes, result_, result_bytes);
}

int rt_blas_prebuild_ptrs(rt_context *ctx, const rt_geometry_desc *const *geoms, uint32_t n_geoms, uint32_t flags, rt_prebuild_info *info) {
    RT_REQUIRE(n_geoms == 0 || geoms != nullptr, "null argument");
    std::vector<rt_geometry_desc> flat(n_geoms);
    for (uint32_t g = 0; g < n_geoms; ++g) {
        RT_REQUIRE(geoms[g] != nullptr, "null geometry descriptor pointer");
        flat[g] = *geoms[g];  // GetGeometryDesc, ARRAY_OF_POINTERS: FL/Util.h:101-114
    }
    return rt_blas_prebuild(ctx, flat.data(), n_geoms, flags, info);
}

int rt_blas_build_ptrs(rt_context *ctx, const rt_geometry_desc *const *geoms, uint32_t n_geoms, uint32_t build_flags, void *scratch,
                       uint64_t scratch_bytes, void *result, uint64_t result_bytes) {
    RT_REQUIRE(n_geoms == 0 || geoms != nullptr, "null argument");
    std::vector<rt_geometry_desc> flat(n_geoms);
    for (uint32_t g = 0; g < n_geoms; ++g) {
        RT_REQUIRE(geoms[g] != nullptr, "null geometry descriptor pointer");
        flat[g] = *geoms[g];
    }
    return rt_blas_build(ctx, flat.data(), n_geoms, build_flags, scratch, scratch_bytes, result, result_bytes);
}

static int tlas_build_impl(rt_context *ctx, const rt_instance_desc *descs, const rt_instance_desc *const *ptrs, uint32_t n,
                           uint32_t build_flags, void *scratch_, uint64_t scratch_bytes, void *result_, uint64_t result_bytes) {
    RT_REQUIRE(ctx && result_, "null argument");
    RT_REQUIRE(n == 0 || ((descs || ptrs) && scratch_), "null argument");
    RT_REQUIRE((uintptr_t(result_) & 63) == 0 && (uintptr_t(scratch_) & 63) == 0, "buffers must be 64-byte aligned");
    RT_REQUIRE(n < (1u << 24), "more than 2^24-1 instances");
    RT_REQUIRE(!performs_update(build_flags) || allows_update(build_flags), "PERFORM_UPDATE without ALLOW_UPDATE");
    Layout L = make_layout(n, true);
    ResultLayout R = make_result_layout(n, true, allows_update(build_flags));
    if ((n > 0 && scratch_bytes < L.total) || result_bytes < R.total) {
        rt_set_error("buffer too small: scratch %llu < %llu or result %llu < %llu", (unsigned long long)scratch_bytes,
                     (unsigned long long)L.total, (unsigned long long)result_bytes, (unsigned long long)R.total);
        return RT_ERR_TOO_SMALL;
    }
    RT_CUDA(cudaSetDevice(ctx->device));
    uint8_t *scratch = static_cast<uint8_t *>(scratch_), *result = static_cast<uint8_t *>(result_);
    cudaStream_t st = ctx->stream;
    int rc = performs_update(build_flags) ? check_updatable(ctx, result, R, n, true) : write_headers(ctx, n, true, build_flags, result, R);
    if (rc || n == 0) return rc;
    uint32_t *aabb_enc = reinterpret_cast<uint32_t *>(scratch + L.aabb_enc);
    k_init_aabb<<<1, 32, 0, st>>>(aabb_enc);
    if (performs_update(build_flags))  // the flag is re-derived from the instances of THIS update (only ever OR-ed below)
        RT_CUDA(cudaMemsetAsync(result + R.ext + offsetof(rt_ext_header, has_procedural), 0, 4, st));
    k_load_instances<<<rt_div_up(n, kThreads), kThreads, 0, st>>>(descs, ptrs, n, reinterpret_cast<rt_aabb_node *>(scratch + L.elems),
                                                                 reinterpret_cast<rt_bvh_metadata *>(scratch + L.meta), aabb_enc,
                                                                 reinterpret_cast<rt_ext_header *>(result + R.ext), ctx->status);
    ctx->launches += 2;
    RT_LAUNCH_CHECK();
    return build_common(ctx, n, true, build_flags, scratch, result, L, R);
}

}  // extern "C"
