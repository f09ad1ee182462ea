// denoise.cu — shared-memory-tiled separable joint-bilateral denoiser + compositor for sm_100a.
//
// Replaces DenoiseCompositor::dispatch's two compute passes (src/DenoiseCompositor.cpp:109-148;
// assets/shaders/BilateralFilter.hlsli:50-118, DenoiseCommon.hlsli:46-77).  Same arithmetic per pixel, in the same
// order (weights LUT, L1 range weight, taps accumulated from -k to +k, color/weight, composite + exposure + Reinhard
// + gamma); what differs is how the taps are fetched.  The reference's 64x1 / 1x64 line groups read 2k+1 LDS texels
// per output; a first version here did the same from a 2-D tile and was bound by shared-memory bandwidth
// (50 LDS.128 per pixel and pass: 138 us per 1080p frame, 22 % of the HBM roofline).  Now:
//   * every thread produces R = 8 consecutive outputs ALONG the filter axis and walks the R + 2k texels they need
//     once, keeping the 8 centre joints and 8 accumulators in registers: (R + 2k) / R = 4 texel fetches per output
//     instead of 25;
//   * the tile is stored as six float planes (rgb of input and joint; alpha is never read), so lanes touch
//     consecutive banks — pass V directly (lanes along x), pass H through a +1-per-8 column padding that spreads the
//     lanes' 8-pixel strides over all 32 banks;
//   * pass H tiles are 256 x 8 pixels (halo overhead 2k/256), pass V tiles 32 x 64 (2k/64); rows are staged with
//     coalesced 16-byte loads and pass H writes its results back through shared memory so stores are coalesced too.
// Out-of-image texels read as 0 for both the input and the joint image (D3D out-of-bounds load).
#include <cuda_fp16.h>

#include <initializer_list>
#include <type_traits>

#include "common.cuh"

namespace {

constexpr int MAX_EXTENT = 20, KERNEL_TAPS = 6;
constexpr int R = 8;                  // outputs per thread along the filter axis
constexpr int kThreadsDn = 256;       // 8 warps
constexpr int H_TW = 32 * R, H_TH = 8;                        // pass H tile: one warp per row, 8 pixels per lane
constexpr int H_PITCH = ((H_TW + 2 * MAX_EXTENT + 8) * 9 + 7) / 8 + 1;  // padded columns: c -> c + (c >> 3); +8: the last unrolled block may read (never use) up to 7 texels past the halo
constexpr int V_TW = 32, V_TH = 8 * R;                        // pass V tile: lanes along x, one 8-row strip per warp
constexpr int V_ROWS = V_TH + 2 * MAX_EXTENT + 8;  // +8: as H_PITCH
constexpr int H_PLANE = H_TH * H_PITCH, V_PLANE = V_ROWS * V_TW;
constexpr size_t H_SMEM = (6 * H_PLANE + 64) * sizeof(float), V_SMEM = (6 * V_PLANE + 64) * sizeof(float);

struct DenoiseArgs {
    const float4 *joint, *input;
    float4 *out;
    int w, h, k;
    int half;  // stores round through fp16 (the reference's intermediate and output targets are R16G16B16A16_FLOAT)
    rt_denoiser_params prm;
    float wts[2 * MAX_EXTENT + 1];
};

__device__ __forceinline__ float4 fetch(const float4 *img, int x, int y, int w, int h) {
    if (x < 0 || y < 0 || x >= w || y >= h) return make_float4(0, 0, 0, 0);
    return __ldg(img + size_t(y) * w + x);
}

__device__ __forceinline__ int hpad(int c) { return c + (c >> 3); }

// Packed fp32 pairs (sm_100 FADD2 / FMUL2 / FFMA2: two IEEE round-to-nearest operations per issue slot, each lane's result
// bit-identical to the scalar instruction).  The kernel is issue-bound (ncu: 66 % of the issue slots, DRAM 16 %), so the
// filter's (texel, output) work is done for two neighbouring outputs per instruction wherever the operation has a packed
// form; |x| and saturate only exist as scalar operand modifiers and stay scalar.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk2(f32x2 v, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}

// PASS 0 = horizontal (DenoiseCompositorH.hlsl), PASS 1 = vertical + composite (DenoiseCompositorV.hlsl).
template <int PASS>
__global__ void __launch_bounds__(kThreadsDn, 3) k_denoise(const __grid_constant__ DenoiseArgs A) {
    extern __shared__ float smem[];
    // pass V sizes its planes for the kernel radius in use (k = 12: 74 KB, three blocks per SM; k = 20: 86 KB, two)
    const int PLANE = PASS == 0 ? H_PLANE : (V_TH + 2 * A.k + 8) * V_TW;
    float *sW = smem;            // 41 tap weights
    float *pl = smem + 64;       // planes: in.r in.g in.b joint.r joint.g joint.b
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int k = A.k;
    if (threadIdx.x < 64) {  // sW[1 + jj] = weight of tap i = jj - k; zero outside the kernel
        const int i = int(threadIdx.x) - 1 - k;
        sW[threadIdx.x] = (i >= -k && i <= k) ? A.wts[i + MAX_EXTENT] : 0.0f;
    }
    // ---- stage the tile and the +-k halo along the filter axis
    int x0, y0;  // first output pixel of this thread
    if (PASS == 0) {
        const int bx = blockIdx.x * H_TW, by = blockIdx.y * H_TH;
        const int cols = H_TW + 2 * k;
        for (int row = warp; row < H_TH; row += kThreadsDn / 32) {
            const int gy = by + row;
            for (int c = lane; c < cols; c += 32) {
                const int gx = bx + c - k;
                const float4 a = fetch(A.input, gx, gy, A.w, A.h), j = fetch(A.joint, gx, gy, A.w, A.h);
                float *q = pl + row * H_PITCH + hpad(c);
                q[0] = a.x, q[PLANE] = a.y, q[2 * PLANE] = a.z, q[3 * PLANE] = j.x, q[4 * PLANE] = j.y, q[5 * PLANE] = j.z;
            }
        }
        x0 = bx + R * lane, y0 = by + warp;
    } else {
        const int bx = blockIdx.x * V_TW, by = blockIdx.y * V_TH;
        const int rows = V_TH + 2 * k;
        const int gx = bx + lane;
        for (int row = warp; row < rows; row += kThreadsDn / 32) {
            const int gy = by + row - k;
            const float4 a = fetch(A.input, gx, gy, A.w, A.h), j = fetch(A.joint, gx, gy, A.w, A.h);
            float *q = pl + row * V_TW + lane;
            q[0] = a.x, q[PLANE] = a.y, q[2 * PLANE] = a.z, q[3 * PLANE] = j.x, q[4 * PLANE] = j.y, q[5 * PLANE] = j.z;
        }
        x0 = bx + lane, y0 = by + R * warp;
    }
    __syncthreads();
    // texel at filter-axis offset j from this thread's first output (j in [-k, R-1+k])
    const float *base = PASS == 0 ? pl + warp * H_PITCH : pl + lane;
    auto at = [&](int j) -> const float * {
        return PASS == 0 ? base + hpad(R * lane + j + k) : base + (R * warp + j + k) * V_TW;
    };
    float cjx[R], cjy[R], cjz[R], ar[R], ag[R], ab[R], aw[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const float *q = at(r);
        cjx[r] = q[3 * PLANE], cjy[r] = q[4 * PLANE], cjz[r] = q[5 * PLANE];
        ar[r] = ag[r] = ab[r] = aw[r] = 0.0f;
    }
    if (A.prm.debugVisualize == 2) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const float *q = at(r);
            ar[r] = q[0], ag[r] = q[PLANE], ab[r] = q[2 * PLANE], aw[r] = 1.0f;
        }
    } else {
        // filterKernel (BilateralFilter.hlsli:75-118) for R outputs at once.  Texel jj (0-based from the first halo
        // texel) is tap i = jj - k - r of output r, valid iff 0 <= jj - r <= 2k; every output still receives its taps in
        // the order i = -k .. k.  The tap weight w[jj - r] lives in ring slot (jj - r) & 7: a slot is written once, when
        // its texel is fetched (r = 0), and read by output r exactly r steps later, so with the jj loop unrolled by 8
        // all slot indices are compile-time constants — one weight fetch per texel instead of one per tap.
        // Outputs r and r + 1 share every instruction that has a packed form.  A tap past an output's last one needs no
        // test: its weight sW[jj - r] is 0 there, and x + 0 * s is x (s is finite), so such a half-pair is value-neutral.
        f32x2 cx2[R / 2], cy2[R / 2], cz2[R / 2], ar2[R / 2], ag2[R / 2], ab2[R / 2], aw2[R / 2];
#pragma unroll
        for (int h = 0; h < R / 2; ++h) {
            cx2[h] = pk2(cjx[2 * h], cjx[2 * h + 1]), cy2[h] = pk2(cjy[2 * h], cjy[2 * h + 1]), cz2[h] = pk2(cjz[2 * h], cjz[2 * h + 1]);
            ar2[h] = ag2[h] = ab2[h] = aw2[h] = pk2(0.0f, 0.0f);
        }
        // ring2[p] = {w[jj], w[jj - 1]}: the weights outputs r and r + 1 apply to texel jj + r, fetched as a pair when texel jj
        // is (the table is stored shifted by one, sW[0] = 0, so that w[-1] reads as 0)
        f32x2 ring2[8];
#pragma unroll
        for (int p = 0; p < 8; ++p) ring2[p] = pk2(0.0f, 0.0f);  // "before the first tap" reads as weight 0
        const f32x2 one2 = pk2(1.0f, 1.0f);
        auto block = [&](const int b, auto firstTag, auto checkTag) {
            constexpr bool FIRST = decltype(firstTag)::value, CHECK = decltype(checkTag)::value;
#pragma unroll
            for (int p = 0; p < 8; ++p) {
                const int jj = 8 * b + p;
                const float *q = at(jj - k);
                const float sx = q[0], sy = q[PLANE], sz = q[2 * PLANE], jx = q[3 * PLANE], jy = q[4 * PLANE], jz = q[5 * PLANE];
                ring2[p] = pk2(sW[jj + 1], sW[jj]);
                const f32x2 sx2 = pk2(sx, sx), sy2 = pk2(sy, sy), sz2 = pk2(sz, sz), jx2 = pk2(jx, jx), jy2 = pk2(jy, jy), jz2 = pk2(jz, jz);
#pragma unroll
                for (int h = 0; h < R / 2; ++h) {
                    const int r = 2 * h;
                    if (FIRST && p < r) continue;              // jj - r < 0: before the first tap of both outputs
                    if (CHECK && jj - r - 1 > 2 * k) continue;  // past the last tap of both
                    float dxl, dxh, dyl, dyh, dzl, dzh;
                    upk2(sub2(jx2, cx2[h]), dxl, dxh), upk2(sub2(jy2, cy2[h]), dyl, dyh), upk2(sub2(jz2, cz2[h]), dzl, dzh);
                    const float ml = __saturatef(((fabsf(dxl) + fabsf(dyl)) + fabsf(dzl)) * 10.0f);
                    const float mh = __saturatef(((fabsf(dxh) + fabsf(dyh)) + fabsf(dzh)) * 10.0f);
                    const f32x2 bw = mul2(ring2[(p - r) & 7], sub2(one2, pk2(ml, mh)));
                    ar2[h] = fma2(sx2, bw, ar2[h]), ag2[h] = fma2(sy2, bw, ag2[h]), ab2[h] = fma2(sz2, bw, ab2[h]);
                    aw2[h] = add2(aw2[h], bw);
                }
            }
        };
        const int nblocks = (2 * k + R + 7) / 8, nfull = (2 * k + 1) / 8;  // blocks b < nfull have jj <= 2k for every p
        block(0, std::true_type{}, std::integral_constant<bool, true>{});
        int b = 1;
        for (; b < nfull; ++b) block(b, std::false_type{}, std::false_type{});
        for (; b < nblocks; ++b) block(b, std::false_type{}, std::true_type{});
#pragma unroll
        for (int h = 0; h < R / 2; ++h) {
            upk2(ar2[h], ar[2 * h], ar[2 * h + 1]), upk2(ag2[h], ag[2 * h], ag[2 * h + 1]);
            upk2(ab2[h], ab[2 * h], ab[2 * h + 1]), upk2(aw2[h], aw[2 * h], aw[2 * h + 1]);
        }
    }
    if (PASS == 0) {
        // results go back through shared memory (the input planes are dead) so that the global stores are coalesced
        __syncthreads();
        if (A.prm.debugVisualize != 2) {
#pragma unroll
            for (int r = 0; r < R; ++r) ar[r] = ar[r] / aw[r], ag[r] = ag[r] / aw[r], ab[r] = ab[r] / aw[r];
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
            float *q = pl + warp * H_PITCH + hpad(R * lane + r);
            q[0] = ar[r], q[PLANE] = ag[r], q[2 * PLANE] = ab[r];
        }
        __syncwarp();
        if (y0 < A.h) {
            const int bx = blockIdx.x * H_TW;
            for (int c = lane; c < H_TW; c += 32) {
                const int x = bx + c;
                if (x < A.w) {
                    const float *q = pl + warp * H_PITCH + hpad(c);
                    float4 v = make_float4(q[0], q[PLANE], q[2 * PLANE], 1.0f);
                    if (A.half) v.x = __half2float(__float2half_rn(v.x)), v.y = __half2float(__float2half_rn(v.y)), v.z = __half2float(__float2half_rn(v.z));
                    A.out[size_t(y0) * A.w + x] = v;
                }
            }
        }
        return;
    }
    // PASS 1: divide, composite (DenoiseCommon.hlsli:56-74) and store; a warp's 32 lanes write 512 contiguous bytes
    if (x0 >= A.w) return;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int y = y0 + r;
        if (y >= A.h) break;
        float cr = ar[r], cg = ag[r], cb = ab[r];
        if (A.prm.debugVisualize != 2) cr = cr / aw[r], cg = cg / aw[r], cb = cb / aw[r];
        if (A.prm.debugVisualize == 0) cr += cjx[r], cg += cjy[r], cb += cjz[r];
        else if (A.prm.debugVisualize == 3) cr = cjx[r], cg = cjy[r], cb = cjz[r];
        cr *= A.prm.exposure, cg *= A.prm.exposure, cb *= A.prm.exposure;
        if (A.prm.tonemap) {  // reinhardToneMap :33-38
            const float lum = luminance(cr, cg, cb);
            const float reinhard = lum / (lum + 1);
            const float s = reinhard / lum;
            cr = fmaxf(cr * s, 0.0f), cg = fmaxf(cg * s, 0.0f), cb = fmaxf(cb * s, 0.0f);
        }
        if (A.prm.gammaCorrect) {
            const float e = 1.0f / A.prm.gamma;
            cr = fminf(fmaxf(powf(cr, e), 0.0f), 1.0f), cg = fminf(fmaxf(powf(cg, e), 0.0f), 1.0f), cb = fminf(fmaxf(powf(cb, e), 0.0f), 1.0f);
        }
        if (A.half) cr = __half2float(__float2half_rn(cr)), cg = __half2float(__float2half_rn(cg)), cb = __half2float(__float2half_rn(cb));
        A.out[size_t(y) * A.w + x0] = make_float4(cr, cg, cb, 1.0f);
    }
}

// ---- rt_denoise_progressive (include/rt_core.h states the filter): one thread per pixel, taps read through L1.  Every
// tap's weight and sum are formed in the order the header and tests/progressive_denoise_reference.py give.
constexpr int PD_TX = 32, PD_TY = 8;

struct ProgDenoiseArgs {
    const float4 *beauty, *albedo, *normal;
    const float4 *src;  // (C, var) of the previous step (iterations)
    float4 *dst;        // (C, var), or (C, 1) rounded as a render target when `last`
    int w, h, step, last, half, nexp;
    float sigma_l, inv_a;
};

__device__ __forceinline__ float normal_weight(float4 np, float4 nq, int nexp) {
    float d = fmaxf(0.0f, (np.x * nq.x + np.y * nq.y) + np.z * nq.z);
    for (int i = 0; i < nexp; ++i) d = d * d;
    return d;
}

__device__ __forceinline__ void pd_store(const ProgDenoiseArgs &A, size_t i, float r, float g, float b, float var) {
    if (!A.last) {
        A.dst[i] = make_float4(r, g, b, var);
        return;
    }
    if (A.half) r = __half2float(__float2half_rn(r)), g = __half2float(__float2half_rn(g)), b = __half2float(__float2half_rn(b));
    A.dst[i] = make_float4(r, g, b, 1.0f);
}

// var0 of pixel (x, y), colour c, normal np: max(0, m2 - m1^2) of L over the wN-weighted 7 x 7 window of the colour image
// A.beauty, 0 for sky
__device__ __forceinline__ float window_variance(const ProgDenoiseArgs &A, int x, int y, float4 c, float4 np) {
    float var = 0.0f;
    if (np.w != 0.0f) {
        float sw = 0.0f, s1 = 0.0f, s2 = 0.0f;
        for (int dy = -3; dy <= 3; ++dy) {
            const int qy = y + dy;
            if (qy < 0 || qy >= A.h) continue;
#pragma unroll
            for (int dx = -3; dx <= 3; ++dx) {
                const int qx = x + dx;
                if (qx < 0 || qx >= A.w) continue;
                const size_t j = size_t(qy) * A.w + qx;
                float wn = 1.0f;
                float4 cq = c;
                if (dx != 0 || dy != 0) {
                    wn = normal_weight(np, __ldg(A.normal + j), A.nexp);
                    if (wn == 0.0f) continue;
                    cq = __ldg(A.beauty + j);
                }
                const float l = luminance(cq.x, cq.y, cq.z);
                s1 = s1 + wn * l, s2 = s2 + wn * (l * l), sw = sw + wn;
            }
        }
        const float m1 = s1 / sw, m2 = s2 / sw;
        var = fmaxf(0.0f, m2 - m1 * m1);
    }
    return var;
}

// (C, var0): var0 = max(0, m2 - m1^2) of L over the wN-weighted 7 x 7 window
__global__ void __launch_bounds__(PD_TX * PD_TY) k_pd_variance(const __grid_constant__ ProgDenoiseArgs A) {
    const int x = blockIdx.x * PD_TX + threadIdx.x, y = blockIdx.y * PD_TY + threadIdx.y;
    if (x >= A.w || y >= A.h) return;
    const size_t i = size_t(y) * A.w + x;
    const float4 c = __ldg(A.beauty + i), np = __ldg(A.normal + i);
    pd_store(A, i, c.x, c.y, c.z, window_variance(A, x, y, c, np));
}

// one a-trous iteration at step A.step: (C, var) from A.src -> A.dst
__global__ void __launch_bounds__(PD_TX * PD_TY) k_pd_atrous(const __grid_constant__ ProgDenoiseArgs A) {
    const int x = blockIdx.x * PD_TX + threadIdx.x, y = blockIdx.y * PD_TY + threadIdx.y;
    if (x >= A.w || y >= A.h) return;
    const size_t i = size_t(y) * A.w + x;
    const float4 cp = __ldg(A.src + i), np = __ldg(A.normal + i);
    if (np.w == 0.0f) {  // sky: copied
        pd_store(A, i, cp.x, cp.y, cp.z, cp.w);
        return;
    }
    const float kH[3] = {0.25f, 0.5f, 0.25f};
    const float kB[5] = {0.0625f, 0.25f, 0.375f, 0.25f, 0.0625f};
    // g(p): the 3 x 3 wN-weighted prefilter of var
    float gs = 0.0f, gw = 0.0f;
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy) {
        const int qy = y + dy;
        if (qy < 0 || qy >= A.h) continue;
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx) {
            const int qx = x + dx;
            if (qx < 0 || qx >= A.w) continue;
            const size_t j = size_t(qy) * A.w + qx;
            float wn = 1.0f, v = cp.w;
            if (dx != 0 || dy != 0) {
                wn = normal_weight(np, __ldg(A.normal + j), A.nexp);
                if (wn == 0.0f) continue;
                v = __ldg(A.src + j).w;
            }
            const float wg = (kH[dx + 1] * kH[dy + 1]) * wn;
            if (wg == 0.0f) continue;
            gs = gs + wg * v, gw = gw + wg;
        }
    }
    const float g = gs / gw;
    const float inv_l = 1.0f / (A.sigma_l * sqrtf(g) + 1e-10f);
    const float lp = luminance(cp.x, cp.y, cp.z);
    const float4 ap = __ldg(A.albedo + i);
    float sr = 0.0f, sg = 0.0f, sb = 0.0f, sv = 0.0f, sw = 0.0f;
#pragma unroll
    for (int dy = -2; dy <= 2; ++dy) {
        const int qy = y + A.step * dy;
        if (qy < 0 || qy >= A.h) continue;
#pragma unroll
        for (int dx = -2; dx <= 2; ++dx) {
            const int qx = x + A.step * dx;
            if (qx < 0 || qx >= A.w) continue;
            const size_t j = size_t(qy) * A.w + qx;
            float w = kB[2] * kB[2];
            float4 cq = cp;
            if (dx != 0 || dy != 0) {
                const float wn = normal_weight(np, __ldg(A.normal + j), A.nexp);
                if (wn == 0.0f) continue;
                cq = __ldg(A.src + j);
                const float4 aq = __ldg(A.albedo + j);
                const float dl = fabsf(lp - luminance(cq.x, cq.y, cq.z));
                const float da = (fabsf(ap.x - aq.x) + fabsf(ap.y - aq.y)) + fabsf(ap.z - aq.z);
                w = ((kB[dx + 2] * kB[dy + 2]) * wn) * expf(-(dl * inv_l + da * A.inv_a));
                if (w == 0.0f) continue;
            }
            sr = sr + w * cq.x, sg = sg + w * cq.y, sb = sb + w * cq.z;
            sv = sv + (w * w) * cq.w, sw = sw + w;
        }
    }
    pd_store(A, i, sr / sw, sg / sw, sb / sw, sv / (sw * sw));
}

// ---- rt_denoise_temporal (include/rt_core.h states the temporal pass): reproject and blend into the history, then the
// variance of the integrated colour, then the a-trous iterations above.  tests/temporal_denoise_reference.py restates it.
struct TemporalArgs {
    const float4 *beauty, *normal, *position;
    const float4 *prev;  // prev_history (4 planes), nullptr: no history
    float4 *hist;        // history (4 planes)
    int w, h;
    float eye[3], jitter[2], U[3], V[3], W[3];  // the previous frame's camera
    float alpha_c, alpha_m, normal_cos, pos_tol;
};

__device__ __forceinline__ float dot3(float ax, float ay, float az, const float b[3]) { return (ax * b[0] + ay * b[1]) + az * b[2]; }

// One pixel of the reprojection and blend.  MOTION (rt_denoise_temporal_motion): the point projected into the previous
// frame and compared with the history's positions is Q = prev_pos[i] instead of this frame's P.
template <bool MOTION>
__device__ __forceinline__ void td_reproject(const TemporalArgs &A, const float4 *prev_pos) {
    const int x = blockIdx.x * PD_TX + threadIdx.x, y = blockIdx.y * PD_TY + threadIdx.y;
    if (x >= A.w || y >= A.h) return;
    const size_t plane = size_t(A.w) * A.h, i = size_t(y) * A.w + x;
    const float4 c = __ldg(A.beauty + i), np = __ldg(A.normal + i), pp = __ldg(A.position + i);
    float hr = 0.0f, hg = 0.0f, hb = 0.0f, hn = 0.0f, h1 = 0.0f, h2 = 0.0f;
    if (A.prev && np.w == 1.0f) {
        const float4 q = MOTION ? __ldg(prev_pos + i) : pp;
        // o' is the progressive primary ray's origin (primary_ray in shade.cuh, jitterScale 30)
        const float rx = q.x - (A.eye[0] + A.jitter[0] * 30.0f), ry = q.y - (A.eye[1] + A.jitter[1] * 30.0f), rz = q.z - (A.eye[2] + 0.0f);
        const float zc = dot3(rx, ry, rz, A.W) / dot3(A.W[0], A.W[1], A.W[2], A.W);
        const float sx = (dot3(rx, ry, rz, A.U) / dot3(A.U[0], A.U[1], A.U[2], A.U)) / zc;
        const float sy = -((dot3(rx, ry, rz, A.V) / dot3(A.V[0], A.V[1], A.V[2], A.V)) / zc);
        const float fx = ((sx + 1.0f) * 0.5f) * float(A.w) - 0.5f, fy = ((sy + 1.0f) * 0.5f) * float(A.h) - 0.5f;
        // outside (-1, w) x (-1, h) every tap is outside the image or has weight 0 (and NaN fails the test)
        if (zc > 0.0f && fx > -1.0f && fx < float(A.w) && fy > -1.0f && fy < float(A.h)) {
            const float x0f = floorf(fx), y0f = floorf(fy);
            const float ax = fx - x0f, ay = fy - y0f;
            const int x0 = int(x0f), y0 = int(y0f);
            const float lim = A.pos_tol * sqrtf((rx * rx + ry * ry) + rz * rz);
            float sw = 0.0f;
#pragma unroll
            for (int dy = 0; dy < 2; ++dy) {
#pragma unroll
                for (int dx = 0; dx < 2; ++dx) {
                    const int qx = x0 + dx, qy = y0 + dy;
                    if (qx < 0 || qy < 0 || qx >= A.w || qy >= A.h) continue;
                    const float wt = (dx ? ax : 1.0f - ax) * (dy ? ay : 1.0f - ay);
                    if (wt == 0.0f) continue;
                    const size_t j = size_t(qy) * A.w + qx;
                    const float4 nq = __ldg(A.prev + 2 * plane + j);
                    if (nq.w != 1.0f || (np.x * nq.x + np.y * nq.y) + np.z * nq.z < A.normal_cos) continue;
                    const float4 pq = __ldg(A.prev + 3 * plane + j);
                    const float ex = pq.x - q.x, ey = pq.y - q.y, ez = pq.z - q.z;
                    if (sqrtf((ex * ex + ey * ey) + ez * ez) > lim) continue;
                    const float4 cq = __ldg(A.prev + j), mq = __ldg(A.prev + plane + j);
                    hr = hr + wt * cq.x, hg = hg + wt * cq.y, hb = hb + wt * cq.z, hn = hn + wt * cq.w;
                    h1 = h1 + wt * mq.x, h2 = h2 + wt * mq.y, sw = sw + wt;
                }
            }
            if (sw > 0.0f) hr = hr / sw, hg = hg / sw, hb = hb / sw, hn = hn / sw, h1 = h1 / sw, h2 = h2 / sw;
        }
    }
    const float n = fminf(hn + 1.0f, 32.0f);
    const float a = fmaxf(1.0f / n, A.alpha_c), am = fmaxf(1.0f / n, A.alpha_m);
    const float l = luminance(c.x, c.y, c.z);
    A.hist[i] = make_float4((1.0f - a) * hr + a * c.x, (1.0f - a) * hg + a * c.y, (1.0f - a) * hb + a * c.z, n);
    A.hist[plane + i] = make_float4((1.0f - am) * h1 + am * l, (1.0f - am) * h2 + am * (l * l), 0.0f, 0.0f);
    A.hist[2 * plane + i] = np;
    A.hist[3 * plane + i] = pp;
}

__global__ void __launch_bounds__(PD_TX * PD_TY) k_td_reproject(const __grid_constant__ TemporalArgs A) { td_reproject<false>(A, nullptr); }

__global__ void __launch_bounds__(PD_TX * PD_TY) k_td_reproject_motion(const __grid_constant__ TemporalArgs A, const float4 *prev_pos) {
    td_reproject<true>(A, prev_pos);
}

// (C, var0) of the integrated colour: A.beauty = history plane 0 (C, n), A.src = history plane 1 (m1, m2)
__global__ void __launch_bounds__(PD_TX * PD_TY) k_td_variance(const __grid_constant__ ProgDenoiseArgs A) {
    const int x = blockIdx.x * PD_TX + threadIdx.x, y = blockIdx.y * PD_TY + threadIdx.y;
    if (x >= A.w || y >= A.h) return;
    const size_t i = size_t(y) * A.w + x;
    const float4 c = __ldg(A.beauty + i), np = __ldg(A.normal + i);
    float var;
    if (c.w >= 4.0f) {
        const float4 m = __ldg(A.src + i);
        var = fmaxf(0.0f, m.y - m.x * m.x);
    } else {
        var = window_variance(A, x, y, c, np);
    }
    pd_store(A, i, c.x, c.y, c.z, var);
}

bool overlap(const void *a, uint64_t na, const void *b, uint64_t nb) { return uintptr_t(a) < uintptr_t(b) + nb && uintptr_t(b) < uintptr_t(a) + na; }

// The a-trous stage's parameters and the image size, as both progressive denoisers check them and pass them to the kernels.
int pd_args(rt_context *ctx, const rt_progressive_denoise_params *prm, uint32_t width, uint32_t height, ProgDenoiseArgs &A) {
    RT_REQUIRE(width > 0 && height > 0, "empty image");
    RT_REQUIRE(width <= 0x7FFFFFFFu && height <= 65535u * PD_TY, "image too large for one launch");
    RT_REQUIRE(prm->iterations <= 5 && prm->normal_exponent_log2 <= 8, "iterations 0..5, normal_exponent_log2 0..8");
    RT_REQUIRE(prm->sigma_luminance > 0.0f && prm->sigma_luminance <= 3.4e38f, "sigma_luminance must be finite and > 0");
    RT_REQUIRE(prm->sigma_albedo >= 0.0f && prm->sigma_albedo <= 3.4e38f, "sigma_albedo must be finite and >= 0");
    A = ProgDenoiseArgs{};
    A.w = int(width), A.h = int(height);
    A.half = int(ctx->render_options.half_render_targets);
    A.nexp = int(prm->normal_exponent_log2);
    A.sigma_l = prm->sigma_luminance;
    A.inv_a = prm->sigma_albedo > 0.0f ? 1.0f / prm->sigma_albedo : 0.0f;
    return RT_OK;
}

// `first` writes (C, var0) to tmp[0] (or out when there are no iterations), then one k_pd_atrous per iteration ping-pongs
// through tmp and the last one writes out
void pd_launch(rt_context *ctx, void (*first)(ProgDenoiseArgs), ProgDenoiseArgs A, int n, float *tmp, float *out) {
    const dim3 grid(rt_div_up(uint32_t(A.w), PD_TX), rt_div_up(uint32_t(A.h), PD_TY)), block(PD_TX, PD_TY);
    float4 *ping[2] = {reinterpret_cast<float4 *>(tmp), reinterpret_cast<float4 *>(tmp) + size_t(A.w) * A.h};
    A.dst = n == 0 ? reinterpret_cast<float4 *>(out) : ping[0];
    A.last = n == 0;
    first<<<grid, block, 0, ctx->stream>>>(A);
    for (int it = 0; it < n; ++it) {
        A.src = ping[it & 1];
        A.step = 1 << it;
        A.last = it == n - 1;
        A.dst = A.last ? reinterpret_cast<float4 *>(out) : ping[(it + 1) & 1];
        k_pd_atrous<<<grid, block, 0, ctx->stream>>>(A);
    }
    ctx->launches += 1 + n;
}

}  // namespace

extern "C" int rt_denoise_progressive(rt_context *ctx, const float *beauty, const float *albedo, const float *normal, float *tmp,
                                      float *out, uint32_t width, uint32_t height, const rt_progressive_denoise_params *prm) {
    RT_REQUIRE(ctx && beauty && albedo && normal && tmp && out && prm, "null argument");
    RT_REQUIRE(((uintptr_t(beauty) | uintptr_t(albedo) | uintptr_t(normal) | uintptr_t(tmp) | uintptr_t(out)) & 15) == 0,
               "images must be 16-byte aligned");
    ProgDenoiseArgs A;
    if (const int e = pd_args(ctx, prm, width, height, A)) return e;
    // byte ranges [p, p + n): out and tmp are written, so neither may share a byte with any other argument
    const uint64_t img = uint64_t(width) * height * 16;
    for (const float *in : {beauty, albedo, normal}) {
        RT_REQUIRE(!overlap(out, img, in, img), "out overlaps an input");
        RT_REQUIRE(!overlap(tmp, 2 * img, in, img), "tmp overlaps an input");
    }
    RT_REQUIRE(!overlap(out, img, tmp, 2 * img), "out overlaps tmp");
    RT_CUDA(cudaSetDevice(ctx->device));
    A.beauty = reinterpret_cast<const float4 *>(beauty);
    A.albedo = reinterpret_cast<const float4 *>(albedo);
    A.normal = reinterpret_cast<const float4 *>(normal);
    pd_launch(ctx, k_pd_variance, A, int(prm->iterations), tmp, out);
    RT_LAUNCH_CHECK();
    return RT_OK;
}

// rt_denoise_temporal (motion == false) and rt_denoise_temporal_motion (motion == true: previous_position is Q)
static int denoise_temporal(rt_context *ctx, const float *beauty, const float *albedo, const float *normal, const float *position,
                            const float *previous_position, bool motion, const rt_camera_params *prev_camera, const float *prev_history,
                            float *history, float *tmp, float *out, uint32_t width, uint32_t height, const rt_temporal_denoise_params *prm) {
    RT_REQUIRE(ctx && beauty && albedo && normal && position && (previous_position || !motion) && history && tmp && out && prm,
               "null argument");
    RT_REQUIRE((prev_camera == nullptr) == (prev_history == nullptr), "prev_camera and prev_history are both given or both NULL");
    RT_REQUIRE(((uintptr_t(beauty) | uintptr_t(albedo) | uintptr_t(normal) | uintptr_t(position) | uintptr_t(previous_position) |
                 uintptr_t(prev_history) | uintptr_t(history) | uintptr_t(tmp) | uintptr_t(out)) & 15) == 0,
               "images must be 16-byte aligned");
    ProgDenoiseArgs A;
    if (const int e = pd_args(ctx, &prm->spatial, width, height, A)) return e;
    RT_REQUIRE(prm->alpha_color > 0.0f && prm->alpha_color <= 1.0f, "alpha_color in (0, 1]");
    RT_REQUIRE(prm->alpha_moments > 0.0f && prm->alpha_moments <= 1.0f, "alpha_moments in (0, 1]");
    RT_REQUIRE(prm->normal_cos >= -1.0f && prm->normal_cos <= 1.0f, "normal_cos in [-1, 1]");
    RT_REQUIRE(prm->position_tolerance >= 0.0f && prm->position_tolerance <= 3.4e38f, "position_tolerance must be finite and >= 0");
    // byte ranges [p, p + n): history, tmp and out are written, so none may share a byte with any other argument
    const uint64_t img = uint64_t(width) * height * 16;
    for (const float *in : {beauty, albedo, normal, position, previous_position, prev_history}) {
        const uint64_t n = in == prev_history ? 4 * img : img;
        if (!in) continue;
        RT_REQUIRE(!overlap(history, 4 * img, in, n), "history overlaps an input or prev_history");
        RT_REQUIRE(!overlap(tmp, 2 * img, in, n), "tmp overlaps an input or prev_history");
        RT_REQUIRE(!overlap(out, img, in, n), "out overlaps an input or prev_history");
    }
    RT_REQUIRE(!overlap(history, 4 * img, tmp, 2 * img) && !overlap(history, 4 * img, out, img) && !overlap(out, img, tmp, 2 * img),
               "history, tmp and out overlap");
    RT_CUDA(cudaSetDevice(ctx->device));
    TemporalArgs T{};
    T.beauty = reinterpret_cast<const float4 *>(beauty);
    T.normal = reinterpret_cast<const float4 *>(normal);
    T.position = reinterpret_cast<const float4 *>(position);
    T.prev = reinterpret_cast<const float4 *>(prev_history);
    T.hist = reinterpret_cast<float4 *>(history);
    T.w = int(width), T.h = int(height);
    if (prev_camera) {
        for (int k = 0; k < 3; ++k)
            T.eye[k] = prev_camera->worldEyePos[k], T.U[k] = prev_camera->U[k], T.V[k] = prev_camera->V[k], T.W[k] = prev_camera->W[k];
        T.jitter[0] = prev_camera->jitters[0], T.jitter[1] = prev_camera->jitters[1];
    }
    T.alpha_c = prm->alpha_color, T.alpha_m = prm->alpha_moments;
    T.normal_cos = prm->normal_cos, T.pos_tol = prm->position_tolerance;
    const dim3 grid(rt_div_up(width, PD_TX), rt_div_up(height, PD_TY)), block(PD_TX, PD_TY);
    if (motion) k_td_reproject_motion<<<grid, block, 0, ctx->stream>>>(T, reinterpret_cast<const float4 *>(previous_position));
    else k_td_reproject<<<grid, block, 0, ctx->stream>>>(T);
    ctx->launches += 1;
    const size_t plane = size_t(width) * height;
    A.beauty = T.hist;  // (C, n): the integrated colour is what the variance and the a-trous stage filter
    A.src = T.hist + plane;
    A.albedo = reinterpret_cast<const float4 *>(albedo);
    A.normal = T.normal;
    pd_launch(ctx, k_td_variance, A, int(prm->spatial.iterations), tmp, out);
    RT_LAUNCH_CHECK();
    return RT_OK;
}

extern "C" int rt_denoise_temporal(rt_context *ctx, const float *beauty, const float *albedo, const float *normal, const float *position,
                                   const rt_camera_params *prev_camera, const float *prev_history, float *history, float *tmp, float *out,
                                   uint32_t width, uint32_t height, const rt_temporal_denoise_params *prm) {
    return denoise_temporal(ctx, beauty, albedo, normal, position, nullptr, false, prev_camera, prev_history, history, tmp, out, width,
                            height, prm);
}

extern "C" int rt_denoise_temporal_motion(rt_context *ctx, const float *beauty, const float *albedo, const float *normal,
                                          const float *position, const float *previous_position, const rt_camera_params *prev_camera,
                                          const float *prev_history, float *history, float *tmp, float *out, uint32_t width,
                                          uint32_t height, const rt_temporal_denoise_params *prm) {
    return denoise_temporal(ctx, beauty, albedo, normal, position, previous_position, true, prev_camera, prev_history, history, tmp, out,
                            width, height, prm);
}

extern "C" int rt_denoise(rt_context *ctx, const float *direct, const float *indirect_specular, float *tmp, float *out, uint32_t width,
                          uint32_t height, const rt_denoiser_params *prm) {
    RT_REQUIRE(ctx && direct && indirect_specular && tmp && out && prm, "null argument");
    RT_REQUIRE(width > 0 && height > 0, "empty image");
    RT_REQUIRE(((uintptr_t(direct) | uintptr_t(indirect_specular) | uintptr_t(tmp) | uintptr_t(out)) & 15) == 0, "images must be 16-byte aligned");
    RT_CUDA(cudaSetDevice(ctx->device));
    DenoiseArgs A{};
    A.joint = reinterpret_cast<const float4 *>(direct);
    A.w = int(width), A.h = int(height);
    // maxKernelSize beyond MAX_EXTENT reads outside the reference's LDS tile (undefined); clamp.
    A.k = prm->maxKernelSize < 0 ? 0 : (prm->maxKernelSize > MAX_EXTENT ? MAX_EXTENT : prm->maxKernelSize);
    A.prm = *prm;
    A.half = int(ctx->render_options.half_render_targets);
    // per-group weight table: BilateralFilter.hlsli:80-90
    for (int i = -MAX_EXTENT; i <= MAX_EXTENT; ++i) {
        int ai = i < 0 ? -i : i;
        float radius = float(prm->maxKernelSize);
        float den = 0.001f + (radius * 0.8f < 0 ? -(radius * 0.8f) : radius * 0.8f);
        int idx = int(float(ai * (KERNEL_TAPS - 1)) / den);
        idx = idx < 0 ? 0 : (idx > KERNEL_TAPS ? KERNEL_TAPS : idx);
        A.wts[i + MAX_EXTENT] = idx < 2 ? 1.0f : (idx < 3 ? 0.9f : (idx < 4 ? 0.75f : (idx < 5 ? 0.6f : (idx < 6 ? 0.5f : 0.0f))));
    }
    // the opt-in is a per-device attribute of the function: set it on every call (a process may hold contexts on several GPUs)
    RT_CUDA(cudaFuncSetAttribute(k_denoise<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(H_SMEM)));
    RT_CUDA(cudaFuncSetAttribute(k_denoise<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(V_SMEM)));
    A.input = reinterpret_cast<const float4 *>(indirect_specular);
    A.out = reinterpret_cast<float4 *>(tmp);
    k_denoise<0><<<dim3(rt_div_up(width, H_TW), rt_div_up(height, H_TH)), kThreadsDn, H_SMEM, ctx->stream>>>(A);
    A.input = reinterpret_cast<const float4 *>(tmp);
    A.out = reinterpret_cast<float4 *>(out);
    const size_t v_smem = (6 * size_t(V_TH + 2 * A.k + 8) * V_TW + 64) * sizeof(float);
    k_denoise<1><<<dim3(rt_div_up(width, V_TW), rt_div_up(height, V_TH)), kThreadsDn, v_smem, ctx->stream>>>(A);
    ctx->launches += 2;
    RT_LAUNCH_CHECK();
    return RT_OK;
}

// ------------------------------------------------------------------------------------------------ adaptive sampling
// rt_adaptive_update: one thread per pixel over 16 x 16 tiles; the 18 x 18 window of "error at most threshold" flags the
// tile's one-pixel dilation reads is computed once per block into shared memory.
namespace {

constexpr int AU_T = 16;

struct AdaptiveArgs {
    const float2 *moments;
    uint32_t *counts;
    uint32_t *active;
    int w, h;
    float threshold, floor;
    uint32_t min_samples, max_samples;
};

// e_q <= threshold for pixel (x, y); true outside the image, which the dilation ignores
__device__ __forceinline__ bool adaptive_error_ok(const AdaptiveArgs &A, int x, int y) {
    if (x < 0 || y < 0 || x >= A.w || y >= A.h) return true;
    const size_t i = size_t(y) * A.w + x;
    const uint32_t n = A.counts[i] & ~RT_ADAPTIVE_CONVERGED;
    if (n < 2) return false;  // sigma = +inf
    const float2 m = __ldg(A.moments + i);
    const float sigma = sqrtf(fmaxf(0.0f, m.y - m.x * m.x) / float(n - 1));
    return sigma / (m.x + A.floor) <= A.threshold;  // NaN fails
}

__global__ void __launch_bounds__(AU_T * AU_T) k_adaptive_update(const __grid_constant__ AdaptiveArgs A) {
    __shared__ uint8_t ok[AU_T + 2][AU_T + 2];
    const int bx = blockIdx.x * AU_T, by = blockIdx.y * AU_T;
    for (int k = threadIdx.y * AU_T + threadIdx.x; k < (AU_T + 2) * (AU_T + 2); k += AU_T * AU_T)
        ok[k / (AU_T + 2)][k % (AU_T + 2)] = adaptive_error_ok(A, bx + k % (AU_T + 2) - 1, by + k / (AU_T + 2) - 1) ? 1 : 0;
    __syncthreads();
    const int x = bx + threadIdx.x, y = by + threadIdx.y;
    bool active = false;
    if (x < A.w && y < A.h) {
        const size_t i = size_t(y) * A.w + x;
        const uint32_t c = A.counts[i], n = c & ~RT_ADAPTIVE_CONVERGED;
        bool conv = (c & RT_ADAPTIVE_CONVERGED) || n >= A.max_samples;
        if (!conv && n >= A.min_samples) {
            conv = true;
#pragma unroll
            for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                for (int dx = 0; dx < 3; ++dx) conv = conv && ok[threadIdx.y + dy][threadIdx.x + dx];
        }
        // only bit 31 of a neighbour's word changes, which adaptive_error_ok masks off
        if (conv && !(c & RT_ADAPTIVE_CONVERGED)) A.counts[i] = c | RT_ADAPTIVE_CONVERGED;
        active = !conv;
    }
    const unsigned b = __ballot_sync(0xffffffffu, active);
    if (A.active && ((threadIdx.y * AU_T + threadIdx.x) & 31) == 0 && b) atomicAdd(A.active, uint32_t(__popc(b)));  // one lane per warp
}

}  // namespace

extern "C" int rt_adaptive_update(rt_context *ctx, const float *moments, uint32_t *counts, uint32_t width, uint32_t height,
                                  const rt_adaptive_params *prm, uint32_t *active_count) {
    RT_REQUIRE(ctx && moments && counts && prm, "null argument");
    RT_REQUIRE(((uintptr_t(counts) | uintptr_t(active_count)) & 3) == 0 && (uintptr_t(moments) & 7) == 0,
               "counts and active_count must be 4-byte and moments 8-byte aligned");
    RT_REQUIRE(width > 0 && height > 0, "empty image");
    RT_REQUIRE(width <= 0x7FFFFFFFu && height <= 65535u * AU_T, "image too large for one launch");
    RT_REQUIRE(prm->threshold >= 0.0f && prm->threshold <= 3.4e38f, "threshold must be finite and >= 0");
    RT_REQUIRE(prm->floor > 0.0f && prm->floor <= 3.4e38f, "floor must be finite and > 0");
    RT_REQUIRE(prm->min_samples >= 1 && prm->min_samples <= prm->max_samples && prm->max_samples <= 0x7FFFFFFFu,
               "1 <= min_samples <= max_samples <= 2^31 - 1");
    const uint64_t px = uint64_t(width) * height;
    RT_REQUIRE(!overlap(counts, 4 * px, moments, 8 * px), "counts overlaps moments");
    RT_REQUIRE(!active_count || (!overlap(active_count, 4, moments, 8 * px) && !overlap(active_count, 4, counts, 4 * px)),
               "active_count overlaps moments or counts");
    RT_CUDA(cudaSetDevice(ctx->device));
    if (active_count) RT_CUDA(cudaMemsetAsync(active_count, 0, 4, ctx->stream));
    const AdaptiveArgs A{reinterpret_cast<const float2 *>(moments), counts, active_count, int(width), int(height), prm->threshold, prm->floor,
                         prm->min_samples, prm->max_samples};
    k_adaptive_update<<<dim3(rt_div_up(width, AU_T), rt_div_up(height, AU_T)), dim3(AU_T, AU_T), 0, ctx->stream>>>(A);
    ctx->launches++;
    RT_LAUNCH_CHECK();
    return RT_OK;
}
