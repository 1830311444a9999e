// preprocess.cu -- per-Gaussian forward stage: near-plane cull, projection, EWA covariance,
// conic, screen radius, tile rectangle, SH -> RGB, per-tile instance counting.
//
// Replaces preprocessCUDA<3> (DGR/cuda_rasterizer/forward.cu:155-256) with its helpers
// in_frustum (auxiliary.h:139-164), computeCov3D (forward.cu:118-152), computeCov2D
// (forward.cu:74-113), computeColorFromSH (forward.cu:20-71), ndc2Pix / getRect
// (auxiliary.h:41-56) and checkFrustum (rasterizer_impl.cu:54-66).
//
// All integer-determining arithmetic follows the op order of the reference's sm_100a SASS; see
// common.cuh for the policy.  Differences in structure (B200-first):
//   * one packed 48-byte record per Gaussian instead of five SoA arrays: the blend kernels
//     fetch it with three 128-bit loads;
//   * the tile rectangle is stored (8 bytes) so the binning pass never recomputes getRect;
//   * per-tile instance counts are accumulated here (RED.ADD on an L2-resident 32 KB table),
//     which replaces the per-Gaussian prefix sum + 64-bit global sort of the reference by a
//     per-tile segmented sort (binning.cu);
//   * conservative alpha>=1/255 extents are derived per Gaussian for sub-tile culling in the
//     blend kernels.
#include <cstdio>

#include "common.cuh"
#include "frosting_attr.cuh"

namespace fb200 {

namespace {

// SH basis constants, the float values nvcc materialised from DGR/cuda_rasterizer/auxiliary.h:22-39
__device__ constexpr float kC0 = 0.28209479177387814f;
__device__ constexpr float kC1 = 0.4886025119029199f;
__device__ constexpr float kC2_0 = 1.0925484305920792f;
__device__ constexpr float kC2_1 = -1.0925484305920792f;
__device__ constexpr float kC2_2 = 0.31539156525252005f;
__device__ constexpr float kC2_3 = -1.0925484305920792f;
__device__ constexpr float kC2_4 = 0.5462742152960396f;
__device__ constexpr float kC3_0 = -0.5900435899266435f;
__device__ constexpr float kC3_1 = 2.890611442640554f;
__device__ constexpr float kC3_2 = -0.4570457994644658f;
__device__ constexpr float kC3_3 = 0.3731763325901154f;
__device__ constexpr float kC3_4 = -0.4570457994644658f;
__device__ constexpr float kC3_5 = 1.445305721320277f;
__device__ constexpr float kC3_6 = -0.5900435899266435f;

struct Cov3 {
    float c0, c1, c2, c3, c4, c5;
};

// computeCov3D, forward.cu:118-152.  q = (r,x,y,z) is used as given (no normalisation).
__device__ __forceinline__ Cov3 cov3d_from_scale_rot(float sx_in, float sy_in, float sz_in, float mod,
                                                     float r, float x, float y, float z) {
    const float sx = fmul(sx_in, mod), sy = fmul(sy_in, mod), sz = fmul(sz_in, mod);
    const float xz = fmul(x, z), rx = fmul(r, x), rz = fmul(r, z), yy = fmul(y, y), zz = fmul(z, z);
    // rotation entries (glm column-major R; Rcr = column c, row r)
    const float e00 = fadd(yy, zz);
    const float e11 = ffma(x, x, zz);
    const float e22 = ffma(x, x, yy);
    const float R00 = fadd(-fadd(e00, e00), 1.0f);
    const float R11 = fadd(-fadd(e11, e11), 1.0f);
    const float R22 = fadd(-fadd(e22, e22), 1.0f);
    float u;
    u = ffma(x, y, -rz); const float R01 = fadd(u, u);   // 2(xy - rz)  col0,row1
    u = ffma(r, y, xz);  const float R02 = fadd(u, u);   // 2(xz + ry)  col0,row2
    u = ffma(x, y, rz);  const float R10 = fadd(u, u);   // 2(xy + rz)  col1,row0
    u = ffma(y, z, -rx); const float R12 = fadd(u, u);   // 2(yz - rx)  col1,row2
    u = ffma(-r, y, xz); const float R20 = fadd(u, u);   // 2(xz - ry)  col2,row0
    u = ffma(y, z, rx);  const float R21 = fadd(u, u);   // 2(yz + rx)  col2,row1
    // M = S * R : M[c][r] = s_r * R[c][r]   (the structural zeros of S add exact zeros)
    const float M00 = fmul(sx, R00), M01 = fmul(sy, R01), M02 = fmul(sz, R02);
    const float M10 = fmul(sx, R10), M11 = fmul(sy, R11), M12 = fmul(sz, R12);
    const float M20 = fmul(sx, R20), M21 = fmul(sy, R21), M22 = fmul(sz, R22);
    // Sigma = M^T M : Sigma[c][r] = dot(M[r][.], M[c][.])
    Cov3 s;
    s.c0 = dot3x(M00, M00, M01, M01, M02, M02);
    s.c1 = dot3x(M00, M10, M01, M11, M02, M12);
    s.c2 = dot3x(M00, M20, M01, M21, M02, M22);
    s.c3 = dot3x(M10, M10, M11, M11, M12, M12);
    s.c4 = dot3x(M10, M20, M11, M21, M12, M22);
    s.c5 = dot3x(M20, M20, M21, M21, M22, M22);
    return s;
}

// computeCov2D, forward.cu:74-113 -> (a, b, c) with the 0.3 low-pass added.
__device__ __forceinline__ float3 cov2d(float px, float py, float pz, float focal_x, float focal_y,
                                        float tan_fovx, float tan_fovy, const Cov3& S,
                                        const float* __restrict__ v) {
    const float tx = affine_row(v, 0, px, py, pz);
    const float ty = affine_row(v, 1, px, py, pz);
    const float tz = affine_row(v, 2, px, py, pz);
    const float limx = fmul(tan_fovx, 1.3f);
    const float limy = fmul(tan_fovy, 1.3f);
    const float txtz = __fdiv_rn(tx, tz);
    const float tytz = __fdiv_rn(ty, tz);
    const float cx = fminf(fmaxf(txtz, -limx), limx);
    const float cy = fminf(fmaxf(tytz, -limy), limy);
    const float tz2 = fmul(tz, tz);
    const float J00 = __fdiv_rn(focal_x, tz);
    const float J02 = __fdiv_rn(fmul(fmul(tz, -cx), focal_x), tz2);   // -(fx * (cx*tz)) / tz^2
    const float J11 = __fdiv_rn(focal_y, tz);
    const float J12 = __fdiv_rn(fmul(fmul(tz, -cy), focal_y), tz2);
    // T = W * J (third column of J is zero).  W[k][r]: W[0]=(v0,v4,v8) W[1]=(v1,v5,v9) W[2]=(v2,v6,v10)
    const float T00 = ffma(v[2], J02, fmul(v[0], J00));
    const float T01 = ffma(v[6], J02, fmul(v[4], J00));
    const float T02 = ffma(v[10], J02, fmul(v[8], J00));
    const float T10 = ffma(v[2], J12, fmul(v[1], J11));
    const float T11 = ffma(v[6], J12, fmul(v[5], J11));
    const float T12 = ffma(v[10], J12, fmul(v[9], J11));
    // P1 = T^T * Vrk^T : P1[c][r] = T[r][0]*S0c + T[r][1]*S1c + T[r][2]*S2c
    const float P00 = dot3x(T00, S.c0, T01, S.c1, T02, S.c2);
    const float P10 = dot3x(T00, S.c1, T01, S.c3, T02, S.c4);
    const float P20 = dot3x(T00, S.c2, T01, S.c4, T02, S.c5);
    const float P01 = dot3x(T10, S.c0, T11, S.c1, T12, S.c2);
    const float P11 = dot3x(T10, S.c1, T11, S.c3, T12, S.c4);
    const float P21 = dot3x(T10, S.c2, T11, S.c4, T12, S.c5);
    // cov = P1 * T
    const float cov00 = dot3x(P00, T00, P10, T01, P20, T02);
    const float cov01 = dot3x(P01, T00, P11, T01, P21, T02);
    const float cov11 = dot3x(P01, T10, P11, T11, P21, T12);
    return make_float3(fadd(cov00, 0.3f), cov01, fadd(cov11, 0.3f));
}

// ndc2Pix, auxiliary.h:41-44: evaluated in double with a contracted DFMA.
__device__ __forceinline__ float ndc2pix(float v, int S) {
    return (float)__dmul_rn(__fma_rn(__dadd_rn((double)v, 1.0), (double)S, -1.0), 0.5);
}

__device__ __forceinline__ uint32_t rect_coord(float v, uint32_t g) {
    int i = __float2int_rz(fmul(v, 0.0625f));
    i = max(0, i);
    return min(g, (uint32_t)i);
}

// The SH row of one Gaussian into registers: 3*M floats, coefficient-major, RGB innermost.
template <bool kAligned>
__device__ __forceinline__ void load_sh(int deg, const float* __restrict__ sh, float* c) {
    const int ncoef = (deg + 1) * (deg + 1);
    if (kAligned) {
        const float4* s4 = reinterpret_cast<const float4*>(sh);
        const int nq = (ncoef * 3 + 3) >> 2;
#pragma unroll
        for (int i = 0; i < 12; ++i) {
            if (i < nq) {
                float4 t = __ldg(s4 + i);
                c[4 * i + 0] = t.x; c[4 * i + 1] = t.y; c[4 * i + 2] = t.z; c[4 * i + 3] = t.w;
            }
        }
    } else {
#pragma unroll
        for (int i = 0; i < 48; ++i)
            if (i < ncoef * 3) c[i] = __ldg(sh + i);
    }
}

// frosting mode: the same row read in place from its two parameter tensors, dc [P,1,3] | rest [P,M-1,3]
// (sh_coordinates = cat(dc, rest), frosting_model.py:733-734); rest rows are 12*(M-1) bytes apart: scalar loads
__device__ __forceinline__ void load_sh_split(int deg, const float* __restrict__ dc, const float* __restrict__ rest,
                                              float* c) {
    const int ncoef = (deg + 1) * (deg + 1);
    c[0] = __ldg(dc); c[1] = __ldg(dc + 1); c[2] = __ldg(dc + 2);
#pragma unroll
    for (int i = 3; i < 48; ++i)
        if (i < ncoef * 3) c[i] = __ldg(rest + i - 3);
}

// computeColorFromSH, forward.cu:20-71.  Returns result before the +0.5 / clamp.
__device__ __forceinline__ void eval_sh(int deg, const float* c, float x, float y, float z,
                                        float& o0, float& o1, float& o2) {
    float r0 = fmul(c[0], kC0), r1 = fmul(c[1], kC0), r2 = fmul(c[2], kC0);
    if (deg > 0) {
        float k;
        k = fmul(y, kC1);
        r0 = ffma(-k, c[3], r0); r1 = ffma(-k, c[4], r1); r2 = ffma(-k, c[5], r2);
        k = fmul(z, kC1);
        r0 = ffma(k, c[6], r0); r1 = ffma(k, c[7], r1); r2 = ffma(k, c[8], r2);
        k = fmul(x, kC1);
        r0 = ffma(-k, c[9], r0); r1 = ffma(-k, c[10], r1); r2 = ffma(-k, c[11], r2);
        if (deg > 1) {
            const float xx = fmul(x, x), yy = fmul(y, y), zz = fmul(z, z);
            const float xy = fmul(y, x), yz = fmul(z, y), xz = fmul(z, x);
            k = fmul(xy, kC2_0);
            r0 = ffma(k, c[12], r0); r1 = ffma(k, c[13], r1); r2 = ffma(k, c[14], r2);
            k = fmul(yz, kC2_1);
            r0 = ffma(k, c[15], r0); r1 = ffma(k, c[16], r1); r2 = ffma(k, c[17], r2);
            const float zz2 = fadd(zz, zz);
            k = fmul(fadd(-yy, fadd(-xx, zz2)), kC2_2);
            r0 = ffma(k, c[18], r0); r1 = ffma(k, c[19], r1); r2 = ffma(k, c[20], r2);
            k = fmul(xz, kC2_3);
            r0 = ffma(k, c[21], r0); r1 = ffma(k, c[22], r1); r2 = ffma(k, c[23], r2);
            const float xx_yy = fadd(xx, -yy);
            k = fmul(xx_yy, kC2_4);
            r0 = ffma(k, c[24], r0); r1 = ffma(k, c[25], r1); r2 = ffma(k, c[26], r2);
            if (deg > 2) {
                k = fmul(fmul(y, kC3_0), ffma(xx, 3.0f, -yy));
                r0 = ffma(k, c[27], r0); r1 = ffma(k, c[28], r1); r2 = ffma(k, c[29], r2);
                k = fmul(fmul(xy, kC3_1), z);
                r0 = ffma(k, c[30], r0); r1 = ffma(k, c[31], r1); r2 = ffma(k, c[32], r2);
                const float f4 = fadd(-yy, ffma(zz, 4.0f, -xx));   // 4zz - xx - yy
                k = fmul(fmul(y, kC3_2), f4);
                r0 = ffma(k, c[33], r0); r1 = ffma(k, c[34], r1); r2 = ffma(k, c[35], r2);
                k = fmul(fmul(z, kC3_3), ffma(yy, -3.0f, ffma(xx, -3.0f, zz2)));
                r0 = ffma(k, c[36], r0); r1 = ffma(k, c[37], r1); r2 = ffma(k, c[38], r2);
                k = fmul(f4, fmul(x, kC3_4));
                r0 = ffma(k, c[39], r0); r1 = ffma(k, c[40], r1); r2 = ffma(k, c[41], r2);
                k = fmul(xx_yy, fmul(z, kC3_5));
                r0 = ffma(k, c[42], r0); r1 = ffma(k, c[43], r1); r2 = ffma(k, c[44], r2);
                k = fmul(fmul(x, kC3_6), ffma(yy, -3.0f, xx));
                r0 = ffma(k, c[45], r0); r1 = ffma(k, c[46], r1); r2 = ffma(k, c[47], r2);
            }
        }
    }
    o0 = r0; o1 = r1; o2 = r2;
}

struct CamConst {
    float view[16];
    float proj[16];
    float campos[3];
};

#ifndef FB200_PRE_CTAS
#define FB200_PRE_CTAS 4
#endif
constexpr int kPreThreads = 256;
constexpr int kPreRounds = 1;        // one round: a longer span only serialises runs of survivors inside a few CTAs
constexpr int kPreSpan = kPreThreads * kPreRounds;     // Gaussians per CTA

// ---- per-tile instance counts for the 32 rectangles of a warp, warp-balanced ----
// The reference's duplicateWithKeys walks each splat's tile rectangle in a serial per-thread double loop
// (rasterizer_impl.cu:98-108) and so did round 1's counting here: one 12x12-tile splat kept its warp busy for 144
// dependent iterations (C5: preprocess 0.77 ms).  Same expansion as scatter_kernel (binning.cu): the warp scans its
// 32 rectangle sizes and walks the concatenated instance list 32 instances per step.
__device__ __forceinline__ void count_tiles(const FwdArgs& a, uint2 rect, int idx, int lane) {
    const unsigned full = 0xffffffffu;
    const uint32_t minx = rect.x & 0xffffu, miny = rect.x >> 16;
    const uint32_t w = (rect.y & 0xffffu) - minx;
    const uint32_t cnt = w * ((rect.y >> 16) - miny);          // 0 unless the Gaussian is rendered
    const unsigned vis = __ballot_sync(full, cnt != 0);
    if (vis == 0) return;
    // FB200_ST_NUM_VISIBLE, and the rendered Gaussians appended to the list the per-Gaussian backward runs over.  The
    // atomic's result is consumed only after the tile walk below, which hides its round trip.
    uint32_t at = 0;
    if (lane == 0) at = atomicAdd(a.counters + 3, (uint32_t)__popc(vis));
    const uint32_t gxw = (uint32_t)a.tiles_x;
    if (__reduce_max_sync(full, cnt) <= 24u) {
        // small rectangles everywhere in the warp (the common frame): the plain per-lane walk is cheaper than the scan
        const uint32_t maxy = rect.y >> 16, maxx = rect.y & 0xffffu;
        if (cnt != 0)
            for (uint32_t ty = miny; ty < maxy; ++ty)
                for (uint32_t tx = minx; tx < maxx; ++tx) atomicAdd(a.tile_count + ty * gxw + tx, 1u);
    } else {
        uint32_t incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(full, incl, o);
            if (lane >= o) incl += t;
        }
        const uint32_t excl = incl - cnt;
        const uint32_t total = __shfl_sync(full, incl, 31);
        const float rw = w ? __frcp_rn((float)w) : 0.f;
        for (uint32_t base = 0; base < total; base += 32) {
            const uint32_t item = base + lane;
            int pos = 0;                      // owner = number of lanes whose inclusive count is <= item
#pragma unroll
            for (int step = 16; step >= 1; step >>= 1) {
                const uint32_t t = __shfl_sync(full, incl, pos + step - 1);
                if (t <= item) pos += step;
            }
            const int owner = min(pos, 31);
            const uint32_t o_excl = __shfl_sync(full, excl, owner);
            const uint32_t o_min = __shfl_sync(full, rect.x, owner);
            const uint32_t o_w = __shfl_sync(full, w, owner);
            const float o_rw = __shfl_sync(full, rw, owner);
            if (item < total) {
                const uint32_t k = item - o_excl;
                // k / o_w through the reciprocal (both < 2^24), corrected by at most one either way
                uint32_t q = __float2uint_rz(__fmul_rn((float)k, o_rw));
                int rem = (int)k - (int)(q * o_w);
                if (rem < 0) { --q; rem += (int)o_w; } else if (rem >= (int)o_w) { ++q; rem -= (int)o_w; }
                const uint32_t ty = (o_min >> 16) + q, tx = (o_min & 0xffffu) + (uint32_t)rem;
                atomicAdd(a.tile_count + ty * gxw + tx, 1u);
            }
        }
    }
    at = __shfl_sync(full, at, 0);
    if (cnt != 0) a.vis_list[at + __popc(vis & ((1u << lane) - 1u))] = (uint32_t)idx;
}

// Everything after the cull for ONE surviving Gaussian: projection, covariance, conic, radius, tile rectangle, colour,
// culling extents, the packed record.  kFrost: attributes come straight from Frosting's parameters (frosting_attr.cuh).
template <bool kFrost>
__device__ __forceinline__ void project_gaussian(const FwdArgs& a, const CamConst& cam, int idx, float px, float py,
                                                 float pz, int& radius, uint2& rect) {
    const float* __restrict__ v = cam.view;
    const float* __restrict__ m = cam.proj;
    const fb200_frosting_params& fr = a.fr;
    const float depth = affine_row(v, 2, px, py, pz);
    const float hx = affine_row(m, 0, px, py, pz);
    const float hy = affine_row(m, 1, px, py, pz);
    const float hw = affine_row(m, 3, px, py, pz);
    const float p_w = __frcp_rn(fadd(hw, 0.0000001f));
    const float projx = fmul(hx, p_w);
    const float projy = fmul(hy, p_w);

    Cov3 S;
    if (kFrost) {
        const float* ls = fr.d_log_scales + 3 * (size_t)idx;
        float nrm;
        const float4 q = frost_normalize(__ldg(reinterpret_cast<const float4*>(fr.d_quats) + idx), nrm);
        S = cov3d_from_scale_rot(expf(__ldg(ls)), expf(__ldg(ls + 1)), expf(__ldg(ls + 2)), a.prm.scale_modifier,
                                 q.x, q.y, q.z, q.w);
    } else if (a.in.d_cov3D_precomp != nullptr) {
        const float* c = a.in.d_cov3D_precomp + 6 * (size_t)idx;
        S.c0 = __ldg(c + 0); S.c1 = __ldg(c + 1); S.c2 = __ldg(c + 2);
        S.c3 = __ldg(c + 3); S.c4 = __ldg(c + 4); S.c5 = __ldg(c + 5);
    } else {
        const float* sc = a.in.d_scales + 3 * (size_t)idx;
        const float4 q = __ldg(reinterpret_cast<const float4*>(a.in.d_rotations) + idx);
        S = cov3d_from_scale_rot(__ldg(sc), __ldg(sc + 1), __ldg(sc + 2), a.prm.scale_modifier, q.x, q.y, q.z, q.w);
    }

    const float3 cov = cov2d(px, py, pz, a.focal_x, a.focal_y, a.prm.tanfovx, a.prm.tanfovy, S, v);
    const float det = ffma(cov.x, cov.z, -fmul(cov.y, cov.y));
    if (det == 0.0f) return;
    const float det_inv = __frcp_rn(det);
    const float conic_x = fmul(cov.z, det_inv);
    const float conic_y = fmul(cov.y, -det_inv);
    const float conic_z = fmul(cov.x, det_inv);
    const float mid = fmul(fadd(cov.x, cov.z), 0.5f);
    const float sq = __fsqrt_rn(fmaxf(ffma(mid, mid, -det), 0.1f));
    const float lambda1 = fadd(mid, sq);
    const float lambda2 = fadd(mid, -sq);
    const float rad_f = fmul(__fsqrt_rn(fmaxf(lambda1, lambda2)), 3.0f);
    const int my_radius = __float2int_ru(rad_f);
    const float Rf = (float)my_radius;
    const float pix_x = ndc2pix(projx, a.prm.image_width);
    const float pix_y = ndc2pix(projy, a.prm.image_height);
    // getRect, auxiliary.h:46-56
    const uint32_t gx = (uint32_t)a.tiles_x, gy = (uint32_t)a.tiles_y;
    const uint32_t minx = rect_coord(fadd(pix_x, -Rf), gx);
    const uint32_t miny = rect_coord(fadd(pix_y, -Rf), gy);
    const uint32_t maxx = rect_coord(fadd(fadd(fadd(pix_x, Rf), 16.0f), -1.0f), gx);
    const uint32_t maxy = rect_coord(fadd(fadd(fadd(pix_y, Rf), 16.0f), -1.0f), gy);
    const uint32_t touched = (maxx - minx) * (maxy - miny);
    if (touched == 0) return;
    radius = my_radius;
    rect = make_uint2(minx | (miny << 16), maxx | (maxy << 16));

    float cr, cg, cb;
    uint8_t clamp_bits = 0;
    if (kFrost || a.in.d_colors_precomp == nullptr) {
        // direction = (p - campos) / |p - campos|   (glm::length = sqrt(dot))
        const float dx = fadd(-cam.campos[0], px);
        const float dy = fadd(-cam.campos[1], py);
        const float dz = fadd(-cam.campos[2], pz);
        const float len = __fsqrt_rn(dot3x(dx, dx, dy, dy, dz, dz));
        const float x = __fdiv_rn(dx, len), y = __fdiv_rn(dy, len), z = __fdiv_rn(dz, len);
        float c[48];
        if (kFrost) {
            load_sh_split(a.prm.sh_degree, fr.d_sh_dc + 3 * (size_t)idx, fr.d_sh_rest + (size_t)idx * fr.sh_rest * 3, c);
        } else {
            const float* sh = a.in.d_shs + (size_t)idx * a.prm.sh_coeffs * 3;
            if ((a.prm.sh_coeffs & 3) == 0) load_sh<true>(a.prm.sh_degree, sh, c);
            else load_sh<false>(a.prm.sh_degree, sh, c);
        }
        float r0, r1, r2;
        eval_sh(a.prm.sh_degree, c, x, y, z, r0, r1, r2);
        // result += 0.5; clamped = result < 0; result = max(result, 0)
        const float s0 = fadd(r0, 0.5f), s1 = fadd(r1, 0.5f), s2 = fadd(r2, 0.5f);
        clamp_bits = (s0 < 0.f ? 1 : 0) | (s1 < 0.f ? 2 : 0) | (s2 < 0.f ? 4 : 0);
        cr = (s0 < 0.f) ? 0.f : s0;
        cg = (s1 < 0.f) ? 0.f : s1;
        cb = (s2 < 0.f) ? 0.f : s2;
    } else {
        const float* c = a.in.d_colors_precomp + 3 * (size_t)idx;
        cr = __ldg(c); cg = __ldg(c + 1); cb = __ldg(c + 2);
    }
    const float opacity = kFrost ? frost_sigmoid(__ldg(fr.d_opacity_logits + idx)) : __ldg(a.in.d_opacities + idx);

    // Conservative extents of {alpha >= 1/255}: |dx| > ext_x  =>  power < -t  for every dy,
    // because max_dy power = -dx^2 / (2 Sigma_xx) and Sigma_xx = cov.x (see DESIGN.md, culling).
    // Margins cover the fp32 rounding of the reference's power/exp/alpha evaluation.
    float ext_x, ext_y, thr;
    {
        const float t = logf(255.0f * opacity);
        const float reach = Rf + 16.0f;
        const float Sq = (fabsf(conic_x) + fabsf(conic_y) + fabsf(conic_z)) * reach * reach;
        const float kappa = fabsf(cov.x * cov.z * det_inv);
        const float tm = (t + 2e-3f + 1e-6f * Sq) * (1.0f + 2e-6f * kappa);
        // level of f = 0.5 (A dx^2 + C dy^2) + B dx dy above which no pixel contributes: tm, plus the rounding
        // of the exact test's own evaluation of f (same magnitude as the reference's, hence the same margin)
        thr = tm + 1e-3f + 1e-6f * Sq;
        if (!(thr == thr) || tm >= 1e30f) thr = __int_as_float(0x7f800000);
        if (tm < 0.0f || opacity <= 0.0f) {
            ext_x = __int_as_float(0xff800000); ext_y = ext_x;   // -inf: can never reach 1/255
        } else if (tm >= 0.0f && tm < 1e30f) {
            ext_x = sqrtf(2.0f * tm * cov.x) * 1.00001f + 1e-3f;
            ext_y = sqrtf(2.0f * tm * cov.z) * 1.00001f + 1e-3f;
            if (!(ext_x >= 0.0f)) ext_x = __int_as_float(0x7f800000);
            if (!(ext_y >= 0.0f)) ext_y = __int_as_float(0x7f800000);
        } else {
            ext_x = __int_as_float(0x7f800000); ext_y = ext_x;   // NaN/inf inputs: never cull
        }
        if (a.prm.debug & 2) { ext_x = __int_as_float(0x7f800000); ext_y = ext_x; thr = ext_x; }
    }

    SplatRec r;
    r.q0 = make_float4(pix_x, pix_y, conic_x, conic_y);
    r.q1 = make_float4(conic_z, opacity, cr, cg);
    r.q2 = make_float4(cb, ext_x, ext_y, thr);
    a.rec[idx] = r;
    a.depth[idx] = depth;
    a.clamped[idx] = clamp_bits;
}

// A CTA owns kPreSpan consecutive Gaussians.  Phase A: every thread culls kPreRounds of them (occlusion lookup +
// near plane: two short load chains) and the survivors -- ~10 % of a Frosting layer under occlusion culling -- are
// compacted into shared memory.  Phase B: the heavy part runs over the compacted list with full warps.  Round 1/2a
// ran the heavy part in place: 11.75 of 32 lanes active per instruction (profiles/r02_c3_v10_summary.json).
template <bool kFrost>
__global__ void __launch_bounds__(kPreThreads, FB200_PRE_CTAS)
preprocess_fwd_kernel(FwdArgs a) {
    __shared__ CamConst cam;
    __shared__ float4 items[kPreSpan];       // {x, y, z, index bits}
    __shared__ int n_items;
    if (threadIdx.x < 16) {
        cam.view[threadIdx.x] = a.in.d_viewmatrix[threadIdx.x];
        cam.proj[threadIdx.x] = a.in.d_projmatrix[threadIdx.x];
    }
    if (threadIdx.x < 3) cam.campos[threadIdx.x] = a.in.d_campos[threadIdx.x];
    if (threadIdx.x == 0) n_items = 0;
    __syncthreads();

    const unsigned full = 0xffffffffu;
    const int P = a.prm.P;
    const int lane = threadIdx.x & 31;
    const int base = blockIdx.x * kPreSpan;
    const float* __restrict__ v = cam.view;

    // ---- phase A: cull ----
    // the occlusion inputs first: the cell -> visible-face gather is a dependent chain of its own, started before the
    // position loads so that the two chains overlap (a culled Gaussian then costs two memory round trips, not three)
    long long cell[kPreRounds];
    uint8_t vis_in[kPreRounds];
#pragma unroll
    for (int r = 0; r < kPreRounds; ++r) {
        const int tid = base + r * kPreThreads + threadIdx.x;
        const int idx = tid < P ? tid : P - 1;
        const bool by_face = a.in.d_face_visible != nullptr && (long long)idx < a.in.n_cell_points;
        cell[r] = by_face ? __ldg(a.in.d_point_cells + idx) : -1;
        vis_in[r] = a.in.d_visibility != nullptr ? __ldg(a.in.d_visibility + idx) : (uint8_t)1;
    }
#pragma unroll
    for (int r = 0; r < kPreRounds; ++r) {
        const int tid = base + r * kPreThreads + threadIdx.x;
        if (base + r * kPreThreads >= P) break;               // CTA-uniform
        const bool valid = tid < P;
        const int idx = valid ? tid : P - 1;
        // occlusion culling: a per-Gaussian mask tensor, or -- without one -- render_mask = face_visible[_point_cell_indices]
        // for the mesh-bound Gaussians, True for the trailing background ones (frosting_model.py:1564-1576), looked up in place
        const uint8_t face_in = cell[r] >= 0 ? __ldg(a.in.d_face_visible + cell[r]) : (uint8_t)1;
        const bool shown = vis_in[r] != 0 && face_in != 0;
        float px = 0.f, py = 0.f, pz = 0.f;
        if (kFrost) {
            if (shown) { float w[6]; int vid[3]; frost_point(a.fr, (size_t)idx, w, vid, px, py, pz); }
        } else {
            px = __ldg(a.in.d_means3D + 3 * (size_t)idx + 0);
            py = __ldg(a.in.d_means3D + 3 * (size_t)idx + 1);
            pz = __ldg(a.in.d_means3D + 3 * (size_t)idx + 2);
        }
        // in_frustum: keep iff !(p_view.z <= 0.2f)
        const float depth = affine_row(v, 2, px, py, pz);
        bool keep = valid && !(depth <= 0.2f);
        if (valid && !keep && a.prm.prefiltered && (!kFrost || shown)) {
            printf("Point is filtered although prefiltered is set. This shouldn't happen!");
            __trap();
        }
        if (!shown) keep = false;
        if (keep) {
            // the SH row (192 B at degree 3) is consumed last, after a chain of dependent loads; start it moving now.
            // Frosting mode at sh_rest == 0 has no rest row (NULL pointer): nothing to prefetch.
            const int row_floats = kFrost ? a.fr.sh_rest * 3 : a.prm.sh_coeffs * 3;
            const char* row = kFrost ? reinterpret_cast<const char*>(a.fr.d_sh_rest + (size_t)idx * row_floats)
                                     : reinterpret_cast<const char*>(a.in.d_shs + (size_t)idx * row_floats);
            if (kFrost ? a.fr.sh_rest > 0 : a.in.d_shs != nullptr) {
                asm volatile("prefetch.global.L1 [%0];" ::"l"(row));
                if (row_floats * 4 > 128) asm volatile("prefetch.global.L1 [%0];" ::"l"(row + 128));
            }
        } else if (valid) {
            a.radii[idx] = 0;
            a.rect[idx] = make_uint2(0u, 0u);
        }
        const unsigned kept = __ballot_sync(full, keep);
        if (kept != 0) {
            int slot = 0;
            if (lane == 0) slot = atomicAdd(&n_items, __popc(kept));
            slot = __shfl_sync(full, slot, 0) + __popc(kept & ((1u << lane) - 1u));
            if (keep) items[slot] = make_float4(px, py, pz, __int_as_float(idx));
        }
    }
    __syncthreads();

    // ---- phase B: project the survivors, full warps ----
    const int n = n_items;
    static_assert(kPreRounds == 1, "phase B below handles one round (n <= kPreThreads)");
    const int jb = threadIdx.x & ~31;
    if (jb < n) {                                                       // warp-uniform
        const int j = jb + lane;
        int radius = 0, idx = 0;
        uint2 rect = make_uint2(0u, 0u);
        if (j < n) {
            const float4 it = items[j];
            idx = __float_as_int(it.w);
            project_gaussian<kFrost>(a, cam, idx, it.x, it.y, it.z, radius, rect);
            a.radii[idx] = radius;
            a.rect[idx] = rect;
        }
        count_tiles(a, rect, idx, lane);
    }
}

__global__ void __launch_bounds__(256)
mark_visible_kernel(int P, const float* __restrict__ means, const float* __restrict__ view,
                    uint8_t* __restrict__ present) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= P) return;
    const float px = means[3 * (size_t)idx], py = means[3 * (size_t)idx + 1], pz = means[3 * (size_t)idx + 2];
    const float depth = affine_row(view, 2, px, py, pz);
    present[idx] = (depth <= 0.2f) ? 0 : 1;
}

}  // namespace

cudaError_t launch_preprocess_fwd(const FwdArgs& a, cudaStream_t s) {
    const int T = a.tiles_x * a.tiles_y;
    // the per-tile counts and the counter words behind them (adjacent in the image workspace) in one memset
    const size_t span = (size_t)(reinterpret_cast<const char*>(a.counters) - reinterpret_cast<const char*>(a.tile_count)) + 64;
    (void)T;
    cudaError_t e = cudaMemsetAsync(a.tile_count, 0, span, s);
    if (e != cudaSuccess) return e;
    if (a.prm.P > 0) {
        const int blocks = (a.prm.P + kPreSpan - 1) / kPreSpan;
        if (a.frosting) preprocess_fwd_kernel<true><<<blocks, kPreThreads, 0, s>>>(a);
        else preprocess_fwd_kernel<false><<<blocks, kPreThreads, 0, s>>>(a);
        count_launch();
    }
    return cudaGetLastError();
}

cudaError_t launch_mark_visible(int P, const float* means, const float* view, uint8_t* present, cudaStream_t s) {
    if (P > 0) { mark_visible_kernel<<<(P + 255) / 256, 256, 0, s>>>(P, means, view, present); count_launch(); }
    return cudaGetLastError();
}

}  // namespace fb200
