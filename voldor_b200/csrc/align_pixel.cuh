// Per-pixel frame-alignment arithmetic shared by every kernel that evaluates it: the reference-ABI kernel
// k_align_eval (align_frame.cu) and the all-pairs solver evaluation k_fa_eval (falign.cu).  Both call
// align_sample(), so a sample of the solver is bit for bit the sample vb_align_frame_eval_strided returns.
//
// Behavioural source: reference gpu-kernels/align_frame.cu:47-134 (rotation by a rotation vector with its
// Jacobians), :137-151 (pinhole helpers), :153-203 (normals, Scharr-like depth/image gradients), :205-381
// (point-to-plane + photometric residual and analytic Jacobian w.r.t. [rvec, tvec, log depth scale, colour
// scale, colour offset]), :383-411 (weighted sqrt-Cauchy loss).  Quirks kept on purpose:
//   * at_safe(x-1) at x == 0 wraps to the LAST column/row, not the first (size_t underflow then min(), SURVEY
//     §9 Q17; gmat.h:181-186) — border normals and gradients use the opposite border;
//   * d(R(r)p)/dr divides some terms by sqrt(theta^2 * theta) = theta^1.5 where the closed form has theta^3
//     (align_frame.cu:71-83).  It is reproduced as is: the contract is the reference's numbers.
// Everything here has internal linkage: each translation unit that includes it gets its own copy.
#pragma once
#include <cfloat>
#include <cmath>
#include "common.cuh"
#include "falign.cuh"

namespace vb {
namespace {

constexpr int kAlignParams = 9;  // reference: align_frame.cu:9

struct F3 {
    float x, y, z;
};
__device__ __forceinline__ F3 f3(float x, float y, float z) { return F3{x, y, z}; }
__device__ __forceinline__ F3 vadd(F3 a, F3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ F3 vsub(F3 a, F3 b) { return f3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ F3 vmul(F3 a, float s) { return f3(a.x * s, a.y * s, a.z * s); }
__device__ __forceinline__ F3 vneg(F3 a) { return f3(-a.x, -a.y, -a.z); }
__device__ __forceinline__ float vdot(F3 a, F3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ F3 vcross(F3 a, F3 b) {
    return f3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
__device__ __forceinline__ float vnorm2(F3 v) { return v.x * v.x + v.y * v.y + v.z * v.z; }

// clamp with the reference's unsigned-wrap behaviour: -1 -> last
__device__ __forceinline__ int safe_idx(int i, int n) { return i < 0 ? n - 1 : (i > n - 1 ? n - 1 : i); }

__device__ __forceinline__ F3 backproject(const AlignIntr& K, float px, float py, float depth) {
    return f3((K.fxi * px + K.cxi) * depth, (K.fyi * py + K.cyi) * depth, depth);
}

// R(rvec) * p with optional Jacobians (align_frame.cu:47-134)
__device__ F3 rotate(F3 p, F3 r, float (*J_r)[3], float (*J_p)[3]) {
    const float theta2 = vnorm2(r);
    const float rv[3] = {r.x, r.y, r.z}, pv[3] = {p.x, p.y, p.z};
    if (theta2 > FLT_EPSILON) {
        const float theta = sqrtf(theta2);
        const float ct = cosf(theta), st = sinf(theta);
        const float theta_inv = 1.f / theta;
        const F3 w = vmul(r, theta_inv);
        const F3 wxp = vcross(w, p);
        const float tmp = vdot(w, p) * (1.0f - ct);
        const float c1 = ct - 1;
        if (J_p) {
            // cos*I + sin*[w]x + (1-cos) w w^T
            const float sgn[3][3] = {{0, -1, 1}, {1, 0, -1}, {-1, 1, 0}};
            for (int i = 0; i < 3; i++)
                for (int j = 0; j < 3; j++) {
                    if (i == j)
                        J_p[i][j] = ct - ((rv[i] * rv[i]) * c1) / theta2;
                    else {
                        const int k = 3 - i - j;
                        J_p[i][j] = sgn[i][j] * (rv[k] * st) / theta - (rv[i] * rv[j] * c1) / theta2;
                    }
                }
        }
        if (J_r) {
            const float t32 = sqrtf(theta2 * theta);  // sic (see header)
            const float D = (r.x * p.x) / theta + (r.y * p.y) / theta + (r.z * p.z) / theta;
            const F3 cr = vcross(r, p);
            const float crv[3] = {cr.x, cr.y, cr.z};
            // d(r x p)_i / d r_j
            const float e[3][3] = {{0, p.z, -p.y}, {-p.z, 0, p.x}, {p.y, -p.x, 0}};
            for (int i = 0; i < 3; i++)
                for (int j = 0; j < 3; j++) {
                    const float rp32 = (rv[j] * rv[0] * pv[0]) / t32 + (rv[j] * rv[1] * pv[1]) / t32 +
                                       (rv[j] * rv[2] * pv[2]) / t32;
                    float v = st * (e[i][j] / theta - (rv[j] * crv[i]) / t32);
                    if (i == j) v -= (c1 * D) / theta;
                    v += (rv[i] * c1 * (rp32 - pv[j] / theta)) / theta;
                    v -= (rv[j] * pv[i] * st) / theta;
                    v += (rv[i] * rv[j] * c1 * D) / t32;
                    v += (rv[i] * rv[j] * st * D) / theta2;
                    v += (rv[j] * ct * (crv[i] / theta)) / theta;
                    J_r[i][j] = v;
                }
        }
        return vadd(vadd(vmul(p, ct), vmul(wxp, st)), vmul(w, tmp));
    }
    const F3 wxp = vcross(r, p);
    if (J_p) {
        J_p[0][0] = 1, J_p[0][1] = -r.z, J_p[0][2] = r.y;
        J_p[1][0] = r.z, J_p[1][1] = 1, J_p[1][2] = -r.x;
        J_p[2][0] = -r.y, J_p[2][1] = r.x, J_p[2][2] = 1;
    }
    if (J_r) {
        J_r[0][0] = 0, J_r[0][1] = p.z, J_r[0][2] = -p.y;
        J_r[1][0] = -p.z, J_r[1][1] = 0, J_r[1][2] = p.x;
        J_r[2][0] = p.y, J_r[2][1] = -p.x, J_r[2][2] = 0;
    }
    return vadd(p, wxp);
}

struct AlignView {
    int w, h;
    AlignIntr K;
    float vbf, crw;
    cudaTextureObject_t images, depths, dimages, normals;
    const float* images_raw;
    size_t images_pitch;
    const float* depths_raw;
    size_t depths_pitch;
    const float* weights;
    int wpitch;
    size_t wplane;
    float* residual;
    float* jacobian;
};

template <typename T>
__device__ __forceinline__ T stack_fetch(cudaTextureObject_t t, float x, float y, int d, int h) {
    return tex2D<T>(t, x + 0.5f, d * (size_t)h + y + 0.5f);
}
__device__ __forceinline__ float raw_at(const float* base, size_t pitch, int h, int x, int y, int d) {
    return *((const float*)((const char*)base + ((size_t)d * h + y) * pitch) + x);
}

// normals (towards the viewer) and Scharr-like gradients for every frame (align_frame.cu:153-203)
__global__ void k_align_prepare(AlignView A, float4* normals, size_t npitch, float2* ddepths, size_t ddpitch,
                                float2* dimages, size_t dipitch, int photo) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    const int f = blockIdx.z;
    if (x >= A.w || y >= A.h) return;
    auto D = [&](int xx, int yy) {
        return raw_at(A.depths_raw, A.depths_pitch, A.h, safe_idx(xx, A.w), safe_idx(yy, A.h), f);
    };
    const F3 p3t = backproject(A.K, (float)x, (float)(y - 1), D(x, y - 1));
    const F3 p3b = backproject(A.K, (float)x, (float)(y + 1), D(x, y + 1));
    const F3 p3l = backproject(A.K, (float)(x - 1), (float)y, D(x - 1, y));
    const F3 p3r = backproject(A.K, (float)(x + 1), (float)y, D(x + 1, y));
    F3 n = vcross(vsub(p3t, p3b), vsub(p3l, p3r));
    const float nn = sqrtf(vnorm2(n));
    n = f3(n.x / nn, n.y / nn, n.z / nn);
    const F3 ray = backproject(A.K, (float)x, (float)y, 1.f);
    if (vdot(ray, n) > 0) n = vneg(n);
    ((float4*)((char*)normals + ((size_t)f * A.h + y) * npitch))[x] = make_float4(n.x, n.y, n.z, 0);
    ((float2*)((char*)ddepths + ((size_t)f * A.h + y) * ddpitch))[x] = make_float2(
        0.3f * (D(x + 1, y) - D(x - 1, y)) + 0.1f * (D(x + 1, y - 1) - D(x - 1, y - 1)) +
            0.1f * (D(x + 1, y + 1) - D(x - 1, y + 1)),
        0.3f * (D(x, y + 1) - D(x, y - 1)) + 0.1f * (D(x - 1, y + 1) - D(x - 1, y - 1)) +
            0.1f * (D(x + 1, y + 1) - D(x + 1, y - 1)));
    if (photo) {
        auto I = [&](int xx, int yy) {
            return raw_at(A.images_raw, A.images_pitch, A.h, safe_idx(xx, A.w), safe_idx(yy, A.h), f);
        };
        ((float2*)((char*)dimages + ((size_t)f * A.h + y) * dipitch))[x] = make_float2(
            0.3f * (I(x + 1, y) - I(x - 1, y)) + 0.1f * (I(x + 1, y - 1) - I(x - 1, y - 1)) +
                0.1f * (I(x + 1, y + 1) - I(x - 1, y + 1)),
            0.3f * (I(x, y + 1) - I(x, y - 1)) + 0.1f * (I(x - 1, y + 1) - I(x - 1, y - 1)) +
                0.1f * (I(x + 1, y + 1) - I(x + 1, y - 1)));
    }
}

// One sample: residual (NaN where the reference marks the pixel invalid) after the weighted sqrt-Cauchy loss, and
// its Jacobian w.r.t. the 9 reference-frame parameters in J (zeros where not computed).  pref / ptar: the 9 float
// parameters of the reference and target frames.  photo / with_jacobian / apply_weights are run-time flags in every
// caller.  Not inlined: the compiler then forms its fused multiply-adds from this body alone, so every kernel that
// calls it (in any translation unit built with the same flags) gets the same instructions and the same bits.
// Inlined, the contractions followed the surrounding kernel and the solver's samples differed in the last bit from
// k_align_eval's once the colour parameters were non-zero.
__device__ __noinline__ float align_sample(const AlignView& A, const float* pref, const float* ptar, int f_ref,
                                              int f_tar, int x, int y, int photo, int with_jacobian,
                                              int apply_weights, float J[kAlignParams]) {
    for (int i = 0; i < kAlignParams; i++) J[i] = 0.f;
    float residual = 0.f;
    const float nanv = __int_as_float(0x7fffffff);
    bool ok = true;

    const F3 rvec = f3(pref[0], pref[1], pref[2]), tvec = f3(pref[3], pref[4], pref[5]);
    const float d_scale_ref = pref[6], c_scale_ref = pref[7], c_offset_ref = pref[8];
    const float p2r_d_bs = raw_at(A.depths_raw, A.depths_pitch, A.h, x, y, f_ref);
    const float p2r_d = p2r_d_bs * expf(d_scale_ref);
    const F3 dp3r_dd = f3(A.K.fxi * x + A.K.cxi, A.K.fyi * y + A.K.cyi, 1.f);
    const F3 p3r = backproject(A.K, (float)x, (float)y, p2r_d);

    float Jw_r[3][3], Jw_p[3][3], Jt_w[3][3];
    const F3 p3w = vadd(rotate(p3r, rvec, with_jacobian ? Jw_r : nullptr, with_jacobian ? Jw_p : nullptr), tvec);
    F3 rvec0 = vneg(f3(ptar[0], ptar[1], ptar[2]));
    const F3 tvec0 = vneg(rotate(f3(ptar[3], ptar[4], ptar[5]), rvec0, nullptr, nullptr));
    const float d_scale_tar = ptar[6], c_scale_tar = ptar[7], c_offset_tar = ptar[8];
    const F3 p3t = vadd(rotate(p3w, rvec0, nullptr, with_jacobian ? Jt_w : nullptr), tvec0);

    float Jp2[2][3];
    Jp2[0][0] = A.K.fx / p3t.z, Jp2[0][1] = 0, Jp2[0][2] = -(A.K.fx * p3t.x) / (p3t.z * p3t.z);
    Jp2[1][0] = 0, Jp2[1][1] = A.K.fy / p3t.z, Jp2[1][2] = -(A.K.fy * p3t.y) / (p3t.z * p3t.z);
    const float p2tx = (A.K.fx * p3t.x) / p3t.z + A.K.cx, p2ty = (A.K.fy * p3t.y) / p3t.z + A.K.cy;
    if (p2tx < 0 || p2tx >= A.w || p2ty < 0 || p2ty >= A.h || p3t.z < 1.f) ok = false;

    if (ok) {
        const float p2t_d = stack_fetch<float>(A.depths, p2tx, p2ty, f_tar, A.h) * expf(d_scale_tar);
        const float4 n4 = stack_fetch<float4>(A.normals, p2tx, p2ty, f_tar, A.h);
        const F3 nvec = f3(n4.x, n4.y, n4.z);
        const F3 ray = vmul(p3t, p2t_d / p3t.z);
        const F3 diff_geo = vmul(nvec, vdot(nvec, vsub(ray, p3t)));
        const F3 tar_geo = vadd(p3t, diff_geo);
        const float gx = (A.K.fx * tar_geo.x) / tar_geo.z + A.K.cx, gy = (A.K.fy * tar_geo.y) / tar_geo.z + A.K.cy;
        if (gx < 0 || gx >= A.w || gy < 0 || gy >= A.h) ok = false;
        if (ok) {
            const float residual_depth = 0.5f * vnorm2(diff_geo);
            const float q = A.vbf / (fmaxf(tar_geo.z, 1.0f) * fmaxf(p3t.z, 1.0f));
            const float drw = q * q;
            float c_ref = 0, c_tar = 0, residual_color = 0;
            if (photo) {
                c_ref = raw_at(A.images_raw, A.images_pitch, A.h, x, y, f_ref) + c_offset_ref;
                const float c_tar_bs = stack_fetch<float>(A.images, p2tx, p2ty, f_tar, A.h) + c_offset_tar;
                c_tar = c_tar_bs * (expf(c_scale_ref) / expf(c_scale_tar));
                residual_color = 0.5f * (c_ref - c_tar) * (c_ref - c_tar);
                residual = drw * residual_depth + A.crw * residual_color;
            } else {
                residual = drw * residual_depth;
            }
            if (with_jacobian) {
                const F3 rd_p3t = vneg(diff_geo);
                F3 rc_p3t = f3(0, 0, 0);
                float rc_cscale = 0, rc_coffset = 0;
                if (photo) {
                    const float rc_ctar = c_tar - c_ref, rc_cref = c_ref - c_tar;
                    const float2 g = stack_fetch<float2>(A.dimages, p2tx, p2ty, f_tar, A.h);
                    const float a0 = g.x * rc_ctar, a1 = g.y * rc_ctar;
                    rc_p3t = f3(a0 * Jp2[0][0] + a1 * Jp2[1][0], a0 * Jp2[0][1] + a1 * Jp2[1][1],
                                a0 * Jp2[0][2] + a1 * Jp2[1][2]);
                    rc_cscale = rc_ctar * c_tar;
                    rc_coffset = rc_cref * 1.f;
                }
                const F3 r_p3t = vadd(vmul(rd_p3t, drw), vmul(rc_p3t, A.crw));
                const float a[3] = {r_p3t.x, r_p3t.y, r_p3t.z};
                float r_p3w[3], r_rvec[3], r_p3r[3];
                for (int j = 0; j < 3; j++) r_p3w[j] = a[0] * Jt_w[0][j] + a[1] * Jt_w[1][j] + a[2] * Jt_w[2][j];
                for (int j = 0; j < 3; j++)
                    r_rvec[j] = r_p3w[0] * Jw_r[0][j] + r_p3w[1] * Jw_r[1][j] + r_p3w[2] * Jw_r[2][j];
                for (int j = 0; j < 3; j++)
                    r_p3r[j] = r_p3w[0] * Jw_p[0][j] + r_p3w[1] * Jw_p[1][j] + r_p3w[2] * Jw_p[2][j];
                J[0] = r_rvec[0], J[1] = r_rvec[1], J[2] = r_rvec[2];
                J[3] = r_p3w[0], J[4] = r_p3w[1], J[5] = r_p3w[2];
                J[6] = vdot(f3(r_p3r[0], r_p3r[1], r_p3r[2]), dp3r_dd) * p2r_d;
                if (photo) J[7] = A.crw * rc_cscale, J[8] = A.crw * rc_coffset;
            }
        }
    }
    if (!ok) residual = nanv;

    // weighted sqrt-Cauchy loss (align_frame.cu:383-411): NaN residuals fail the '>' test and stay NaN
    float weight = 1.f;
    if (apply_weights) weight = A.weights[(size_t)f_ref * A.wplane + (size_t)y * A.wpitch + x];
    const float residual2 = weight * residual;
    if (residual2 > FLT_EPSILON) {
        const float loss = logf(residual2 + 1.f);
        const float dloss = 1.f / (residual2 + 1.f);
        const float sqrt_loss = sqrtf(loss);
        const float dsqrt = 0.5f / sqrt_loss;
        residual = sqrt_loss;
        if (with_jacobian)
            for (int i = 0; i < kAlignParams; i++) J[i] *= (dsqrt * dloss * weight);
    }
    return residual;
}

}  // namespace
}  // namespace vb
