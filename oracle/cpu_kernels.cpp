// TEST INFRASTRUCTURE (oracle). Not part of the shipped product.
//
// CPU port of the EM hot path behind the same library-level ABI (symbols prefixed cpu_), plain C++ with
// OpenMP over pixels / hypotheses.  It restates the reference's CUDA kernels line by line in scalar FP32:
//   residual model            gpu-kernels/residual_model.h:6-68
//   stacked bilinear fetch    gpu-kernels/gmat.h:39-66,175-179 (CUDA linear filtering emulated: 8-bit weights,
//                             layers stacked in y, clamp at the stack border)
//   depth step                gpu-kernels/optimize_depth.cu:84-291 (kernels), :462-494 (schedule)
//   forward-backward smoother gpu-kernels/fb_smooth.h:29-107
//   per-pixel XORWOW          cuRAND's own curand_init/curand_uniform compiled for the host
//                             (curand_kernel.h:60-62 QUALIFIERS override) -> identical streams
//   P3P instance collector    gpu-kernels/collect_p3p_instances.cu:57-145
//   batched P3P               gpu-kernels/solve_batch_lambdatwist.cu:11-42 with the reference's own
//                             lambdatwist/*.h compiled for the host when /root/reference is available at build
//                             time (HAVE_REF_LAMBDATWIST), R->rvec by ../voldor_b200/csrc/host_math.h (the
//                             reference's CPU branch uses cv::Rodrigues there, voldor/geometry.cpp:118)
//   mean-shift                gpu-kernels/meanshift.cu:12-150 + reduce_vector_sum.h:12-57 (same tree order)
//   robust Gaussian fit       gpu-kernels/fit_robust_gaussian.cu:56-286 + aux_funs.cpp:101-141
// Purpose: (1) GPU-less logic tests, (2) the `cpu_baseline` / `--impl reference` leg of bench.py (the reference
// has no CPU implementation of the E/M steps: voldor.cpp:254,274 call CUDA; SURVEY §0), (3) tolerance-level
// cross-check of the GPU results.  Bit-level truth for parity is oracle/_ref (the reference kernels
// themselves on the GPU); libm's powf/expf/logf differ from libdevice in the last bits, so this port is
// compared with tolerances and "fraction of pixels within tolerance".
// PARITY PINNING: the reference ships no tests or golden vectors (SURVEY §4); this port is pinned against
// outputs of the reference kernels generated on the GPU box (tests/golden/*.npz, tests/make_golden.py).
#define QUALIFIERS static inline
#include <cuda_runtime.h>
#include <curand_kernel.h>

#include "../voldor_b200/csrc/host_math.h"
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#ifdef HAVE_REF_LAMBDATWIST
#include "lambdatwist/lambdatwist_p4p.h"
#else
// without the reference checkout: the product's lambda-twist lanes, built for the host (individually rounded operations,
// the same hypotheses bit for bit as the reference kernels: tests/test_cpu_p3p_quad.py)
#include "../voldor_b200/csrc/p3p_twist_quad.cuh"
#endif

namespace {

// ---------------------------------------------------------------------------------------------------
// residual model (residual_model.h)
// ---------------------------------------------------------------------------------------------------
inline float fmag_c(float fmag) {
    fmag = std::fmin(std::fmax(fmag * 0.5f, 2.f), 100.f);
    return 1.0f + -0.0022f * fmag;
}
inline float fmag_scale(float fmag) {
    fmag = std::fmin(std::fmax(fmag * 0.5f, 2.f), 100.f);
    return 0.01f * std::exp(0.09f * fmag);
}
inline float fisk_pdf(float x, float c, float scale) {
    x = std::fmax(x * 0.5f, FLT_EPSILON);
    const float q = (x * x) / scale;
    return (c * std::pow(q, -c - 1.f) * std::pow(1 + std::pow(q, -c), -2.f)) / scale;
}
inline float l2n(float x, float y) { return std::sqrt(x * x + y * y); }
inline float fun_rigidness(float dx1, float dy1, float dx2, float dy2, float lambda, float abs_rf) {
    const float obs = l2n(dx2, dy2) / abs_rf;
    const float diff = l2n(dx1 - dx2, dy1 - dy2) / abs_rf;
    const float c = fmag_c(obs), s = fmag_scale(obs);
    const float p = fisk_pdf(diff, c, s), mu = fisk_pdf(lambda * obs, c, s);
    return p / (p + mu);
}
inline float fun_depth_rigidness(float d1, float d2, float basefocal, float omega, float abs_rf) {
    const float disp1 = (basefocal / d1) / abs_rf, disp2 = (basefocal / d2) / abs_rf;
    const float diff = std::fabs(disp1 - disp2);
    const float c = fmag_c(disp2), s = fmag_scale(disp2);
    const float p = fisk_pdf(diff, c, s), mu = fisk_pdf(omega * disp2, c, s);
    return p / (p + mu);
}

// ---------------------------------------------------------------------------------------------------
// stacked layered image with emulated CUDA bilinear filtering (gmat.h)
// ---------------------------------------------------------------------------------------------------
template <int CH>
struct Stack {
    std::vector<float> data;
    int w = 0, h = 0, layers = 0;
    bool ensure(int w_, int h_, int l_) {  // lazy layers: keep a larger allocation (gmat.h:19-22)
        if (w_ == w && h_ == h && l_ <= layers) return false;
        w = w_, h = h_, layers = l_;
        data.assign((size_t)w * h * layers * CH, 0.f);
        return true;
    }
    float* layer(int d) { return data.data() + (size_t)d * w * h * CH; }
    inline void tex(float x, float y, int d, float* out) const {
        // tex2D(x + 0.5, d*h + y + 0.5), linear filter, clamp, unnormalised
        const float xb = (x + 0.5f) - 0.5f, yb = ((float)((size_t)d * h) + y + 0.5f) - 0.5f;
        const float fx = std::floor(xb), fy = std::floor(yb);
        const float a = std::floor((xb - fx) * 256.f + 0.5f) * (1.f / 256.f);
        const float b = std::floor((yb - fy) * 256.f + 0.5f) * (1.f / 256.f);
        const int H = h * layers;
        const int x0 = std::min(std::max((int)fx, 0), w - 1), x1 = std::min(std::max((int)fx + 1, 0), w - 1);
        const int y0 = std::min(std::max((int)fy, 0), H - 1), y1 = std::min(std::max((int)fy + 1, 0), H - 1);
        for (int c = 0; c < CH; c++) {
            const float t00 = data[((size_t)y0 * w + x0) * CH + c], t10 = data[((size_t)y0 * w + x1) * CH + c];
            const float t01 = data[((size_t)y1 * w + x0) * CH + c], t11 = data[((size_t)y1 * w + x1) * CH + c];
            out[c] = (1 - a) * (1 - b) * t00 + a * (1 - b) * t10 + (1 - a) * b * t01 + a * b * t11;
        }
    }
};

struct Cam {
    float K4[4], K4inv[4];
    float R[16][9], t[16][3];
};
inline void set_K(Cam& c, const float* K) {
    c.K4[0] = K[0], c.K4[1] = K[2], c.K4[2] = K[4], c.K4[3] = K[5];
    c.K4inv[0] = 1.f / K[0], c.K4inv[1] = -K[2] / K[0], c.K4inv[2] = 1.f / K[4], c.K4inv[3] = -K[5] / K[4];
}
inline void p2_to_p3(const Cam& C, float px, float py, float depth, float& ox, float& oy, float& oz) {
    ox = (C.K4inv[0] * px + C.K4inv[1]) * depth, oy = (C.K4inv[2] * py + C.K4inv[3]) * depth, oz = depth;
}
inline void p3_to_p2(const Cam& C, float ox, float oy, float oz, float& px, float& py) {
    px = (C.K4[0] * ox + C.K4[1] * oz) / oz, py = (C.K4[2] * oy + C.K4[3] * oz) / oz;
}
inline void trans(const float* R, const float* t, float& ox, float& oy, float& oz) {
    const float a = ox * R[0] + oy * R[1] + oz * R[2], b = ox * R[3] + oy * R[4] + oz * R[5],
                c = ox * R[6] + oy * R[7] + oz * R[8];
    ox = a + t[0], oy = b + t[1], oz = c + t[2];
}

// ---------------------------------------------------------------------------------------------------
// depth step state (optimize_depth.cu:45-52)
// ---------------------------------------------------------------------------------------------------
struct DepthState {
    int w = 0, h = 0;
    std::vector<curandStateXORWOW_t> rng;
    Stack<2> flows;
    Stack<1> rig, dp, dp_pconf, dp_conf;
    std::vector<float> depth, cost;
    Cam cam, pcam;
    int N = 0, N_dp = 0;
    float abs_rf, basefocal, lambda, omega, delta, disp_delta, range_factor;

    float pixel_cost(int px, int py, float d) const {  // optimize_depth.cu:140-198
        float cost_sum = 0, wsum = 0, ox, oy, oz, px1 = (float)px, py1 = (float)py, px2, py2;
        p2_to_p3(cam, (float)px, (float)py, d, ox, oy, oz);
        for (int f = 0; f < N; f++) {
            trans(cam.R[f], cam.t[f], ox, oy, oz);
            p3_to_p2(cam, ox, oy, oz, px2, py2);
            if (oz > 0 && px1 >= 0 && px1 < w && py1 >= 0 && py1 < h) {
                float d2[2];
                flows.tex(px1, py1, f, d2);
                const float dx1 = px2 - px1, dy1 = py2 - py1;
                px1 = px2, py1 = py2;
                const float wgt = rig.data[((size_t)f * h + py) * w + px];
                cost_sum -= wgt * std::log(fun_rigidness(dx1, dy1, d2[0], d2[1], lambda, abs_rf));
                wsum += wgt;
            }
        }
        for (int f = 0; f < N_dp; f++) {
            p2_to_p3(cam, (float)px, (float)py, d, ox, oy, oz);
            trans(pcam.R[f], pcam.t[f], ox, oy, oz);
            p3_to_p2(cam, ox, oy, oz, px1, py1);
            if (oz > 0 && px1 >= 0 && px1 < w && py1 >= 0 && py1 < h) {
                float td, tp, tc;
                dp.tex(px1, py1, f, &td), dp_pconf.tex(px1, py1, f, &tp), dp_conf.tex(px1, py1, f, &tc);
                if (td > 0) {
                    const float wgt = tp * tc * ((disp_delta > 0 && f == 0) ? disp_delta : delta);
                    cost_sum -= wgt * std::log(fun_depth_rigidness(oz, td, basefocal, omega, abs_rf));
                    wsum += wgt;
                }
            }
        }
        if (wsum == 0) return INFINITY;
        return cost_sum / std::fmax(wsum, FLT_EPSILON);
    }
    inline void try_depth(int x, int y, float cand) {
        const float c = pixel_cost(x, y, cand);
        float& cc = cost[(size_t)y * w + x];
        if (c < cc) depth[(size_t)y * w + x] = cand, cc = c;
    }
    void update_rigidness() {  // optimize_depth.cu:84-138
#pragma omp parallel for schedule(dynamic, 4)
        for (int y = 0; y < h; y++)
            for (int x = 0; x < w; x++) {
                const float d = depth[(size_t)y * w + x];
                float ox, oy, oz, px1 = (float)x, py1 = (float)y, px2, py2;
                p2_to_p3(cam, (float)x, (float)y, d, ox, oy, oz);
                for (int f = 0; f < N; f++) {
                    trans(cam.R[f], cam.t[f], ox, oy, oz);
                    p3_to_p2(cam, ox, oy, oz, px2, py2);
                    float r = 0;
                    if (oz > 0 && px1 >= 0 && px1 < w && py1 >= 0 && py1 < h) {
                        float d2[2];
                        flows.tex(px1, py1, f, d2);
                        const float dx1 = px2 - px1, dy1 = py2 - py1;
                        px1 = px2, py1 = py2;
                        r = fun_rigidness(dx1, dy1, d2[0], d2[1], lambda, abs_rf);
                    }
                    rig.data[((size_t)f * h + y) * w + x] = r;
                }
                for (int f = 0; f < N_dp; f++) {
                    p2_to_p3(cam, (float)x, (float)y, d, ox, oy, oz);
                    trans(pcam.R[f], pcam.t[f], ox, oy, oz);
                    p3_to_p2(cam, ox, oy, oz, px1, py1);
                    float& conf = dp_conf.data[((size_t)f * h + y) * w + x];
                    if (oz > 0 && px1 >= 0 && px1 < w && py1 >= 0 && py1 < h) {
                        float td;
                        dp.tex(px1, py1, f, &td);
                        if (td > 0) conf = fun_depth_rigidness(oz, td, basefocal, omega, abs_rf);
                    } else
                        conf = 0;
                }
            }
    }
};

// fb_smooth.h:29-107 on a stack of `layers` maps
void fb_smooth(float* maps, int layers, int w, int h, float s0e, float nc) {
    const size_t plane = (size_t)w * h;
    std::vector<float> F(plane * layers), B(plane * layers);
    auto fwd = [&](float p, float e) {
        const float s0 = (p * (1.f - nc) + (1.f - p) * nc) * s0e, s1 = (p * nc + (1.f - p) * (1 - nc)) * e;
        return s1 / (s0 + s1);
    };
    auto bwd = [&](float p, float e) {
        const float s0 = p * e * (1.f - nc) + (1.f - p) * nc * s0e, s1 = p * e * nc + (1.f - p) * (1.f - nc) * s0e;
        return s1 / (s0 + s1);
    };
    auto post = [&]() {
#pragma omp parallel for
        for (long long i = 0; i < (long long)(plane * layers); i++) {
            const float s0 = (1.f - F[i]) * (1.f - B[i]), s1 = F[i] * B[i];
            maps[i] = s1 / (s0 + s1);
        }
    };
#pragma omp parallel for collapse(2)
    for (int d = 0; d < layers; d++)
        for (int y = 0; y < h; y++) {
            float* e = maps + d * plane + (size_t)y * w;
            float p = e[0];
            for (int i = 0; i < w; i++) F[d * plane + (size_t)y * w + i] = p = fwd(p, e[i]);
            p = e[w - 1];
            for (int i = w - 1; i >= 0; i--) B[d * plane + (size_t)y * w + i] = p = bwd(p, e[i]);
        }
    post();
#pragma omp parallel for collapse(2)
    for (int d = 0; d < layers; d++)
        for (int x = 0; x < w; x++) {
            float* e = maps + d * plane + x;
            float p = e[0];
            for (int i = 0; i < h; i++) F[d * plane + (size_t)i * w + x] = p = fwd(p, e[(size_t)i * w]);
            p = e[(size_t)(h - 1) * w];
            for (int i = h - 1; i >= 0; i--) B[d * plane + (size_t)i * w + x] = p = bwd(p, e[(size_t)i * w]);
        }
    post();
}

DepthState g_depth;

// ---------------------------------------------------------------------------------------------------
// reduce_vector_sum.h tree: 512-element blocks, pairs (i, i+256), strides 128..1, recursive over block results
// ---------------------------------------------------------------------------------------------------
float tree_sum(std::vector<float> v) {
    while (v.size() > 1) {
        const size_t n = v.size(), nb = (n + 511) / 512;
        std::vector<float> out(nb);
        for (size_t b = 0; b < nb; b++) {
            float s[256];
            for (int t = 0; t < 256; t++) {
                const size_t idx = b * 512 + t;
                s[t] = 0;
                if (idx < n) {
                    s[t] = v[idx];
                    if (idx + 256 < n) s[t] += v[idx + 256];
                }
            }
            for (int stride = 128; stride >= 1; stride >>= 1)
                for (int t = 0; t < stride; t++) s[t] += s[t + stride];
            out[b] = s[0];
        }
        v.swap(out);
    }
    return v.empty() ? 0.f : v[0];
}

}  // namespace

double inverse(double* mat, double* mat_inv, int N);  // oracle/ref_shim/aux_shim.cpp (linked in, C++ linkage)
double regularize_covar_LW_given_lambda(double* mat, double* mat_ret, double lambda, int dims);

extern "C" {

// optimize_depth.cu:293-520
int cpu_optimize_depth_gpu(float** h_flows, float** h_rig, float** h_o_rig, float** h_dp, float** h_pc, float** h_cf,
                           float** h_o_cf, float* h_depth, float* h_o_depth, float* h_K, float** h_Rs, float** h_ts,
                           float** h_dp_Rs, float** h_dp_ts, float abs_rf, int N, int N_dp, int w, int h,
                           float basefocal, int n_rand, int gstep, int lwidth, float lambda, float omega,
                           float disp_delta, float delta, int fb, float s0e, float nc, float range_factor,
                           int rig_only) {
    DepthState& S = g_depth;
    const size_t npx = (size_t)w * h;
    S.N = N, S.N_dp = N_dp;
    S.abs_rf = abs_rf, S.basefocal = basefocal, S.lambda = lambda, S.omega = omega, S.delta = delta;
    S.disp_delta = disp_delta, S.range_factor = range_factor;
    if (h_K) set_K(S.cam, h_K);
    if (S.w != w || S.h != h) {
        S.w = w, S.h = h;
        S.rng.resize(npx);
#pragma omp parallel for
        for (long long i = 0; i < (long long)npx; i++) curand_init(233ULL, (unsigned long long)i, 0ULL, &S.rng[i]);
        S.cost.assign(npx, 0), S.depth.assign(npx, 0);
        S.flows = Stack<2>(), S.rig = Stack<1>(), S.dp = Stack<1>(), S.dp_pconf = Stack<1>(), S.dp_conf = Stack<1>();
    }
    if (h_depth) memcpy(S.depth.data(), h_depth, npx * sizeof(float));
    if (N > 0) {
        if (h_Rs)
            for (int f = 0; f < N; f++) memcpy(S.cam.R[f], h_Rs[f], 36);
        if (h_ts)
            for (int f = 0; f < N; f++) memcpy(S.cam.t[f], h_ts[f], 12);
        S.flows.ensure(w, h, N), S.rig.ensure(w, h, N);
        if (h_flows)
            for (int f = 0; f < N; f++) memcpy(S.flows.layer(f), h_flows[f], npx * 2 * sizeof(float));
        if (h_rig)
            for (int f = 0; f < N; f++) memcpy(S.rig.layer(f), h_rig[f], npx * sizeof(float));
    }
    if (N_dp > 0) {
        if (h_dp_Rs)
            for (int f = 0; f < N_dp; f++) memcpy(S.pcam.R[f], h_dp_Rs[f], 36);
        if (h_dp_ts)
            for (int f = 0; f < N_dp; f++) memcpy(S.pcam.t[f], h_dp_ts[f], 12);
        S.dp.ensure(w, h, N_dp), S.dp_pconf.ensure(w, h, N_dp), S.dp_conf.ensure(w, h, N_dp);
        if (h_dp)
            for (int f = 0; f < N_dp; f++) memcpy(S.dp.layer(f), h_dp[f], npx * sizeof(float));
        if (h_pc)
            for (int f = 0; f < N_dp; f++) memcpy(S.dp_pconf.layer(f), h_pc[f], npx * sizeof(float));
        if (h_cf)
            for (int f = 0; f < N_dp; f++) memcpy(S.dp_conf.layer(f), h_cf[f], npx * sizeof(float));
    }
    if (!rig_only) {
        if (fb) {
            if (N > 0) fb_smooth(S.rig.data.data(), N, w, h, s0e, nc);
            if (N_dp > 0) fb_smooth(S.dp_conf.data.data(), N_dp, w, h, s0e, nc);
        }
        // cost map + random samples (optimize_depth.cu:269-284,472-478)
#pragma omp parallel for schedule(dynamic, 4)
        for (int y = 0; y < h; y++)
            for (int x = 0; x < w; x++) {
                const size_t i = (size_t)y * w + x;
                S.cost[i] = S.pixel_cost(x, y, S.depth[i]);
                for (int it = 0; it < n_rand; it++) {
                    const float d = 1.0f / (range_factor * curand_uniform(&S.rng[i]) + (1.0f / 1e5f));
                    S.try_depth(x, y, d);
                }
            }
        if (gstep > 0) {  // global propagation L2R, B2T, R2L, T2B (optimize_depth.cu:209-235,480-485)
#pragma omp parallel for
            for (int y = 0; y < h; y++)
                for (int x = 1; x < w; x += gstep) S.try_depth(x, y, S.depth[(size_t)y * w + x - 1]);
#pragma omp parallel for
            for (int x = 0; x < w; x++)
                for (int y = h - 2; y >= 0; y -= gstep) S.try_depth(x, y, S.depth[(size_t)(y + 1) * w + x]);
#pragma omp parallel for
            for (int y = 0; y < h; y++)
                for (int x = w - 2; x >= 0; x -= gstep) S.try_depth(x, y, S.depth[(size_t)y * w + x + 1]);
#pragma omp parallel for
            for (int x = 0; x < w; x++)
                for (int y = 1; y < h; y += gstep) S.try_depth(x, y, S.depth[(size_t)(y - 1) * w + x]);
        }
        if (lwidth > 0) {  // local propagation, same order (optimize_depth.cu:237-267,486-491)
            const int nsx = (w + lwidth - 1) / lwidth, nsy = (h + lwidth - 1) / lwidth;
#pragma omp parallel for collapse(2)
            for (int y = 0; y < h; y++)
                for (int sx = 0; sx < nsx; sx++) {
                    const int p0 = sx * lwidth;
                    for (int x = std::max(1, p0 + 1); x < std::min(w, p0 + lwidth); x++)
                        S.try_depth(x, y, S.depth[(size_t)y * w + x - 1]);
                }
#pragma omp parallel for collapse(2)
            for (int x = 0; x < w; x++)
                for (int sy = 0; sy < nsy; sy++) {
                    const int p0 = sy * lwidth;
                    for (int y = std::min(h - 2, p0 + lwidth - 2); y >= std::max(0, p0); y--)
                        S.try_depth(x, y, S.depth[(size_t)(y + 1) * w + x]);
                }
#pragma omp parallel for collapse(2)
            for (int y = 0; y < h; y++)
                for (int sx = 0; sx < nsx; sx++) {
                    const int p0 = sx * lwidth;
                    for (int x = std::min(w - 2, p0 + lwidth - 2); x >= std::max(0, p0); x--)
                        S.try_depth(x, y, S.depth[(size_t)y * w + x + 1]);
                }
#pragma omp parallel for collapse(2)
            for (int x = 0; x < w; x++)
                for (int sy = 0; sy < nsy; sy++) {
                    const int p0 = sy * lwidth;
                    for (int y = std::max(1, p0 + 1); y < std::min(h, p0 + lwidth); y++)
                        S.try_depth(x, y, S.depth[(size_t)(y - 1) * w + x]);
                }
        }
    }
    S.update_rigidness();
    if (h_o_depth) memcpy(h_o_depth, S.depth.data(), npx * sizeof(float));
    if (h_o_rig)
        for (int f = 0; f < N; f++) memcpy(h_o_rig[f], S.rig.layer(f), npx * sizeof(float));
    if (h_o_cf)
        for (int f = 0; f < N_dp; f++) memcpy(h_o_cf[f], S.dp_conf.layer(f), npx * sizeof(float));
    return 0;
}

// collect_p3p_instances.cu:70-250
int cpu_collect_p3p_instances(float** h_flows, float** h_rig, float* h_depth, float* h_K, float** h_Rs, float** h_ts,
                              float* o_p2, float* o_p3, int N, int w, int h, int active_idx, float rig_thresh,
                              float rig_sum_thresh, float min_d, float max_d, int max_trace) {
    static Stack<2> flows;
    static Stack<1> rig;
    static std::vector<float> depth;
    static Cam cam;
    const size_t npx = (size_t)w * h;
    if (h_K) set_K(cam, h_K);
    if (h_Rs)
        for (int f = 0; f < N; f++) memcpy(cam.R[f], h_Rs[f], 36);
    if (h_ts)
        for (int f = 0; f < N; f++) memcpy(cam.t[f], h_ts[f], 12);
    flows.ensure(w, h, N), rig.ensure(w, h, N);
    if (h_flows)
        for (int f = 0; f < N; f++) memcpy(flows.layer(f), h_flows[f], npx * 2 * sizeof(float));
    if (h_rig)
        for (int f = 0; f < N; f++) memcpy(rig.layer(f), h_rig[f], npx * sizeof(float));
    if (depth.size() != npx) depth.assign(npx, 0);
    if (h_depth) memcpy(depth.data(), h_depth, npx * sizeof(float));
#pragma omp parallel for schedule(dynamic, 4)
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++) {
            const size_t i = (size_t)y * w + x;
            float* p2 = o_p2 + i * 2;
            float* p3 = o_p3 + i * 3;
            p2[0] = p2[1] = p3[0] = p3[1] = p3[2] = NAN;
            const float d = depth[i];
            if (d < min_d || (max_d > 0 && d > max_d)) continue;
            if (rig_sum_thresh > N + 1) {
                float s = 0;
                for (int f = 0; f < N; f++) s += rig.data[(size_t)f * npx + i];
                if (s < rig_sum_thresh) continue;
            }
            int n_trace = 0;
            float tp = 1;
            for (int f = active_idx; f >= (max_trace > 0 ? std::max(0, active_idx - max_trace + 1) : 0); f--) {
                tp *= rig.data[(size_t)f * npx + i];
                if (tp > rig_thresh)
                    n_trace++;
                else
                    break;
            }
            if (n_trace <= 0) continue;
            bool out = false;
            float px = 0, py = 0, ox, oy, oz;
            p2_to_p3(cam, (float)x, (float)y, d, ox, oy, oz);
            for (int f = 0; f <= active_idx; f++) {
                if (f >= active_idx - n_trace + 1) {
                    if (f == active_idx - n_trace + 1) p3_to_p2(cam, ox, oy, oz, px, py);
                    if (px > 0 && px < w && py > 0 && py < h) {
                        float d2[2];
                        flows.tex(px, py, f, d2);
                        px += d2[0], py += d2[1];
                    } else {
                        out = true;
                        break;
                    }
                }
                if (f < active_idx) trans(cam.R[f], cam.t[f], ox, oy, oz);
            }
            if (!out && oz > min_d && (max_d <= 0 || oz < max_d)) p2[0] = px, p2[1] = py, p3[0] = ox, p3[1] = oy, p3[2] = oz;
        }
    return 0;
}

// solve_batch_lambdatwist.cu:11-102 (indices from the same cuRAND streams)
int cpu_solve_batch_p3p_lambdatwist_gpu(float* h_p3s, float* h_p2s, float* o_rvecs, float* o_tvecs, float* h_K,
                                        int N_pts, int N_poses) {
#ifdef HAVE_REF_LAMBDATWIST
    const float fx = h_K[0], cx = h_K[2], fy = h_K[4], cy = h_K[5];
#pragma omp parallel for schedule(dynamic, 64)
    for (int idx = 0; idx < N_poses; idx++) {
        curandStateXORWOW_t st;
        curand_init(233ULL, (unsigned long long)idx, 0ULL, &st);
        int i[4];
        for (int k = 0; k < 4; k++) i[k] = std::min((int)(curand_uniform(&st) * N_pts), N_pts - 1);
        float R[3][3], t[3];
        const bool ok = lambdatwist_p4p<float, float, 5>(&h_p2s[i[0] * 2], &h_p2s[i[1] * 2], &h_p2s[i[2] * 2],
                                                         &h_p2s[i[3] * 2], &h_p3s[i[0] * 3], &h_p3s[i[1] * 3],
                                                         &h_p3s[i[2] * 3], &h_p3s[i[3] * 3], fx, fy, cx, cy, R, t);
        float* rv = o_rvecs + idx * 3;
        float* tv = o_tvecs + idx * 3;
        if (!ok) {
            rv[0] = rv[1] = rv[2] = tv[0] = tv[1] = tv[2] = NAN;
            continue;
        }
        tv[0] = t[0], tv[1] = t[1], tv[2] = t[2];
        vb::hm::matrix_to_rvec(&R[0][0], rv);
    }
    return 0;
#else
    const float fx = h_K[0], cx = h_K[2], fy = h_K[4], cy = h_K[5];
#pragma omp parallel for schedule(dynamic, 64)
    for (int idx = 0; idx < N_poses; idx++) {
        curandStateXORWOW_t st;
        curand_init(233ULL, (unsigned long long)idx, 0ULL, &st);
        float uv[8];
        vb::quad::Vec3f X[4];
        for (int k = 0; k < 4; k++) {
            const int i = std::min((int)(curand_uniform(&st) * N_pts), N_pts - 1);
            uv[2 * k] = h_p2s[2 * i], uv[2 * k + 1] = h_p2s[2 * i + 1];
            X[k] = vb::quad::Vec3f{h_p3s[3 * i], h_p3s[3 * i + 1], h_p3s[3 * i + 2]};
        }
        vb::quad::Pose P[4];
        bool exists[4];
        float err[4];
        for (int q = 0; q < 4; q++) err[q] = 0.f, exists[q] = vb::quad::twist_lane(q, uv, X, fx, fy, cx, cy, P[q], err[q]);
        const int best = vb::quad::pick_by_fourth_point(exists, err);
        float* rv = o_rvecs + idx * 3;
        float* tv = o_tvecs + idx * 3;
        if (best < 0) {
            rv[0] = rv[1] = rv[2] = tv[0] = tv[1] = tv[2] = NAN;
            continue;
        }
        tv[0] = P[best].t[0], tv[1] = P[best].t[1], tv[2] = P[best].t[2];
        vb::hm::matrix_to_rvec(P[best].R, rv);
    }
    return 0;
#endif
}
int cpu_solve_batch_p3p_ap3p_gpu(float* a, float* b, float* c, float* d, float* e, int n, int m) {
    // the CPU port carries one minimal solver; AP3P parity is checked against oracle/_ref on the GPU
    return cpu_solve_batch_p3p_lambdatwist_gpu(a, b, c, d, e, n, m);
}

// meanshift.cu:34-150
int cpu_meanshift_gpu(float* space, float kernel_var, float* io_mean, float* o_conf, int* used_iters, int external,
                      int N, int dims, float eps, int max_iters, int max_trials, float good_conf) {
    std::vector<float> c_mean(io_mean, io_mean + dims), wv(N);
    std::vector<std::vector<float>> ws(dims, std::vector<float>(N));
    auto weights = [&](bool only_w) {
#pragma omp parallel for
        for (int i = 0; i < N; i++) {
            float l2 = 0;
            for (int d = 0; d < dims; d++) l2 += (space[i * dims + d] - c_mean[d]) * (space[i * dims + d] - c_mean[d]);
            const float wgt = std::exp(-l2 / (2 * kernel_var));
            wv[i] = wgt;
            if (!only_w)
                for (int d = 0; d < dims; d++) ws[d][i] = space[i * dims + d] * wgt;
        }
    };
    if (!external) {
        float best = 0;
        int best_idx = -1;
        for (int trial = 0; trial < max_trials; trial++) {
            const int idx = rand() % N;
            for (int d = 0; d < dims; d++) c_mean[d] = space[idx * dims + d];
            weights(true);
            const float s = tree_sum(wv);
            if (s > best) best = s, best_idx = idx;
            if (best > good_conf * N) break;
        }
        for (int d = 0; d < dims; d++) c_mean[d] = space[best_idx * dims + d];
    }
    if (used_iters) *used_iters = 0;
    for (int iter = 0; iter < max_iters; iter++) {
        weights(false);
        const float wsum = tree_sum(wv);
        std::vector<float> m(dims);
        for (int d = 0; d < dims; d++) m[d] = tree_sum(ws[d]) / wsum;
        if (o_conf) *o_conf = wsum / N;
        if (used_iters) *used_iters = iter + 1;
        float disp = 0;
        for (int d = 0; d < dims; d++) disp += (io_mean[d] - m[d]) * (io_mean[d] - m[d]);
        disp = std::sqrt(disp);
        for (int d = 0; d < dims; d++) io_mean[d] = m[d];
        if (disp < eps) break;
        for (int d = 0; d < dims; d++) c_mean[d] = io_mean[d];
    }
    return 0;
}

// fit_robust_gaussian.cu:101-286 (dims must be 6: aux functions are 6x6, aux_funs.cpp:101-119)
int cpu_fit_robust_gaussian(float* space, float* io_mean, float* io_covar, float trunc_sigma, float reg_lambda,
                            float* o_density, int* used_iters, int N, int dims, float eps, int max_iters) {
    if (dims != 6) return 1;
    const int cd = 21;
    float ht_weight = 0, mean[6], cov[21], cinv[21];
    double full[36], inv[36];
    for (int d = 0; d < 6; d++) mean[d] = io_mean[d];
    for (int d1 = 0; d1 < 6; d1++)
        for (int d2 = 0; d2 <= d1; d2++) cov[(d1 * d1 + d1) / 2 + d2] = io_covar[d1 * 6 + d2];
    std::vector<float> W(N);
    std::vector<std::vector<float>> WS(6, std::vector<float>(N)), WC(cd, std::vector<float>(N));
    if (used_iters) *used_iters = 0;
    int iter;
    bool reliable = true;
    for (iter = 0; iter < max_iters; iter++) {
        for (int d1 = 0; d1 < 6; d1++)
            for (int d2 = 0; d2 <= d1; d2++) full[d1 * 6 + d2] = full[d2 * 6 + d1] = (double)cov[(d1 * d1 + d1) / 2 + d2];
        if (iter > 0 && reg_lambda > 0) regularize_covar_LW_given_lambda(full, full, reg_lambda, 6);
        if (inverse(full, inv, 6) <= 0) {
            reliable = false;
            break;
        }
        for (int d1 = 0; d1 < 6; d1++)
            for (int d2 = 0; d2 <= d1; d2++)
                cov[(d1 * d1 + d1) / 2 + d2] = (float)full[d1 * 6 + d2], cinv[(d1 * d1 + d1) / 2 + d2] = (float)inv[d1 * 6 + d2];
        const float prev = ht_weight / N;
#pragma omp parallel for
        for (int i = 0; i < N; i++) {
            float diff[6], z = 0;
            for (int d = 0; d < 6; d++) diff[d] = space[i * 6 + d] - mean[d];
            for (int d1 = 0; d1 < 6; d1++) {
                float tmp = 0;
                for (int d2 = 0; d2 < 6; d2++)
                    tmp += (d1 >= d2 ? cinv[(d1 * d1 + d1) / 2 + d2] : cinv[(d2 * d2 + d2) / 2 + d1]) * diff[d2];
                z += tmp * diff[d1];
            }
            const float wgt = std::sqrt(z) < trunc_sigma ? 1.f : 0.f;
            W[i] = wgt;
            for (int d = 0; d < 6; d++) WS[d][i] = wgt * space[i * 6 + d];
            for (int d1 = 0; d1 < 6; d1++)
                for (int d2 = 0; d2 <= d1; d2++) WC[(d1 * d1 + d1) / 2 + d2][i] = wgt * diff[d1] * diff[d2];
        }
        ht_weight = tree_sum(W);
        if (!std::isfinite(ht_weight)) {
            reliable = false;
            break;
        }
        if (std::fabs(ht_weight / N - prev) < eps) break;
        for (int d = 0; d < 6; d++) mean[d] = tree_sum(WS[d]) / ht_weight;
        for (int k = 0; k < cd; k++) cov[k] = tree_sum(WC[k]) / ht_weight;
    }
    if (reliable) {
        if (o_density) *o_density = ht_weight / N;
        if (used_iters) *used_iters = iter;
        for (int d1 = 0; d1 < 6; d1++)
            for (int d2 = 0; d2 <= d1; d2++) io_covar[d1 * 6 + d2] = io_covar[d2 * 6 + d1] = cov[(d1 * d1 + d1) / 2 + d2];
        for (int d = 0; d < 6; d++) io_mean[d] = mean[d];
    }
    return reliable ? 0 : 1;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
// frame alignment (SURVEY §8a row 10).  Restates gpu-kernels/align_frame.cu: rotation by a rotation vector with
// its two Jacobians (:47-134; the rvec Jacobian keeps the reference's theta^(3/2) where the analytic derivative
// has theta^3, SURVEY §9 Q17-Q18), projections (:136-150), normals and image gradients (:152-209; out-of-range
// neighbours go through at_safe, whose unsigned index wraps -1 to the LAST row/column, gmat.h:181-186), the
// point-to-plane + colour residual and its Jacobian (:211-376), the weighted sqrt-Cauchy loss (:378-403) and the two
// entry points (:414-554).  PARITY UNPINNED in round 1: no golden vector of the reference exists for it yet; it is
// checked for internal consistency on the CPU and cross-checked against the CUDA path on the GPU at 1e-3.
// ---------------------------------------------------------------------------------------------------
namespace {

struct V3 {
    float x, y, z;
};
inline V3 v3(float x, float y, float z) { return V3{x, y, z}; }
inline V3 operator+(V3 a, V3 b) { return v3(a.x + b.x, a.y + b.y, a.z + b.z); }
inline V3 operator-(V3 a, V3 b) { return v3(a.x - b.x, a.y - b.y, a.z - b.z); }
inline V3 operator*(V3 a, float s) { return v3(a.x * s, a.y * s, a.z * s); }
inline float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
inline V3 cross(V3 a, V3 b) { return v3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }

// q = R(r) p; J_r = dq/dr (reference closed form), J_p = dq/dp = R
V3 rotate_rvec(V3 p, V3 r, float J_r[3][3], float J_p[3][3]) {
    const float th2 = dot(r, r);
    const float rv[3] = {r.x, r.y, r.z}, pv[3] = {p.x, p.y, p.z};
    if (!(th2 > FLT_EPSILON)) {  // first-order branch
        const float S[3][3] = {{0, -r.z, r.y}, {r.z, 0, -r.x}, {-r.y, r.x, 0}};
        const float Sp[3][3] = {{0, p.z, -p.y}, {-p.z, 0, p.x}, {p.y, -p.x, 0}};
        for (int i = 0; i < 3; i++)
            for (int j = 0; j < 3; j++) {
                if (J_p) J_p[i][j] = (i == j ? 1.f : 0.f) + S[i][j];
                if (J_r) J_r[i][j] = Sp[i][j];
            }
        return p + cross(r, p);
    }
    const float th = std::sqrt(th2), c = std::cos(th), s = std::sin(th), cm1 = c - 1;
    const V3 w = r * (1.f / th);
    if (J_p) {  // c I + s [w]x + (1 - c) w w^T, written with r and theta like the reference
        const float sg[3][3] = {{0, -1, 1}, {1, 0, -1}, {-1, 1, 0}};
        for (int i = 0; i < 3; i++)
            for (int j = 0; j < 3; j++)
                J_p[i][j] = i == j ? c - ((rv[i] * rv[i]) * cm1) / th2
                                   : sg[i][j] * (rv[3 - i - j] * s) / th - (rv[i] * rv[j] * cm1) / th2;
    }
    if (J_r) {
        const float t32 = std::sqrt(th2 * th);  // theta^(3/2): the reference's expression, not theta^3
        const float wp = (r.x * p.x) / th + (r.y * p.y) / th + (r.z * p.z) / th;
        const V3 rxp = cross(r, p);
        const float cx[3] = {rxp.x, rxp.y, rxp.z};
        const float dcx[3][3] = {{0, p.z, -p.y}, {-p.z, 0, p.x}, {p.y, -p.x, 0}};  // d(r x p)_i / d r_j
        for (int i = 0; i < 3; i++)
            for (int j = 0; j < 3; j++) {
                const float rrp = (rv[j] * rv[0] * pv[0]) / t32 + (rv[j] * rv[1] * pv[1]) / t32 + (rv[j] * rv[2] * pv[2]) / t32;
                float v = s * (dcx[i][j] / th - (rv[j] * cx[i]) / t32);
                if (i == j) v -= (cm1 * wp) / th;
                v += (rv[i] * cm1 * (rrp - pv[j] / th)) / th;
                v -= (rv[j] * pv[i] * s) / th;
                v += (rv[i] * rv[j] * cm1 * wp) / t32;
                v += (rv[i] * rv[j] * s * wp) / th2;
                v += (rv[j] * c * (cx[i] / th)) / th;
                J_r[i][j] = v;
            }
    }
    return p * c + cross(w, p) * s + w * (dot(w, p) * (1.0f - c));
}

struct AlignState {
    int N = 0, w = 0, h = 0;
    bool photo = false;
    float fx = 0, cx = 0, fy = 0, cy = 0, fxi = 0, cxi = 0, fyi = 0, cyi = 0, vbf = 0, crw = 0;
    Stack<1> images, depths;
    Stack<2> dimages;
    Stack<4> normals;
    std::vector<float> weights;
    float p_ref[9] = {0}, p_tar[9] = {0};
    V3 lift(float px, float py, float d) const { return v3((fxi * px + cxi) * d, (fyi * py + cyi) * d, d); }
    void drop(V3 p, float& px, float& py) const { px = (fx * p.x) / p.z + cx, py = (fy * p.y) / p.z + cy; }
    static int wrap(int i, int n) { return i < 0 ? n - 1 : (i > n - 1 ? n - 1 : i); }  // at_safe on size_t
    float safe(const Stack<1>& m, int x, int y, int f) const {
        return m.data[((size_t)f * h + wrap(y, h)) * w + wrap(x, w)];
    }
    // 0.3 / 0.1 / 0.1 central differences (align_frame.cu:176-183,196-204)
    void gradient(const Stack<1>& m, int x, int y, int f, float& gx, float& gy) const {
        gx = 0.3f * (safe(m, x + 1, y, f) - safe(m, x - 1, y, f)) + 0.1f * (safe(m, x + 1, y - 1, f) - safe(m, x - 1, y - 1, f)) +
             0.1f * (safe(m, x + 1, y + 1, f) - safe(m, x - 1, y + 1, f));
        gy = 0.3f * (safe(m, x, y + 1, f) - safe(m, x, y - 1, f)) + 0.1f * (safe(m, x - 1, y + 1, f) - safe(m, x - 1, y - 1, f)) +
             0.1f * (safe(m, x + 1, y + 1, f) - safe(m, x + 1, y - 1, f));
    }
} g_align;

}  // namespace

extern "C" {

int cpu_align_frame_init_gpu(float** h_images, float** h_depths, float** h_weights, float* h_K, float vbf, float crw,
                             int N, int w, int h) {
    AlignState& A = g_align;
    A.N = N, A.w = w, A.h = h, A.vbf = vbf, A.crw = crw;
    A.fx = h_K[0], A.cx = h_K[2], A.fy = h_K[4], A.cy = h_K[5];
    A.fxi = 1.f / h_K[0], A.cxi = -h_K[2] / h_K[0], A.fyi = 1.f / h_K[4], A.cyi = -h_K[5] / h_K[4];
    const size_t npx = (size_t)w * h;
    A.photo = h_images && crw > 0;
    A.depths.ensure(w, h, N), A.normals.ensure(w, h, N);
    A.weights.assign(npx * N, 0.f);
    for (int f = 0; f < N; f++) {
        memcpy(A.depths.layer(f), h_depths[f], npx * sizeof(float));
        memcpy(A.weights.data() + f * npx, h_weights[f], npx * sizeof(float));
    }
    if (A.photo) {
        A.images.ensure(w, h, N), A.dimages.ensure(w, h, N);
        for (int f = 0; f < N; f++) memcpy(A.images.layer(f), h_images[f], npx * sizeof(float));
    }
    for (int f = 0; f < N; f++) {
#pragma omp parallel for
        for (int y = 0; y < h; y++)
            for (int x = 0; x < w; x++) {
                // normal from the four neighbours, turned towards the camera
                const V3 t = A.lift((float)x, (float)(y - 1), A.safe(A.depths, x, y - 1, f));
                const V3 b = A.lift((float)x, (float)(y + 1), A.safe(A.depths, x, y + 1, f));
                const V3 l = A.lift((float)(x - 1), (float)y, A.safe(A.depths, x - 1, y, f));
                const V3 r = A.lift((float)(x + 1), (float)y, A.safe(A.depths, x + 1, y, f));
                V3 n = cross(t - b, l - r);
                const float len = std::sqrt(dot(n, n));
                n = v3(n.x / len, n.y / len, n.z / len);
                if (dot(A.lift((float)x, (float)y, 1.f), n) > 0) n = n * -1.f;
                float* o = A.normals.layer(f) + ((size_t)y * w + x) * 4;
                o[0] = n.x, o[1] = n.y, o[2] = n.z, o[3] = 0;
                if (A.photo) {
                    float* g = A.dimages.layer(f) + ((size_t)y * w + x) * 2;
                    A.gradient(A.images, x, y, f, g[0], g[1]);
                }
            }
    }
    return 0;
}

int cpu_align_frame_eval_gpu(int ref_fid, int tar_fid, const float* h_params_ref, const float* h_params_tar,
                             float* h_o_residual, float* h_o_jacobian, int apply_weights) {
    AlignState& A = g_align;
    if (h_params_ref) memcpy(A.p_ref, h_params_ref, sizeof(A.p_ref));
    if (h_params_tar) memcpy(A.p_tar, h_params_tar, sizeof(A.p_tar));
    const int w = A.w, h = A.h;
    const bool want_jac = h_o_jacobian != nullptr;
    std::vector<float> res((size_t)w * h, 0.f), jac(want_jac ? (size_t)w * h * 9 : 0, 0.f);
    const float* pr = A.p_ref;
    const float* pt = A.p_tar;
    // target pose inverted once: world -> target camera
    const V3 r_tar = v3(-pt[0], -pt[1], -pt[2]);
    const V3 t_tar = rotate_rvec(v3(pt[3], pt[4], pt[5]), r_tar, nullptr, nullptr) * -1.f;
#pragma omp parallel for
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++) {
            const size_t px = (size_t)y * w + x;
            const float nan = std::nanf("");
            // reference pixel -> world -> target camera
            const float d_ref = A.depths.data[((size_t)ref_fid * h + y) * w + x] * std::exp(pr[6]);
            const V3 ray = v3(A.fxi * x + A.cxi, A.fyi * y + A.cyi, 1.f);  // d p3r / d depth
            const V3 p3r = ray * d_ref;
            float Jw_r[3][3], Jw_p[3][3], Jt_w[3][3];
            const V3 p3w = rotate_rvec(p3r, v3(pr[0], pr[1], pr[2]), want_jac ? Jw_r : nullptr, want_jac ? Jw_p : nullptr) +
                           v3(pr[3], pr[4], pr[5]);
            const V3 p3t = rotate_rvec(p3w, r_tar, nullptr, want_jac ? Jt_w : nullptr) + t_tar;
            float u, v;
            A.drop(p3t, u, v);
            if (u < 0 || u >= w || v < 0 || v >= h || p3t.z < 1.f) {
                res[px] = nan;
                continue;
            }
            float dt, nt[4];
            A.depths.tex(u, v, tar_fid, &dt);
            dt *= std::exp(pt[6]);
            A.normals.tex(u, v, tar_fid, nt);
            const V3 n = v3(nt[0], nt[1], nt[2]);
            // point-to-plane offset between the target surface point on the same ray and the warped point
            const V3 on_ray = p3t * (dt / p3t.z);
            const V3 off = n * dot(n, on_ray - p3t);
            const V3 hit = p3t + off;
            float hu, hv;
            A.drop(hit, hu, hv);
            if (hu < 0 || hu >= w || hv < 0 || hv >= h) {
                res[px] = nan;
                continue;
            }
            const float r_depth = 0.5f * dot(off, off);
            const float q = A.vbf / (std::fmax(hit.z, 1.0f) * std::fmax(p3t.z, 1.0f));
            const float drw = q * q;
            float c_ref = 0, c_tar = 0, r_color = 0;
            if (A.photo) {
                float ci;
                A.images.tex(u, v, tar_fid, &ci);
                c_ref = A.images.data[((size_t)ref_fid * h + y) * w + x] + pr[8];
                c_tar = (ci + pt[8]) * (std::exp(pr[7]) / std::exp(pt[7]));
                r_color = 0.5f * (c_ref - c_tar) * (c_ref - c_tar);
            }
            res[px] = A.photo ? drw * r_depth + A.crw * r_color : drw * r_depth;
            if (!want_jac) continue;
            // d residual / d p3t: geometric part -off (weights drw treated as constants, like the reference),
            // colour part through the image gradient and the projection
            V3 g = off * -drw;
            float dres_dcs = 0, dres_dco = 0;
            if (A.photo) {
                float gi[2];
                A.dimages.tex(u, v, tar_fid, gi);
                const float dc = c_tar - c_ref;
                const float P[2][3] = {{A.fx / p3t.z, 0, -(A.fx * p3t.x) / (p3t.z * p3t.z)},
                                       {0, A.fy / p3t.z, -(A.fy * p3t.y) / (p3t.z * p3t.z)}};
                const float gu = gi[0] * dc, gv = gi[1] * dc;
                g = g + v3(gu * P[0][0] + gv * P[1][0], gu * P[0][1] + gv * P[1][1], gu * P[0][2] + gv * P[1][2]) * A.crw;
                dres_dcs = A.crw * (dc * c_tar);
                dres_dco = A.crw * ((c_ref - c_tar) * 1.f);
            }
            const float gv3[3] = {g.x, g.y, g.z};
            float gw[3], gr[3], gp[3];
            for (int j = 0; j < 3; j++) gw[j] = gv3[0] * Jt_w[0][j] + gv3[1] * Jt_w[1][j] + gv3[2] * Jt_w[2][j];
            for (int j = 0; j < 3; j++) gr[j] = gw[0] * Jw_r[0][j] + gw[1] * Jw_r[1][j] + gw[2] * Jw_r[2][j];
            for (int j = 0; j < 3; j++) gp[j] = gw[0] * Jw_p[0][j] + gw[1] * Jw_p[1][j] + gw[2] * Jw_p[2][j];
            float* J = jac.data() + px * 9;
            J[0] = gr[0], J[1] = gr[1], J[2] = gr[2];
            J[3] = gw[0], J[4] = gw[1], J[5] = gw[2];  // d p3w / d tvec = I
            J[6] = (gp[0] * ray.x + gp[1] * ray.y + gp[2] * ray.z) * d_ref;  // through depth * exp(scale)
            J[7] = dres_dcs, J[8] = dres_dco;
        }
    // weighted sqrt-Cauchy loss on residual and Jacobian
#pragma omp parallel for
    for (int i = 0; i < w * h; i++) {
        const float wgt = apply_weights ? A.weights[(size_t)ref_fid * w * h + i] : 1.f;
        const float r2 = wgt * res[i];
        if (r2 > FLT_EPSILON) {
            const float loss = std::log(r2 + 1.f), root = std::sqrt(loss);
            res[i] = root;
            if (want_jac) {
                const float k = (0.5f / root) * (1.f / (r2 + 1.f)) * wgt;
                for (int c = 0; c < 9; c++) jac[(size_t)i * 9 + c] *= k;
            }
        }
    }
    if (h_o_residual) memcpy(h_o_residual, res.data(), res.size() * sizeof(float));
    if (want_jac) memcpy(h_o_jacobian, jac.data(), jac.size() * sizeof(float));
    return 0;
}

}  // extern "C"
