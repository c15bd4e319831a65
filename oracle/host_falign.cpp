// TEST INFRASTRUCTURE (oracle).  Host restatement of frame alignment (DESIGN.md §9): a plain loop that evaluates every
// connectivity pair through a per-sample evaluation bound at run time, builds the normal equations with the summation
// tree of voldor_b200/csrc/falign_math.h, and steps with the same restated Levenberg-Marquardt header.
//
// The evaluation behind it (dlopen + symbol prefix, like host_voldor.cpp):
//   prefix "cpu_": the CPU port (oracle/cpu_kernels.cpp), full-resolution evaluation, subsampled here;
//   prefix "vb_" : this library's vb_align_frame_eval_strided (use_strided = 1), or its full-resolution
//                  vb_align_frame_eval_gpu with the full residual and Jacobian downloaded per evaluation and
//                  subsampled here (use_strided = 0) — the reference's own data flow;
//   prefix "ref_": the reference's kernels (oracle/_ref), full resolution.
#include <dlfcn.h>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>
#include <vector>
#include "../voldor_b200/csrc/falign_math.h"

namespace {

using namespace vb::fa;
using fn_init = int (*)(float**, float**, float**, float*, float, float, int, int, int);
using fn_eval = int (*)(int, int, const float*, const float*, float*, float*, int);
using fn_strided = int (*)(int, int, const float*, const float*, float*, float*, int, int);

struct Eval {
    fn_init init = nullptr;
    fn_eval full = nullptr;
    fn_strided strided = nullptr;
} g_eval;

struct Problem {
    int N, w, h, stride, n, ow;
    const std::vector<int>* pairs;
    std::vector<float> res, jac, fres, fjac;
};

// per-sample residual + Jacobian of pair p at (pref, ptar), packed like vb_align_frame_eval_strided
bool eval_pair(Problem& P, int p, const float* pref, const float* ptar, bool weights_and_jac, int stride) {
    const int ref = (*P.pairs)[p * 3], tar = (*P.pairs)[p * 3 + 1];
    const int ow = (P.w + stride - 1) / stride, oh = (P.h + stride - 1) / stride;
    const size_t n = (size_t)ow * oh;
    P.res.resize(n), P.jac.resize(n * kP);
    float* jac = weights_and_jac ? P.jac.data() : nullptr;
    if (g_eval.strided && stride > 1)
        return g_eval.strided(ref, tar, pref, ptar, P.res.data(), jac, weights_and_jac, stride) == 0;
    const size_t npx = (size_t)P.w * P.h;
    P.fres.resize(npx), P.fjac.resize(npx * kP);
    if (g_eval.full(ref, tar, pref, ptar, P.fres.data(), jac ? P.fjac.data() : nullptr, weights_and_jac) != 0)
        return false;
    for (int gy = 0; gy < oh; gy++)
        for (int gx = 0; gx < ow; gx++) {
            const size_t k = (size_t)gy * ow + gx, px = (size_t)gy * stride * P.w + (size_t)gx * stride;
            P.res[k] = P.fres[px];
            if (jac) memcpy(&P.jac[k * kP], &P.fjac[px * kP], kP * sizeof(float));
        }
    return true;
}

// the summation tree over n samples: blocks of 256 by reduce_block, block sums in order from +0
double tree_sum(const std::vector<double>& v) {
    double s = 0.0, blk[kBlock];
    for (size_t b = 0; b < v.size(); b += kBlock) {
        for (int i = 0; i < kBlock; i++) blk[i] = b + i < v.size() ? v[b + i] : 0.0;
        s = vb::hm::det::add(s, reduce_block(blk));
    }
    return s;
}

// normal equations of every pair at (ref = xr, target = xt) -> frame sums fs[N][kQ]
bool normal_equations(Problem& P, const double (*xr)[kP], const double (*xt)[kP], bool use_factor,
                      std::vector<double>& fs) {
    const int npairs = (int)P.pairs->size() / 3;
    std::vector<double> pair_sums((size_t)npairs * kQ), v;
    for (int p = 0; p < npairs; p++) {
        float pref[kP], ptar[kP];
        params_float(xr[(*P.pairs)[p * 3]], pref);
        params_float(xt[(*P.pairs)[p * 3 + 1]], ptar);
        if (!eval_pair(P, p, pref, ptar, true, P.stride)) return false;
        const float factor = use_factor ? (float)(*P.pairs)[p * 3 + 2] : 1.f;
        const size_t n = P.res.size();
        std::vector<float> f(n), J(n * kP);
        for (size_t k = 0; k < n; k++) {
            const bool ok = std::isfinite(P.res[k]);
            f[k] = ok ? P.res[k] : 0.f;
            for (int i = 0; i < kP; i++) J[k * kP + i] = (ok ? P.jac[k * kP + i] : 0.f) * factor;
        }
        v.resize(n);
        for (int q = 0; q < kQ; q++) {
            for (size_t k = 0; k < n; k++) v[k] = sample_quantity(q, f[k], &J[k * kP]);
            pair_sums[(size_t)p * kQ + q] = tree_sum(v);
        }
    }
    fs.assign((size_t)P.N * kQ, 0.0);
    for (int f = 0; f < P.N; f++)
        for (int q = 0; q < kQ; q++) fs[(size_t)f * kQ + q] = frame_sum(pair_sums.data(), P.pairs->data(), npairs, f, q);
    return true;
}

}  // namespace

extern "C" {

// choose the evaluation behind the restatement; use_strided: call <prefix>align_frame_eval_strided when present
int oracle_falign_bind(const char* lib_path, const char* prefix, int use_strided) {
    void* h = dlopen(lib_path, RTLD_NOW | RTLD_LOCAL);
    if (!h) {
        printf("oracle falign: dlopen(%s) failed: %s\n", lib_path, dlerror());
        return -1;
    }
    const std::string p = prefix;
    Eval e;
    e.init = (fn_init)dlsym(h, (p + "align_frame_init_gpu").c_str());
    e.full = (fn_eval)dlsym(h, (p + "align_frame_eval_gpu").c_str());
    e.strided = use_strided ? (fn_strided)dlsym(h, (p + "align_frame_eval_strided").c_str()) : nullptr;
    if (!e.init || !e.full) return -1;
    g_eval = e;
    return 0;
}

// falign restated over the bound evaluation; same arguments and outputs as vb_py_falign_wrapper_ex (no samples)
int oracle_falign(const float* depths, const float* images, const float* weights, const float* poses_init,
                  float* poses_ret, const int* connectivity, int n_connectivity, float* poses_covar,
                  float* scaling_factor, float* visibility_mat, float* consistency_mat, int N, int w, int h, float fx,
                  float fy, float cx, float cy, float vbf, float crw, int optimize_7dof, int stride, float bound,
                  int* iters_run, int* reason, double* costs, float* stats) {
    auto t0 = std::chrono::steady_clock::now();
    std::vector<int> pairs;
    if (!g_eval.init || N < 2 || N > kMaxFrames || stride < 1 || !parse_pairs(connectivity, n_connectivity, N, pairs))
        return -1;
    const int npairs = (int)pairs.size() / 3;
    const bool photo = images != nullptr && crw > 0;
    const size_t npx = (size_t)w * h;
    std::vector<float*> d(N), im(N), wt(N);
    std::vector<float> ones(npx, 1.f);
    for (int i = 0; i < N; i++) {
        d[i] = (float*)depths + i * npx;
        im[i] = photo ? (float*)images + i * npx : nullptr;
        wt[i] = weights ? (float*)weights + i * npx : ones.data();
    }
    float K[9] = {fx, 0, cx, 0, fy, cy, 0, 0, 1};
    if (g_eval.init(photo ? im.data() : nullptr, d.data(), wt.data(), K, vbf, crw, N, w, h) != 0) return -2;

    Problem P;
    P.N = N, P.w = w, P.h = h, P.stride = stride, P.pairs = &pairs;
    std::vector<int> is_ref(N, 0);
    for (int p = 0; p < npairs; p++) is_ref[pairs[p * 3]] = 1;
    std::unique_ptr<Lm> L(new Lm);
    lm_init(*L, N, optimize_7dof, photo, poses_init, is_ref.data());
    std::vector<double> fs;
    if (!normal_equations(P, L->x, L->x, true, fs)) return -2;
    lm_start(*L, fs.data());
    while (L->reason == kRunning) {
        if (!normal_equations(P, L->xc, L->x, true, fs)) return -2;
        lm_candidate(*L, fs.data());
    }
    auto t1 = std::chrono::steady_clock::now();

    // covariance: un-doubled Jacobian at the final state
    if (!normal_equations(P, L->x, L->x, false, fs)) return -2;
    finish(*L, fs.data(), optimize_7dof, poses_ret, poses_covar);
    for (int f = 0; f < N; f++) scaling_factor[f] = optimize_7dof ? (float)std::exp(L->x[f][6]) : 1.f;
    // scores: full resolution, unweighted
    for (int i = 0; i < N * N; i++) visibility_mat[i] = consistency_mat[i] = std::nanf("");
    std::vector<double> v0, v1;
    for (int p = 0; p < npairs; p++) {
        float pr[kP], pt[kP];
        params_float(L->x[pairs[p * 3]], pr);
        params_float(L->x[pairs[p * 3 + 1]], pt);
        if (!eval_pair(P, p, pr, pt, false, 1)) return -2;
        v0.resize(P.res.size()), v1.resize(P.res.size());
        for (size_t k = 0; k < P.res.size(); k++) {
            double q[2];
            score_quantities(P.res[k], (double)bound, q);
            v0[k] = q[0], v1[k] = q[1];
        }
        const double s[2] = {tree_sum(v0), tree_sum(v1)};
        const int at = pairs[p * 3] * N + pairs[p * 3 + 1];
        pair_scores(s, w, h, &visibility_mat[at], &consistency_mat[at]);
    }
    if (iters_run) *iters_run = L->iter;
    if (reason) *reason = L->reason;
    if (costs) costs[0] = L->cost0, costs[1] = L->cost;
    if (stats) {
        auto t2 = std::chrono::steady_clock::now();
        stats[0] = (float)std::chrono::duration<double, std::milli>(t2 - t0).count();
        stats[1] = 0;
        stats[2] = (float)std::chrono::duration<double, std::milli>(t1 - t0).count();
        stats[3] = (float)std::chrono::duration<double, std::milli>(t2 - t1).count();
    }
    return 0;
}

// the shared step header, for the GPU-less tests: one damped, Jacobi-scaled step of a single frame block and the
// trust-region rules.  H: 45 packed entries, g, D: 9 each, act: P indices.  out: delta[P], m, ok.
int oracle_falign_frame_step(const double* H, const double* g, const double* D, const int* act, int P, double radius,
                             double* delta, double* m) {
    std::unique_ptr<Lm> L(new Lm);
    L->N = 1, L->P = P;
    for (int i = 0; i < P; i++) L->act[i] = act[i];
    for (int t = 0; t < kTri; t++) L->H[0][t] = H[t];
    for (int j = 0; j < kP; j++) L->g[0][j] = g[j], L->D[0][j] = D[j];
    return frame_step(*L, 0, radius, delta, m) ? 1 : 0;
}

// one lm_candidate() from a given state: in[0..4] = cost, model_change, radius, decrease_factor, candidate cost;
// returns the reason; out[0..3] = radius, decrease_factor, accepted (0/1), iterations
int oracle_falign_lm_rules(const double* in, double* out) {
    std::unique_ptr<Lm> L(new Lm);
    const int is_ref[1] = {1};
    lm_init(*L, 1, 0, 0, nullptr, is_ref);
    for (int t = 0; t < kTri; t++) L->H[0][t] = 0;
    for (int j = 0; j < 6; j++) L->H[0][tri(j, j)] = 1.0, L->D[0][j] = 1.0, L->g[0][j] = 1.0, L->xc[0][j] = 0.5;
    L->cost = in[0], L->model_change = in[1], L->radius = in[2], L->decrease_factor = in[3];
    std::vector<double> fs(kQ, 0.0);
    fs[0] = 2.0 * in[4];
    for (int j = 0; j < 6; j++) fs[1 + j] = 1.0, fs[1 + kP + tri(j, j)] = 1.0;
    lm_candidate(*L, fs.data());
    out[0] = L->radius, out[1] = L->decrease_factor, out[2] = L->n_accepted, out[3] = L->iter;
    return L->reason;
}

}  // extern "C"
