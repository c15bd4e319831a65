// Frame alignment: the normal-equation summation tree and the restated Levenberg-Marquardt step, shared by the
// device solver (falign.cu) and its host restatement (oracle/host_falign.cpp).
//
// Every floating-point operation below is an individually rounded IEEE double operation (hm::det: *_rn intrinsics
// on the device, -ffp-contract=off on the host), so the device and the host produce the same bits from the same
// per-sample residuals and Jacobians.  DESIGN.md §9 states the contract; the points that rest on Ceres' documented
// behaviour rather than on the reference's own code are marked there.
#pragma once
#include <cmath>
#include <utility>
#include <vector>
#include "host_math.h"

namespace vb {
namespace fa {

constexpr int kP = 9;            // parameters per frame: rvec(3), t(3), log depth scale, colour scale, colour offset
constexpr int kTri = 45;         // unique entries of a 9x9 symmetric block
constexpr int kQ = 1 + kP + kTri;  // per-sample quantities: f^2, J_i f, J_i J_j (i <= j)
constexpr int kMaxFrames = 64;
constexpr int kBlock = 256;      // samples per reduction block: 8 warps of 32

// termination reasons (FalignInfo::reason)
enum Reason {
    kRunning = 0,
    kGradientTolerance = 1,
    kParameterTolerance = 2,
    kFunctionTolerance = 3,
    kMinTrustRegionRadius = 4,
    kMaxIterations = 5,
    kInvalidSteps = 6,
};

// Solver settings: the reference's (frame-alignment/align_frame.cpp:142-156) and Ceres' defaults for the rest.
constexpr int kMaxIters = 100;
constexpr double kInitialRadius = 1.0;
constexpr double kMaxRadius = 1e16;
constexpr double kMinRadius = 1e-32;
constexpr double kMinRelativeDecrease = 1e-3;
constexpr double kFunctionTol = 1e-6;
constexpr double kGradientTol = 1e-10;
constexpr double kParameterTol = 1e-8;
constexpr double kMinDiagonal = 1e-6;
constexpr double kMaxDiagonal = 1e32;
constexpr int kMaxInvalidSteps = 5;

// index of J_i J_j (i <= j) in the packed upper triangle
VB_HD inline int tri(int i, int j) { return i * kP - (i * (i - 1)) / 2 + (j - i); }

// ---- summation tree -----------------------------------------------------------------------------------------------
// The samples of a pair are cut into blocks of 256 consecutive samples (packed index (y/s)*ceil(w/s) + x/s); a
// missing sample contributes +0.  Inside a block each warp of 32 is summed by halving (a[i] += a[i + h] for
// h = 16, 8, 4, 2, 1), then the 8 warp sums by halving (h = 4, 2, 1).  The block sums of a pair are added in block
// order, starting from +0.  reduce_block() is the first two levels; the device does them with shuffles.
VB_HD inline double reduce_block(double* v /*[256], clobbered*/) {
    using namespace hm::det;
    for (int w = 0; w < 8; w++)
        for (int h = 16; h >= 1; h >>= 1)
            for (int i = 0; i < h; i++) v[w * 32 + i] = add(v[w * 32 + i], v[w * 32 + i + h]);
    double s[8];
    for (int w = 0; w < 8; w++) s[w] = v[w * 32];
    for (int h = 4; h >= 1; h >>= 1)
        for (int i = 0; i < h; i++) s[i] = add(s[i], s[i + h]);
    return s[0];
}

// quantity q of one sample with residual f and Jacobian J (already zeroed where f is not finite, already doubled
// for a bi-connected pair).  Products of two floats are exact in double.
VB_HD inline double sample_quantity(int q, float f, const float* J) {
    using namespace hm::det;
    if (q == 0) return mul((double)f, (double)f);
    if (q <= kP) return mul((double)J[q - 1], (double)f);
    int t = q - 1 - kP, i = 0;
    while (t >= kP - i) t -= kP - i, i++;
    return mul((double)J[i], (double)J[i + t]);
}

// ---- the solver state -----------------------------------------------------------------------------------------------
// One problem: N frames, the active parameter indices act[0..P) shared by every frame (pose, + scale with 7-DoF,
// + colour with photo consistency), and which frames own a parameter block (frames that are the ref of a pair).
struct Lm {
    int N, P, act[kP];
    int active[kMaxFrames];
    int iter, reason, n_invalid, n_accepted;
    double radius, decrease_factor, cost, cost0, model_change;
    double x[kMaxFrames][kP];   // accepted state (the "user state" every target reads)
    double xc[kMaxFrames][kP];  // point being evaluated (candidate)
    double g[kMaxFrames][kP];   // gradient J^T f at x
    double H[kMaxFrames][kTri]; // J^T J at x (upper triangle, full 9x9 layout)
    double D[kMaxFrames][kP];   // Jacobi scaling 1 / (1 + ||J_col||), from the first evaluation
};

VB_HD inline void lm_init(Lm& L, int N, int optimize_7dof, int photo, const float* poses_init /*[N][6] or null*/,
                          const int* is_ref /*[N]*/) {
    L.N = N, L.P = 0;
    for (int i = 0; i < 6; i++) L.act[L.P++] = i;
    if (optimize_7dof) L.act[L.P++] = 6;
    if (photo) L.act[L.P++] = 7, L.act[L.P++] = 8;
    for (int i = L.P; i < kP; i++) L.act[i] = -1;
    L.iter = 0, L.reason = kRunning, L.n_invalid = 0, L.n_accepted = 0;
    L.radius = kInitialRadius, L.decrease_factor = 2.0, L.cost = 0, L.cost0 = 0, L.model_change = 0;
    for (int f = 0; f < kMaxFrames; f++) {
        L.active[f] = f < N ? is_ref[f] : 0;
        for (int j = 0; j < kP; j++) {
            const double v = (f < N && poses_init && j < 6) ? (double)poses_init[f * 6 + j] : 0.0;
            L.x[f][j] = v, L.xc[f][j] = v, L.g[f][j] = 0, L.D[f][j] = 0;
        }
        for (int t = 0; t < kTri; t++) L.H[f][t] = 0;
    }
}

// float parameters handed to the per-pixel evaluation (frame-alignment/align_frame_cost_fun.h:129-152): inactive
// entries of the state stay 0, so all 9 are converted
VB_HD inline void params_float(const double* x9, float* p9) {
    for (int j = 0; j < kP; j++) p9[j] = (float)x9[j];
}

// frame f's sums: its pairs as ref, in connectivity order, starting from +0.  pairs: [npairs][3] = ref, tar, factor.
VB_HD inline double frame_sum(const double* pair_sums /*[npairs][kQ]*/, const int* pairs, int npairs, int f, int q) {
    double s = 0.0;
    for (int p = 0; p < npairs; p++)
        if (pairs[p * 3] == f) s = hm::det::add(s, pair_sums[p * kQ + q]);
    return s;
}

// score quantities of one full-resolution unweighted sample: finite count and 1 - min(r^2, b) / b
// (frame-alignment/align_frame_cost_fun.h:96-127)
VB_HD inline void score_quantities(float r, double bound, double* v /*[2]*/) {
    using namespace hm::det;
    if (!(fabs((double)r) < INFINITY)) {
        v[0] = 0.0, v[1] = 0.0;
        return;
    }
    double b2 = mul((double)r, (double)r);
    b2 = b2 < bound ? b2 : bound;
    v[0] = 1.0, v[1] = sub(1.0, div(b2, bound));
}

// visibility and consistency of a pair from its two score sums
VB_HD inline void pair_scores(const double* s /*[2]*/, int w, int h, float* vis, float* cons) {
    using namespace hm::det;
    *vis = (float)div(s[0], (double)w * (double)h);
    *cons = (float)div(s[1], s[0] > 1.0 ? s[0] : 1.0);
}

// cost = 1/2 sum f^2 over the frames (frame order)
VB_HD inline double total_cost(const Lm& L, const double* fs /*[N][kQ]*/) {
    using namespace hm::det;
    double s = 0.0;
    for (int f = 0; f < L.N; f++)
        if (L.active[f]) s = add(s, fs[f * kQ]);
    return mul(0.5, s);
}

// In-place Cholesky A = L L^T of an n x n row-major matrix (lower triangle written); false on a non-positive or
// non-finite pivot.  Inner sums run k = 0, 1, ... in order.
VB_HD inline bool cholesky(double* A, int n) {
    using namespace hm::det;
    for (int j = 0; j < n; j++) {
        double s = A[j * n + j];
        for (int k = 0; k < j; k++) s = sub(s, mul(A[j * n + k], A[j * n + k]));
        if (!(s > 0.0) || !(s < INFINITY)) return false;
        const double d = root(s);
        A[j * n + j] = d;
        for (int i = j + 1; i < n; i++) {
            double t = A[i * n + j];
            for (int k = 0; k < j; k++) t = sub(t, mul(A[i * n + k], A[j * n + k]));
            A[i * n + j] = div(t, d);
        }
    }
    return true;
}

// solve L L^T x = b in place (b -> x)
VB_HD inline void cholesky_solve(const double* Lc, int n, double* b) {
    using namespace hm::det;
    for (int i = 0; i < n; i++) {
        double t = b[i];
        for (int k = 0; k < i; k++) t = sub(t, mul(Lc[i * n + k], b[k]));
        b[i] = div(t, Lc[i * n + i]);
    }
    for (int i = n - 1; i >= 0; i--) {
        double t = b[i];
        for (int k = i + 1; k < n; k++) t = sub(t, mul(Lc[k * n + i], b[k]));
        b[i] = div(t, Lc[i * n + i]);
    }
}

// Damped, Jacobi-scaled step of one frame: (Hs + clamp(diag Hs)/radius) ds = -gs with Hs = D H D, gs = D g; the
// unscaled step D ds goes to delta.  m receives gs^T ds + 1/2 ds^T Hs ds.  False when the factorisation fails.
VB_HD inline bool frame_step(const Lm& L, int f, double radius, double* delta /*[kP]*/, double* m) {
    using namespace hm::det;
    const int P = L.P;
    double A[kP * kP], Hs[kP * kP], gs[kP], ds[kP];
    for (int i = 0; i < P; i++) {
        const int ai = L.act[i];
        gs[i] = mul(L.D[f][ai], L.g[f][ai]);
        for (int j = 0; j < P; j++) {
            const int aj = L.act[j];
            const double h = L.H[f][ai <= aj ? tri(ai, aj) : tri(aj, ai)];
            Hs[i * P + j] = mul(mul(L.D[f][ai], h), L.D[f][aj]);
            A[i * P + j] = Hs[i * P + j];
        }
    }
    for (int i = 0; i < P; i++) {
        double d = Hs[i * P + i];
        d = d < kMinDiagonal ? kMinDiagonal : (d > kMaxDiagonal ? kMaxDiagonal : d);
        A[i * P + i] = add(A[i * P + i], div(d, radius));
    }
    if (!cholesky(A, P)) return false;
    for (int i = 0; i < P; i++) ds[i] = -gs[i];
    cholesky_solve(A, P, ds);
    double gd = 0.0, quad = 0.0;
    for (int i = 0; i < P; i++) {
        gd = add(gd, mul(gs[i], ds[i]));
        double r = 0.0;
        for (int j = 0; j < P; j++) r = add(r, mul(Hs[i * P + j], ds[j]));
        quad = add(quad, mul(ds[i], r));
    }
    *m = add(gd, mul(0.5, quad));
    for (int i = 0; i < P; i++) delta[i] = mul(L.D[f][L.act[i]], ds[i]);
    return true;
}

// max |x - (x - g)| over the parameters of the problem (Ceres' projected gradient norm for a Euclidean space)
VB_HD inline double gradient_max_norm(const Lm& L) {
    using namespace hm::det;
    double m = 0.0;
    for (int f = 0; f < L.N; f++)
        if (L.active[f])
            for (int i = 0; i < L.P; i++) {
                const int a = L.act[i];
                const double v = fabs(sub(L.x[f][a], sub(L.x[f][a], L.g[f][a])));
                m = v > m ? v : m;
            }
    return m;
}

// The iteration-end checks of Ceres' trust-region loop, in its order: iteration limit, gradient tolerance,
// minimum radius.  Returns true when the solve goes on.
VB_HD inline bool can_continue(Lm& L) {
    if (L.iter >= kMaxIters) return L.reason = kMaxIterations, false;
    if (gradient_max_norm(L) <= kGradientTol) return L.reason = kGradientTolerance, false;
    if (L.radius <= kMinRadius) return L.reason = kMinTrustRegionRadius, false;
    return true;
}

// Compute steps until one is valid (then xc = x + delta and the parameter tolerance is tested) or the solve ends.
VB_HD inline void next_candidate(Lm& L) {
    using namespace hm::det;
    while (true) {
        bool ok = true;
        double msum = 0.0, delta[kMaxFrames][kP];
        for (int f = 0; f < L.N && ok; f++) {
            if (!L.active[f]) continue;
            double m;
            ok = frame_step(L, f, L.radius, delta[f], &m);
            msum = add(msum, m);
        }
        const double model_change = -msum;
        if (!ok || !(model_change > 0.0) || !(model_change < INFINITY)) {  // invalid step
            if (++L.n_invalid >= kMaxInvalidSteps) {
                L.reason = kInvalidSteps;
                return;
            }
            L.radius = div(L.radius, L.decrease_factor);
            L.decrease_factor = mul(L.decrease_factor, 2.0);
            L.iter++;
            if (!can_continue(L)) return;
            continue;
        }
        L.n_invalid = 0;
        L.model_change = model_change;
        double xn = 0.0, sn = 0.0;
        for (int f = 0; f < L.N; f++) {
            for (int j = 0; j < kP; j++) L.xc[f][j] = L.x[f][j];
            if (!L.active[f]) continue;
            for (int i = 0; i < L.P; i++) {
                const int a = L.act[i];
                L.xc[f][a] = add(L.x[f][a], delta[f][i]);
                const double d = sub(L.x[f][a], L.xc[f][a]);
                xn = add(xn, mul(L.x[f][a], L.x[f][a]));
                sn = add(sn, mul(d, d));
            }
        }
        if (root(sn) <= mul(kParameterTol, add(root(xn), kParameterTol))) L.reason = kParameterTolerance;
        return;
    }
}

// take the sums fs (one evaluation's frame sums) as the normal equations at x
VB_HD inline void take_normal_equations(Lm& L, const double* fs) {
    for (int f = 0; f < L.N; f++) {
        for (int j = 0; j < kP; j++) L.g[f][j] = fs[f * kQ + 1 + j];
        for (int t = 0; t < kTri; t++) L.H[f][t] = fs[f * kQ + 1 + kP + t];
    }
}

// Iteration zero: fs = sums of the evaluation at x (ref and target both x).  Sets the Jacobi scaling, then either
// ends the solve or leaves the first candidate in xc.
VB_HD inline void lm_start(Lm& L, const double* fs) {
    using namespace hm::det;
    take_normal_equations(L, fs);
    L.cost = L.cost0 = total_cost(L, fs);
    for (int f = 0; f < L.N; f++)
        for (int j = 0; j < kP; j++) L.D[f][j] = div(1.0, add(1.0, root(L.H[f][tri(j, j)])));
    if (!can_continue(L)) return;
    next_candidate(L);
}

// One iteration after the candidate xc was evaluated (ref = xc, target = x): fs = its sums.  Function tolerance,
// step quality, accept (x = xc, the same sums become the normal equations at the new x: the target state lags one
// iteration, so they are exact) or reject, radius update, iteration-end checks, next candidate.
VB_HD inline void lm_candidate(Lm& L, const double* fs) {
    using namespace hm::det;
    const double cost_c = total_cost(L, fs);
    if (fabs(sub(L.cost, cost_c)) <= mul(kFunctionTol, L.cost)) {
        L.reason = kFunctionTolerance;
        return;
    }
    const double rho = div(sub(L.cost, cost_c), L.model_change);
    if (rho > kMinRelativeDecrease) {
        for (int f = 0; f < L.N; f++)
            for (int j = 0; j < kP; j++) L.x[f][j] = L.xc[f][j];
        L.cost = cost_c;
        take_normal_equations(L, fs);
        const double t = sub(mul(2.0, rho), 1.0);
        double shrink = sub(1.0, mul(mul(t, t), t));
        shrink = shrink > 1.0 / 3.0 ? shrink : 1.0 / 3.0;
        L.radius = div(L.radius, shrink);
        L.radius = L.radius < kMaxRadius ? L.radius : kMaxRadius;
        L.decrease_factor = 2.0;
        L.n_accepted++;
    } else {
        L.radius = div(L.radius, L.decrease_factor);
        L.decrease_factor = mul(L.decrease_factor, 2.0);
    }
    L.iter++;
    if (!can_continue(L)) return;
    next_candidate(L);
}

// Covariance of frame f: inverse of its whole active block (un-doubled J^T J at the final state).  cov receives the
// P x P inverse (row-major).  False when the block is not positive definite.
VB_HD inline bool block_inverse(const double* H /*[kTri]*/, const int* act, int P, double* cov /*[P*P]*/) {
    double A[kP * kP];
    for (int i = 0; i < P; i++)
        for (int j = 0; j < P; j++) {
            const int ai = act[i], aj = act[j];
            A[i * P + j] = H[ai <= aj ? tri(ai, aj) : tri(aj, ai)];
        }
    if (!cholesky(A, P)) return false;
    for (int c = 0; c < P; c++) {
        double e[kP];
        for (int i = 0; i < P; i++) e[i] = i == c ? 1.0 : 0.0;
        cholesky_solve(A, P, e);
        for (int i = 0; i < P; i++) cov[i * P + c] = e[i];
    }
    return true;
}

// Output assembly shared by both sides: poses (N,6) and covariances (N,C,C) with C = 6 or 7, from the final state and
// the frame sums fs of the covariance evaluation.  A frame without a parameter block or a block that is not positive
// definite makes every covariance 0.  (The scaling factors exp(scale) are taken on the host by both sides.)
VB_HD inline void finish(const Lm& L, const double* fs, int optimize_7dof, float* poses, float* covar) {
    const int C = optimize_7dof ? 7 : 6;
    bool ok = true;
    for (int f = 0; f < L.N; f++) {
        for (int j = 0; j < 6; j++) poses[f * 6 + j] = (float)L.x[f][j];
        ok = ok && L.active[f];
    }
    for (int i = 0; i < L.N * C * C; i++) covar[i] = 0.f;
    for (int f = 0; f < L.N && ok; f++) {
        double cov[kP * kP];
        ok = block_inverse(fs + f * kQ + 1 + kP, L.act, L.P, cov);
        if (!ok) break;
        for (int i = 0; i < 6; i++)
            for (int j = 0; j < 6; j++) covar[(f * C + i) * C + j] = (float)cov[i * L.P + j];
        if (optimize_7dof) covar[(f * C + 6) * C + 6] = (float)cov[6 * L.P + 6];
    }
    if (!ok)
        for (int i = 0; i < L.N * C * C; i++) covar[i] = 0.f;
}

// Parses the connectivity list (pairs terminated by -1; n_ints = its length in ints, or < 0 when unknown).  Empty /
// NULL means every ordered pair ref != tar.  Returns false on an entry out of [0, N) or a missing terminator.
// pairs: [npairs][3] = ref, tar, Jacobian factor (2 when the reverse pair is also connected).  Host only.
inline bool parse_pairs(const int* conn, int n_ints, int N, std::vector<int>& pairs) {
    std::vector<std::pair<int, int>> cp;
    if (conn) {
        int i = 0;
        while (true) {
            if (n_ints >= 0 && i >= n_ints) return false;  // no terminator inside the array
            if (conn[i] == -1) break;
            if (n_ints >= 0 && i + 1 >= n_ints) return false;
            const int a = conn[i], b = conn[i + 1];
            if (a < 0 || a >= N || b < 0 || b >= N) return false;
            cp.push_back({a, b});
            i += 2;
        }
    }
    if (cp.empty())
        for (int r = 0; r < N; r++)
            for (int t = 0; t < N; t++)
                if (r != t) cp.push_back({r, t});
    pairs.clear();
    for (auto& c : cp) {
        bool bi = false;
        for (auto& d : cp) bi = bi || (d.first == c.second && d.second == c.first);
        pairs.push_back(c.first), pairs.push_back(c.second), pairs.push_back(bi ? 2 : 1);
    }
    return true;
}

}  // namespace fa
}  // namespace vb
