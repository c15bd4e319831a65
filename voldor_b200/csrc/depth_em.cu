// Depth M-step / rigidness E-step kernels for sm_100a.
//
// What the reference does (gpu-kernels/optimize_depth.cu:462-494, fb_smooth.h:72-107) in 26+ launches over
// texture-backed GMats, restructured for B200:
//   * forward-backward smoothing: row chains are walked from shared-memory tiles that are loaded/stored
//     fully coalesced (one warp = 32 rows, 32-column tiles, register prefetch of the next tile), both
//     directions of a pass run in one launch; column chains are naturally coalesced.
//   * cost map + all `n_rand_samples` random candidates are ONE kernel: depth, best cost and the XORWOW
//     state live in registers for the whole search; the reference reloads/stores the 48-byte curandState
//     and the cost map in each of its 1+10 launches (optimize_depth.cu:269-284,472-478).
//   * global propagation with step>1 has no intra-pass dependency (writes x≡1 mod step, reads x-1), so it
//     runs on (w/step)*h lanes instead of the reference's h (or w) threads (optimize_depth.cu:209-235).
//   * local propagation keeps its sequential 31-long chains (optimize_depth.cu:237-267).
// Candidate costs use explicitly rounded FP32 arithmetic in the reference's evaluation order
// (residual_model.cuh) because the argmin over candidates must reproduce the reference's decisions.
#include "depth_em.cuh"
#include "residual_model.cuh"
#include "geometry.cuh"
#include <cmath>
#include <curand_kernel.h>

namespace vb {

namespace {

constexpr unsigned long long kRandSeed = 233;  // reference: gpu-kernels/utils.h:18
constexpr float kMaximumDepth = 1e5f;          // reference: optimize_depth.cu:15

// Kernel-side view of the window state.
struct DepthView {
    int N, N_dp, w, h;
    int pitch;      // elements, for depth/cost/rig/rng planes
    size_t plane;   // pitch*h
    float abs_rf, basefocal, lambda, omega, delta, disp_delta, range_factor;
    cudaTextureObject_t flows_tex, dp_tex, dp_pconf_tex, dp_conf_tex;
    float* rig;
    float* depth;
    float* cost;
    uint32_t* rng;
    float* dp_conf;
    int dp_conf_pitch;      // elements
    size_t dp_conf_plane;   // elements per layer
};

// ------------------------------------------------------------------------------------------------
// The likelihood terms of hypothesising `depth` at a pixel (reference: optimize_depth.cu:84-138,140-198).
// Every kernel that evaluates a term goes through these helpers, so the rounding order is written down once.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool in_image(const DepthView& A, float x, float y) {
    return x >= 0 && x < (float)A.w && y >= 0 && y < (float)A.h;
}

// The chain of flow frames: the candidate's point is moved from frame to frame, and frame f fetches its observed flow
// where the last frame that took part projected the point (the pixel itself before any did).
struct FlowChain {
    float ox, oy, oz;  // the point in the camera of the last frame stepped to
    float px1, py1;    // fetch position of the next frame
};
__device__ __forceinline__ FlowChain flow_chain(const CamBlock& C, float fpx, float fpy, float depth) {
    FlowChain ch;
    backproject(C, fpx, fpy, depth, ch.ox, ch.oy, ch.oz);
    ch.px1 = fpx, ch.py1 = fpy;
    return ch;
}
// Steps the chain to frame f and projects the point to (px2, py2).  Frame f takes part when the point lies in front of
// its camera and its fetch position (fx, fy) is inside the image; its rigid flow is then (px2 - fx, py2 - fy).  Only a
// frame that takes part moves the fetch position on, so a later frame can fetch at a stale one (SURVEY §9 Q6).
__device__ __forceinline__ bool flow_step(const DepthView& A, const CamBlock& C, int f, FlowChain& ch, float& fx,
                                          float& fy, float& px2, float& py2) {
    rigid_move(C.R[f], C.t[f], ch.ox, ch.oy, ch.oz);
    project(C, ch.ox, ch.oy, ch.oz, px2, py2);
    fx = ch.px1, fy = ch.py1;
    if (!(ch.oz > 0 && in_image(A, fx, fy))) return false;
    ch.px1 = px2, ch.py1 = py2;
    return true;
}

// Depth prior p seen from the candidate: out of view when the point lies behind the prior's camera or projects outside
// the image, no depth where the prior holds none, else the term takes part with weight `wgt` and posterior `r`.
// Callers that need only one of the two leave the other to dead-code elimination.
enum PriorSight { kPriorOutOfView, kPriorNoDepth, kPriorTakesPart };
__device__ __forceinline__ PriorSight prior_term(const DepthView& A, const CamBlock& C, const PriorCamBlock& PC, int p,
                                                 float fpx, float fpy, float depth, float& wgt, float& r) {
    float ox, oy, oz, ux, uy;
    backproject(C, fpx, fpy, depth, ox, oy, oz);
    rigid_move(PC.R[p], PC.t[p], ox, oy, oz);
    project(C, ox, oy, oz, ux, uy);
    if (!(oz > 0 && in_image(A, ux, uy))) return kPriorOutOfView;
    const float target_depth = fetch_stack<float>(A.dp_tex, ux, uy, p, A.h);
    const float target_pconf = fetch_stack<float>(A.dp_pconf_tex, ux, uy, p, A.h);
    const float target_conf = fetch_stack<float>(A.dp_conf_tex, ux, uy, p, A.h);
    if (!(target_depth > 0)) return kPriorNoDepth;
    // prior 0 is the disparity prior when the caller passes disp_delta > 0 (SURVEY §9 Q21)
    const float scale = (A.disp_delta > 0 && p == 0) ? A.disp_delta : A.delta;
    wgt = f_mul(f_mul(target_pconf, target_conf), scale);
    r = depth_rigidness(oz, target_depth, A.basefocal, A.omega, A.abs_rf);
    return kPriorTakesPart;
}

// The cost of a candidate: the weighted mean of -log r over the terms that take part, summed in term order
// (flows f = 0..N-1, then priors 0..N_dp-1); INF when none does.
struct CostSum {
    float cost = 0.f, weight = 0.f;
    __device__ __forceinline__ void add(float wgt, float log_r) {
        cost = f_fma(-wgt, log_r, cost);
        weight = f_add(weight, wgt);
    }
    __device__ __forceinline__ float value() const {
        return weight == 0 ? INFINITY : f_div(cost, fmaxf(weight, FLT_EPSILON));
    }
};

// cost of hypothesising `depth` at pixel (px,py)   (reference: optimize_depth.cu:140-198)
__device__ float pixel_cost(const DepthView& A, const CamBlock& C, const PriorCamBlock& PC, int px, int py,
                            float depth) {
    const float fpx = (float)px, fpy = (float)py;
    const float* wgt_ptr = A.rig + (size_t)py * A.pitch + px;
    CostSum sum;
    FlowChain ch = flow_chain(C, fpx, fpy, depth);
    for (int f = 0; f < A.N; f++) {
        float fx, fy, px2, py2;
        if (flow_step(A, C, f, ch, fx, fy, px2, py2)) {
            const float2 obs = fetch_stack<float2>(A.flows_tex, fx, fy, f, A.h);
            const float r = flow_rigidness(f_sub(px2, fx), f_sub(py2, fy), obs.x, obs.y, A.lambda, A.abs_rf);
            sum.add(wgt_ptr[(size_t)f * A.plane], logf(r));
        }
    }
    for (int p = 0; p < A.N_dp; p++) {
        float wgt, r;
        if (prior_term(A, C, PC, p, fpx, fpy, depth, wgt, r) == kPriorTakesPart) sum.add(wgt, logf(r));
    }
    return sum.value();
}

__device__ __forceinline__ void try_candidate(const DepthView& A, const CamBlock& C, const PriorCamBlock& PC, int x,
                                              int y, float cand) {
    const size_t idx = (size_t)y * A.pitch + x;
    // a candidate equal to the pixel's own depth reproduces cost[idx] exactly and the strict '<' rejects it
    if (__float_as_uint(A.depth[idx]) == __float_as_uint(cand)) return;
    const float c = pixel_cost(A, C, PC, x, y, cand);
    if (c < A.cost[idx]) {  // strict '<' (reference: optimize_depth.cu:201-207)
        A.depth[idx] = cand;
        A.cost[idx] = c;
    }
}

// ------------------------------------------------------------------------------------------------
// XORWOW (Marsaglia) stream per pixel, bit-compatible with cuRAND's curand_init(seed, subsequence, 0):
// state words are produced by curand_init itself, the step below is the published recurrence
// (x ^= x>>2; ... ; d += 362437) and the uniform mapping is cuRAND's (0,1] = u32*2^-32 + 2^-33.
// ------------------------------------------------------------------------------------------------
struct Xorwow {
    uint32_t d, v0, v1, v2, v3, v4;
};
__device__ __forceinline__ float xorwow_uniform(Xorwow& s) {
    const uint32_t t = s.v0 ^ (s.v0 >> 2);
    s.v0 = s.v1, s.v1 = s.v2, s.v2 = s.v3, s.v3 = s.v4;
    s.v4 = (s.v4 ^ (s.v4 << 4)) ^ (t ^ (t << 1));
    s.d += 362437u;
    const uint32_t r = s.v4 + s.d;
    return f_fma((float)r, 2.3283064365386963e-10f, 2.3283064365386963e-10f / 2.0f);
}

__global__ void k_seed_rng(uint32_t* rng, int w, int h, int pitch, size_t plane) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    curandStateXORWOW_t st;
    curand_init(kRandSeed, (unsigned long long)(y * w + x), 0, &st);  // reference: optimize_depth.cu:286-291
    const size_t idx = (size_t)y * pitch + x;
    rng[idx] = st.d;
    rng[idx + plane] = st.v[0];
    rng[idx + 2 * plane] = st.v[1];
    rng[idx + 3 * plane] = st.v[2];
    rng[idx + 4 * plane] = st.v[3];
    rng[idx + 5 * plane] = st.v[4];
}

// ------------------------------------------------------------------------------------------------
// fused: cost of the current depth + n_rand random candidates   (reference: optimize_depth.cu:269-284)
// with EXACT early rejection of hopeless candidates, as a per-lane state machine.
//
// A candidate is kept only if its cost S/W is strictly below the pixel's best cost.  Every likelihood term
// -w*log(r) is >= 0 (w >= 0, r in [0,1]) and the weights are known before the candidate is evaluated, so after any
// prefix of the terms  S_k / W_ub  is a lower bound of the final cost, W_ub being the in-order sum of ALL weights the
// candidate could collect.  Floating-point addition, fma with a non-negative product and division are monotone, so
// the bound also holds for the rounded quantities: once  S_k >= round_up(best * max(W_ub, eps))  the reference's own
// comparison `cost < best` is certain to fail and the remaining terms need not be evaluated.  No decision changes
// (bit-identical depth / cost / RNG state); a pixel with a negative or NaN weight, a NaN best cost or the evaluation of
// the current depth itself are never pruned.  On the benchmark windows a random candidate survives 2.1 of its 8 terms
// on average (68 % are rejected by the first one).  Without any term every cost is INF: the current depth stays, no
// draw is accepted (INF < INF fails, and reject_at is INF) and the stream still advances n_rand draws.
//
// Lanes would leave candidates at different frames, so each lane runs its own (candidate, frame) state machine and
// every pass of the loop evaluates ONE term per lane: a lane that rejects early moves straight on to its next
// candidate while its neighbours continue theirs; the warp leaves the loop when its slowest lane has consumed its
// 1 + n_rand candidates.  The camera blocks are staged in shared memory because the frame index is per lane.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
    k_cost_and_random_search_pruned(const DepthView A, const __grid_constant__ CamBlock Cg,
                                    const __grid_constant__ PriorCamBlock PCg, int n_rand) {
    __shared__ CamBlock C;
    __shared__ PriorCamBlock PC;
    {
        const int tid = threadIdx.y * blockDim.x + threadIdx.x, nthr = blockDim.x * blockDim.y;
        for (int k = tid; k < (int)(sizeof(CamBlock) / sizeof(float)); k += nthr)
            reinterpret_cast<float*>(&C)[k] = reinterpret_cast<const float*>(&Cg)[k];
        if (A.N_dp > 0)
            for (int k = tid; k < (int)(sizeof(PriorCamBlock) / sizeof(float)); k += nthr)
                reinterpret_cast<float*>(&PC)[k] = reinterpret_cast<const float*>(&PCg)[k];
    }
    __syncthreads();
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= A.w || y >= A.h) return;
    const size_t idx = (size_t)y * A.pitch + x;
    const float fpx = (float)x, fpy = (float)y;

    Xorwow s = {0, 0, 0, 0, 0, 0};
    if (n_rand > 0) {
        s.d = A.rng[idx];
        s.v0 = A.rng[idx + A.plane];
        s.v1 = A.rng[idx + 2 * A.plane];
        s.v2 = A.rng[idx + 3 * A.plane];
        s.v3 = A.rng[idx + 4 * A.plane];
        s.v4 = A.rng[idx + 5 * A.plane];
    }
    float best_depth = A.depth[idx];
    float best_cost = 0.f;
    // frame 0 always fetches at the pixel itself: its observed flow and Fisk model are the same for every candidate
    float2 obs0 = make_float2(0.f, 0.f);
    ObservedFlowModel m0;
    m0.k.c = m0.k.s = m0.mu = 0.f;
    if (A.N > 0) {
        obs0 = fetch_stack<float2>(A.flows_tex, fpx, fpy, 0, A.h);
        m0 = observed_flow_model(obs0.x, obs0.y, A.lambda, A.abs_rf);
    }
    // everything the flow terms of ANY candidate of this pixel can add to the weight sum, summed in term order
    const float* wgt_ptr = A.rig + idx;
    float w_flows = 0.f;
    bool weights_ok = true;
    for (int f = 0; f < A.N; f++) {
        const float wgt = wgt_ptr[(size_t)f * A.plane];
        w_flows = f_add(w_flows, wgt);
        weights_ok = weights_ok && (wgt >= 0.f);
    }
    const int n_terms = A.N + A.N_dp;

    int it = -1, f = 0;
    float cand = best_depth, reject_at = 0.f;
    FlowChain ch = {0.f, 0.f, 0.f, fpx, fpy};
    CostSum sum;
    bool prune = false;
    while (true) {
        if (f == 0) {  // a new candidate: it == -1 is the current depth (never pruned), it >= 0 the random draws
            cand = best_depth;
            if (it >= 0) {
                const float u = xorwow_uniform(s);
                // d = 1/(range_factor*U + 1/MAXIMUM_DEPTH)   (reference: optimize_depth.cu:273)
                cand = __frcp_rn(f_fma(A.range_factor, u, 1.0f / kMaximumDepth));
            }
            ch = flow_chain(C, fpx, fpy, cand);
            sum = CostSum();
            prune = it >= 0 && weights_ok;
            if (prune) {
                float w_ub = w_flows;
                for (int p = 0; p < A.N_dp; p++) {  // the prior terms' weights depend on the candidate: look ahead
                    float wgt, r;
                    if (prior_term(A, C, PC, p, fpx, fpy, cand, wgt, r) == kPriorTakesPart) {
                        w_ub = f_add(w_ub, wgt);
                        prune = prune && (wgt >= 0.f);
                    }
                }
                reject_at = __fmul_ru(best_cost, fmaxf(w_ub, FLT_EPSILON));
            }
        }
        if (f < A.N) {  // likelihood term of flow f
            float fx, fy, px2, py2;
            if (flow_step(A, C, f, ch, fx, fy, px2, py2)) {
                float2 obs = obs0;
                ObservedFlowModel m = m0;
                if (f != 0) {
                    obs = fetch_stack<float2>(A.flows_tex, fx, fy, f, A.h);
                    m = observed_flow_model(obs.x, obs.y, A.lambda, A.abs_rf);
                }
                const float r = flow_rigidness_given(f_sub(px2, fx), f_sub(py2, fy), obs.x, obs.y, m, A.abs_rf);
                sum.add(wgt_ptr[(size_t)f * A.plane], logf(r));
            }
        } else if (f < n_terms) {  // likelihood term of prior f - N
            float wgt, r;
            if (prior_term(A, C, PC, f - A.N, fpx, fpy, cand, wgt, r) == kPriorTakesPart) sum.add(wgt, logf(r));
        }
        f++;
        const bool rejected = prune && sum.cost >= reject_at;
        if (f >= n_terms || rejected) {
            if (!rejected) {
                const float c = sum.value();
                if (it < 0 || c < best_cost) best_depth = cand, best_cost = c;
            }
            it++, f = 0;
            if (it >= n_rand) break;
        }
    }
    if (n_rand > 0) {
        A.rng[idx] = s.d;
        A.rng[idx + A.plane] = s.v0;
        A.rng[idx + 2 * A.plane] = s.v1;
        A.rng[idx + 3 * A.plane] = s.v2;
        A.rng[idx + 4 * A.plane] = s.v3;
        A.rng[idx + 5 * A.plane] = s.v4;
    }
    A.depth[idx] = best_depth;
    A.cost[idx] = best_cost;
}

// ------------------------------------------------------------------------------------------------
// global propagation, step > 1: every evaluation of one direction is independent
//   L2R: x = 1, 1+step, ...   takes depth(x-1)        R2L: x = w-2, w-2-step, ... takes depth(x+1)
//   T2B: y = 1, 1+step, ...   takes depth(y-1)        B2T: y = h-2, ...           takes depth(y+1)
// (reference: optimize_depth.cu:209-235)
// ------------------------------------------------------------------------------------------------
enum { DIR_L2R = 0, DIR_T2B = 1, DIR_R2L = 2, DIR_B2T = 3 };

template <int DIR>
__global__ void __launch_bounds__(128)
    k_global_propagation(const DepthView A, const __grid_constant__ CamBlock C,
                         const __grid_constant__ PriorCamBlock PC, int step) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;  // index along the strided axis
    const int o = blockIdx.y * blockDim.y + threadIdx.y;  // index along the other axis
    int x, y, sx, sy;
    if (DIR == DIR_L2R) {
        x = 1 + k * step, y = o, sx = x - 1, sy = y;
    } else if (DIR == DIR_R2L) {
        x = A.w - 2 - k * step, y = o, sx = x + 1, sy = y;
    } else if (DIR == DIR_T2B) {
        x = o, y = 1 + k * step, sx = x, sy = y - 1;
    } else {
        x = o, y = A.h - 2 - k * step, sx = x, sy = y + 1;
    }
    if (x < 0 || y < 0 || x >= A.w || y >= A.h) return;
    try_candidate(A, C, PC, x, y, A.depth[(size_t)sy * A.pitch + sx]);
}

// ------------------------------------------------------------------------------------------------
// Cooperative candidate cost: the N flow terms and N_dp prior terms of ONE candidate are evaluated by a group
// of G >= N + N_dp lanes (one term per lane: the texture fetch and the ~600-instruction Fisk posterior run in
// parallel), then combined in the reference's order f = 0..N-1, priors 0..N_dp-1 with the same fused multiply-adds, so
// the result is bit-identical to pixel_cost().  The fetch position of frame f depends on the in-view tests of all
// earlier frames (stale px1 rule, SURVEY §9 Q6): either every lane walks the whole pose chain for itself (SHARE =
// false, shortest dependent path — small launches), or the lanes share the projections and settle the rule with two
// ballots (SHARE = true, a fifth fewer instructions — launches that fill the GPU; see launch_local_group).
// The result is returned on every lane of the group.
// ------------------------------------------------------------------------------------------------
template <int G, bool SHARE>
__device__ __forceinline__ float pixel_cost_group(const DepthView& A, const CamBlock& C, const PriorCamBlock& PC,
                                                  int px, int py, float depth, int gl, unsigned gmask, int gbase) {
    // lane gl owns term gl: terms 0..N-1 are flows, N..N+N_dp-1 priors
    const float fpx = (float)px, fpy = (float)py;
    float fx = 0.f, fy = 0.f, px2 = 0.f, py2 = 0.f;
    bool valid = false;
    float my_w = 0.f, my_log = 0.f;
    if constexpr (SHARE) {
        // Every lane still walks the rigid moves (frame f's camera-space point is a running product), but only lane f
        // projects frame f — the two IEEE divisions and the in-view tests of a frame are done once per group instead
        // of once per lane.  Which frames take part and where each one fetches from (the position of the last earlier
        // frame that took part, or the pixel itself) follows from two group-wide bit masks: Z_f = "point in front of
        // camera f", P_f = "projection of frame f inside the image".
        float ox, oy, oz, mx = 0.f, my = 0.f, mz = 0.f;
        backproject(C, fpx, fpy, depth, ox, oy, oz);
        for (int f = 0; f < A.N; f++) {
            rigid_move(C.R[f], C.t[f], ox, oy, oz);
            if (f == gl) mx = ox, my = oy, mz = oz;
        }
        bool in_front = false, inside = false;
        if (gl < A.N) {
            project(C, mx, my, mz, px2, py2);
            in_front = mz > 0;
            inside = in_image(A, px2, py2);
        }
        const unsigned zb = __ballot_sync(gmask, in_front) >> gbase;
        const unsigned pb = __ballot_sync(gmask, inside) >> gbase;
        const unsigned all = (A.N >= 32) ? 0xffffffffu : ((1u << A.N) - 1u);
        int src = gl - 1;  // frame whose projected position this lane's frame fetches at; -1 = the pixel itself
        valid = gl < A.N;
        if ((zb & pb & all) != all) {
            // some frame drops out: replay the reference's sequential rule (stale px1, SURVEY §9 Q6) on the masks
            bool at_inside = true;  // the pixel itself lies inside the image
            int last = -1;
            valid = false;
            for (int f = 0; f < A.N; f++) {
                const bool v = ((zb >> f) & 1u) && at_inside;
                if (f == gl) valid = v, src = last;
                if (v) last = f, at_inside = (pb >> f) & 1u;
            }
        }
        const float sx = __shfl_sync(gmask, px2, gbase + max(src, 0));
        const float sy = __shfl_sync(gmask, py2, gbase + max(src, 0));
        fx = src < 0 ? fpx : sx, fy = src < 0 ? fpy : sy;
    } else {
        FlowChain ch = flow_chain(C, fpx, fpy, depth);
        for (int f = 0; f < A.N; f++) {
            float sfx, sfy, spx2, spy2;
            if (flow_step(A, C, f, ch, sfx, sfy, spx2, spy2) && f == gl)
                fx = sfx, fy = sfy, px2 = spx2, py2 = spy2, valid = true;
        }
    }
    if (valid) {
        const float2 obs = fetch_stack<float2>(A.flows_tex, fx, fy, gl, A.h);
        my_w = A.rig[(size_t)gl * A.plane + (size_t)py * A.pitch + px];
        my_log = logf(flow_rigidness(f_sub(px2, fx), f_sub(py2, fy), obs.x, obs.y, A.lambda, A.abs_rf));
    }
    const int pf = gl - A.N;
    if (pf >= 0 && pf < A.N_dp) {
        float wgt, r;
        if (prior_term(A, C, PC, pf, fpx, fpy, depth, wgt, r) == kPriorTakesPart)
            my_w = wgt, my_log = logf(r), valid = true;
    }
    CostSum sum;
    const unsigned taking_part = __ballot_sync(gmask, valid) >> gbase;
    for (int k = 0; k < A.N + A.N_dp && k < G; k++) {
        const float w = __shfl_sync(gmask, my_w, gbase + k);
        const float lg = __shfl_sync(gmask, my_log, gbase + k);
        if ((taking_part >> k) & 1u) sum.add(w, lg);
    }
    return sum.value();
}

// ------------------------------------------------------------------------------------------------
// local propagation: sequential chain inside each `width`-pixel segment (reference: optimize_depth.cu:237-267),
// with G lanes per chain: block = 128 threads = 128/G chains.  chain index c -> (o, seg) with o fastest, o = index
// along the other axis.  Also serves global propagation with step == 1 (one segment = the whole row/column).
// ------------------------------------------------------------------------------------------------
template <int DIR, int G, bool SHARE>
__global__ void __launch_bounds__(128)
    k_local_propagation_group(const DepthView A, const __grid_constant__ CamBlock C,
                              const __grid_constant__ PriorCamBlock PC, int width, int n_other, int n_seg) {
    const int lane = threadIdx.x & 31;
    const int gl = lane % G;
    const int gbase = lane - gl;
    const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << gbase);
    const int chain = (blockIdx.x * 128 + threadIdx.x) / G;
    if (chain >= n_other * n_seg) return;
    const int o = chain % n_other, seg = chain / n_other;
    const bool rowdir = (DIR == DIR_L2R || DIR == DIR_R2L);
    const int len = rowdir ? A.w : A.h;
    const int p0 = seg * width;
    int first, last, step;  // positions visited along the axis, inclusive
    if (DIR == DIR_L2R || DIR == DIR_T2B) {
        first = max(1, p0 + 1), last = min(len, p0 + width) - 1, step = 1;
    } else {
        first = min(len - 2, p0 + width - 2), last = max(0, p0), step = -1;
    }
    const int count = (last - first) * step + 1;
    if (count <= 0) return;
    // the candidate for position p is the (possibly just updated) depth of position p - step
    int sx = rowdir ? first - step : o, sy = rowdir ? o : first - step;
    float cand = A.depth[(size_t)sy * A.pitch + sx];
    int i = 0, pos = first;
    while (true) {
        // A position that already holds the candidate's depth (bit for bit) cannot accept it: the candidate's cost is
        // the very number stored in cost[] (same function of the same depth, weights and poses within this depth
        // step), the comparison is strict, and the candidate handed on is unchanged.  About 44 % of the propagation
        // candidates are such copies, so they are stepped over without evaluating the likelihood terms.  The chains
        // of a warp run through this loop independently and meet again for the next evaluation.
        while (i < count) {
            const int x = rowdir ? pos : o, y = rowdir ? o : pos;
            if (__float_as_uint(A.depth[(size_t)y * A.pitch + x]) != __float_as_uint(cand)) break;
            i++, pos += step;
        }
        if (i >= count) break;
        const int x = rowdir ? pos : o, y = rowdir ? o : pos;
        const size_t idx = (size_t)y * A.pitch + x;
        const float c = pixel_cost_group<G, SHARE>(A, C, PC, x, y, cand, gl, gmask, gbase);
        const float cur_cost = A.cost[idx];
        if (c < cur_cost) {
            if (gl == 0) A.depth[idx] = cand, A.cost[idx] = c;
            // cand stays: it is now this pixel's depth
        } else {
            cand = A.depth[idx];
        }
        i++, pos += step;
    }
}

// ------------------------------------------------------------------------------------------------
// E-step: rigidness of every flow and confidence of every prior at the current depth
// (reference: optimize_depth.cu:84-138)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
    k_update_rigidness(const DepthView A, const __grid_constant__ CamBlock C,
                       const __grid_constant__ PriorCamBlock PC) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= A.w || y >= A.h) return;
    const size_t idx = (size_t)y * A.pitch + x;
    const float fpx = (float)x, fpy = (float)y;
    const float depth = A.depth[idx];

    FlowChain ch = flow_chain(C, fpx, fpy, depth);
    for (int f = 0; f < A.N; f++) {
        float fx, fy, px2, py2;
        float r = 0.f;
        if (flow_step(A, C, f, ch, fx, fy, px2, py2)) {
            const float2 obs = fetch_stack<float2>(A.flows_tex, fx, fy, f, A.h);
            r = flow_rigidness(f_sub(px2, fx), f_sub(py2, fy), obs.x, obs.y, A.lambda, A.abs_rf);
        }
        A.rig[idx + (size_t)f * A.plane] = r;
    }

    for (int p = 0; p < A.N_dp; p++) {
        float* conf = A.dp_conf + (size_t)p * A.dp_conf_plane + (size_t)y * A.dp_conf_pitch + x;
        float wgt, r;
        const PriorSight sight = prior_term(A, C, PC, p, fpx, fpy, depth, wgt, r);
        // confidence is left untouched where the prior has no depth (SURVEY §9 Q19)
        if (sight == kPriorTakesPart)
            *conf = r;
        else if (sight == kPriorOutOfView)
            *conf = 0.f;
    }
}

// ------------------------------------------------------------------------------------------------
// forward-backward smoothing of a stack of probability maps (2-state HMM along rows, then columns)
// (reference: fb_smooth.h:29-69).  Rounding points follow the reference build.
// ------------------------------------------------------------------------------------------------
struct HmmConst {
    float nc, one_m_nc, s0e;
};
__device__ __forceinline__ float hmm_forward(float p, float e, const HmmConst& k) {
    const float om = f_sub(1.f, p);
    const float u0 = f_fma(k.one_m_nc, p, f_mul(k.nc, om));
    const float u1 = f_fma(k.nc, p, f_mul(k.one_m_nc, om));
    const float s1 = f_mul(u1, e);
    return f_div(s1, f_fma(k.s0e, u0, s1));
}
__device__ __forceinline__ float hmm_backward(float p, float e, const HmmConst& k) {
    const float pe = f_mul(p, e);
    const float om = f_sub(1.f, p);
    const float s0 = f_fma(k.s0e, f_mul(k.nc, om), f_mul(k.one_m_nc, pe));
    const float s1 = f_fma(k.s0e, f_mul(k.one_m_nc, om), f_mul(k.nc, pe));
    return f_div(s1, f_add(s0, s1));
}
__device__ __forceinline__ float hmm_posterior(float fwd, float bwd) {
    const float s1 = f_mul(bwd, fwd);
    return f_div(s1, f_fma(f_sub(1.f, fwd), f_sub(1.f, bwd), s1));
}

struct StackView {
    float* base;
    int pitch;      // elements
    size_t plane;   // elements
};

// rows: grid (ceil(h/32), layers, 2 directions), block 32.  Lane l owns row y0+l; 32x32 tiles are staged
// through shared memory so global traffic is 128-byte coalesced and the dependent chain reads smem.
__global__ void __launch_bounds__(32)
    k_fb_rows(StackView E, StackView F, StackView B, int w, int h, HmmConst k) {
    __shared__ float tin[32][33];
    __shared__ float tout[32][33];
    const int lane = threadIdx.x;
    const int y0 = blockIdx.x * 32;
    const int layer = blockIdx.y;
    const bool fwd = blockIdx.z == 0;
    const float* e = E.base + (size_t)layer * E.plane;
    float* out = (fwd ? F.base + (size_t)layer * F.plane : B.base + (size_t)layer * B.plane);
    const int out_pitch = fwd ? F.pitch : B.pitch;
    const int T = VB_DIV_CEIL(w, 32);
    const int rows = min(32, h - y0);
    const int y = y0 + lane;

    float nxt[32];
    {
        const int x0 = (fwd ? 0 : T - 1) * 32;
#pragma unroll
        for (int r = 0; r < 32; r++)
            nxt[r] = (r < rows && x0 + lane < w) ? e[(size_t)(y0 + r) * E.pitch + x0 + lane] : 0.f;
    }
    float p = 0.f;
    if (y < h) p = e[(size_t)y * E.pitch + (fwd ? 0 : w - 1)];

    for (int t = 0; t < T; t++) {
        const int x0 = (fwd ? t : T - 1 - t) * 32;
#pragma unroll
        for (int r = 0; r < 32; r++) tin[r][lane] = nxt[r];
        __syncwarp();
        if (t + 1 < T) {
            const int xn = (fwd ? t + 1 : T - 2 - t) * 32;
#pragma unroll
            for (int r = 0; r < 32; r++)
                nxt[r] = (r < rows && xn + lane < w) ? e[(size_t)(y0 + r) * E.pitch + xn + lane] : 0.f;
        }
        if (y < h) {
            const int cols = min(32, w - x0);
            if (fwd) {
                for (int i = 0; i < cols; i++) {
                    p = hmm_forward(p, tin[lane][i], k);
                    tout[lane][i] = p;
                }
            } else {
                for (int i = cols - 1; i >= 0; i--) {
                    p = hmm_backward(p, tin[lane][i], k);
                    tout[lane][i] = p;
                }
            }
        }
        __syncwarp();
        if (x0 + lane < w) {
            for (int r = 0; r < rows; r++) out[(size_t)(y0 + r) * out_pitch + x0 + lane] = tout[r][lane];
        }
        __syncwarp();
    }
}

// columns: thread per column, grid (ceil(w/128), layers, 2 directions)
__global__ void __launch_bounds__(128)
    k_fb_cols(StackView E, StackView F, StackView B, int w, int h, HmmConst k) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= w) return;
    const int layer = blockIdx.y;
    const bool fwd = blockIdx.z == 0;
    const float* __restrict__ e = E.base + (size_t)layer * E.plane + x;
    float* __restrict__ out = (fwd ? F.base + (size_t)layer * F.plane : B.base + (size_t)layer * B.plane) + x;
    const int out_pitch = fwd ? F.pitch : B.pitch;
    constexpr int U = 8;
    if (fwd) {
        float p = e[0];
        for (int y = 0; y < h; y += U) {
            float ev[U];
#pragma unroll
            for (int j = 0; j < U; j++) ev[j] = (y + j < h) ? e[(size_t)(y + j) * E.pitch] : 0.f;
#pragma unroll
            for (int j = 0; j < U; j++)
                if (y + j < h) {
                    p = hmm_forward(p, ev[j], k);
                    out[(size_t)(y + j) * out_pitch] = p;
                }
        }
    } else {
        float p = e[(size_t)(h - 1) * E.pitch];
        for (int y = h - 1; y >= 0; y -= U) {
            float ev[U];
#pragma unroll
            for (int j = 0; j < U; j++) ev[j] = (y - j >= 0) ? e[(size_t)(y - j) * E.pitch] : 0.f;
#pragma unroll
            for (int j = 0; j < U; j++)
                if (y - j >= 0) {
                    p = hmm_backward(p, ev[j], k);
                    out[(size_t)(y - j) * out_pitch] = p;
                }
        }
    }
}

__global__ void __launch_bounds__(256) k_fb_posterior(StackView E, StackView F, StackView B, int w, int h) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    const int layer = blockIdx.z;
    if (x >= w || y >= h) return;
    const float f = F.base[(size_t)layer * F.plane + (size_t)y * F.pitch + x];
    const float b = B.base[(size_t)layer * B.plane + (size_t)y * B.pitch + x];
    E.base[(size_t)layer * E.plane + (size_t)y * E.pitch + x] = hmm_posterior(f, b);
}

// E_in -> E_out (may alias: the reference smooths in place)
void fb_smooth_stack(StackView E_in, StackView E, StackView F, StackView B, int layers, int w, int h, float s0_ems_prob,
                     float no_change_prob, cudaStream_t s) {
    HmmConst k;
    k.nc = no_change_prob;
    k.one_m_nc = 1.f - no_change_prob;
    k.s0e = s0_ems_prob;
    const dim3 pb(32, 8), pg(VB_DIV_CEIL(w, 32), VB_DIV_CEIL(h, 8), layers);
    k_fb_rows<<<dim3(VB_DIV_CEIL(h, 32), layers, 2), 32, 0, s>>>(E_in, F, B, w, h, k);
    k_fb_posterior<<<pg, pb, 0, s>>>(E, F, B, w, h);
    k_fb_cols<<<dim3(VB_DIV_CEIL(w, 128), layers, 2), 128, 0, s>>>(E, F, B, w, h, k);
    k_fb_posterior<<<pg, pb, 0, s>>>(E, F, B, w, h);
}

// One lane per likelihood term of a candidate (see pixel_cost_group): a 31-long chain then costs ~1 term of latency per
// step instead of N + N_dp.  G is the smallest power of two >= max(N + N_dp, 1), so one warp always holds a group.
static_assert(kMaxFrames + kMaxPriorFrames <= 32, "the likelihood terms of a candidate must fit one warp");

template <int DIR, int G>
void launch_local_group(const DepthView& A, const CamBlock& C, const PriorCamBlock& PC, int width, int other,
                        int nseg, cudaStream_t s) {
    const long long threads = (long long)other * nseg * G;
    const unsigned blocks = (unsigned)VB_DIV_CEIL(threads, 128);
    // Sharing the projections of a candidate across the lanes of its group (pixel_cost_group) removes a fifth of the
    // instructions but lengthens the dependent path of one evaluation (projection -> ballot -> shuffle -> fetch instead
    // of projections overlapping the next rigid move).  Measured alone: 0.449 -> 0.401 ms at 16 warps per SM (640x480x8),
    // 0.307 -> 0.375 ms at 2 warps per SM (320x240x4).  A launch that cannot fill the GPU anyway keeps every lane
    // self-contained.
    static const int sms = [] {
        int dev = 0, n = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        return n;
    }();
    if (threads / 32 >= 8LL * sms)
        k_local_propagation_group<DIR, G, true><<<blocks, 128, 0, s>>>(A, C, PC, width, other, nseg);
    else
        k_local_propagation_group<DIR, G, false><<<blocks, 128, 0, s>>>(A, C, PC, width, other, nseg);
}

template <int DIR>
void launch_local(const DepthView& A, const CamBlock& C, const PriorCamBlock& PC, int width, cudaStream_t s) {
    const bool rowdir = (DIR == DIR_L2R || DIR == DIR_R2L);
    const int len = rowdir ? A.w : A.h, other = rowdir ? A.h : A.w;
    const int nseg = VB_DIV_CEIL(len, width);
    const int terms = A.N + A.N_dp;
    if (terms > 16)
        launch_local_group<DIR, 32>(A, C, PC, width, other, nseg, s);
    else if (terms > 8)
        launch_local_group<DIR, 16>(A, C, PC, width, other, nseg, s);
    else if (terms > 4)
        launch_local_group<DIR, 8>(A, C, PC, width, other, nseg, s);
    else if (terms > 2)
        launch_local_group<DIR, 4>(A, C, PC, width, other, nseg, s);
    else if (terms > 1)
        launch_local_group<DIR, 2>(A, C, PC, width, other, nseg, s);
    else
        launch_local_group<DIR, 1>(A, C, PC, width, other, nseg, s);
}

template <int DIR>
void launch_global(const DepthView& A, const CamBlock& C, const PriorCamBlock& PC, int step, cudaStream_t s) {
    const bool rowdir = (DIR == DIR_L2R || DIR == DIR_R2L);
    const int len = rowdir ? A.w : A.h, other = rowdir ? A.h : A.w;
    if (step == 1) {
        // a chain: local propagation with one segment spanning the whole axis
        launch_local<DIR>(A, C, PC, len, s);
        return;
    }
    const int n = (len - 2) / step + 1;  // number of evaluated positions along the axis (len >= 2)
    if (len < 2) return;
    if (rowdir)
        k_global_propagation<DIR><<<dim3(VB_DIV_CEIL(n, 8), VB_DIV_CEIL(other, 16)), dim3(8, 16), 0, s>>>(A, C, PC, step);
    else
        k_global_propagation<DIR><<<dim3(VB_DIV_CEIL(n, 4), VB_DIV_CEIL(other, 32)), dim3(4, 32), 0, s>>>(A, C, PC, step);
}

// Adds the duration of what issue() enqueues on stream s to (ms, count) when profiling is switched on.  Timing a
// region needs a sync, so it is only done then.
template <class Issue>
void timed(KernelProfile& prof, cudaStream_t s, double& ms, long long& count, Issue&& issue) {
    if (!prof.enabled) {
        issue();
        return;
    }
    if (!prof.ev0) cudaEventCreate(&prof.ev0), cudaEventCreate(&prof.ev1);
    cudaEventRecord(prof.ev0, s);
    issue();
    cudaEventRecord(prof.ev1, s);
    cudaEventSynchronize(prof.ev1);
    float t = 0;
    cudaEventElapsedTime(&t, prof.ev0, prof.ev1);
    ms += t, count++;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
int DepthEM::init_stream() {
    if (!stream) {
        VB_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        VB_CUDA(cudaStreamCreateWithFlags(&side, cudaStreamNonBlocking));
        VB_CUDA(cudaEventCreateWithFlags(&ev_rig_ready, cudaEventDisableTiming));
        VB_CUDA(cudaEventCreateWithFlags(&ev_smooth_done, cudaEventDisableTiming));
        cudaDeviceProp prop;
        int dev = 0;
        cudaGetDevice(&dev);
        if (cudaGetDeviceProperties(&prop, dev) == cudaSuccess) n_sm = prop.multiProcessorCount;
    }
    return 0;
}

void DepthEM::invalidate_smoothing() {
    if (smooth_layers > 0 && stream) cudaStreamWaitEvent(stream, ev_smooth_done, 0);
    smooth_layers = 0;
}

// Block height of the 1-thread-per-pixel search kernel: pick the shape whose grid fills the last wave best
// (tail balance on 148 SMs); resident blocks per SM come from the occupancy calculator.
static int pick_search_block_y(int w, int h, int n_sm) {
    static int per_sm[9] = {0};
    static std::mutex per_sm_mutex;  // contexts call this from different host threads
    std::lock_guard<std::mutex> lock(per_sm_mutex);
    const int cand[4] = {6, 5, 8, 4};
    int best = 8;
    double best_eff = -1;
    for (int by : cand) {
        if (!per_sm[by]) {
            int nb = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_cost_and_random_search_pruned, 32 * by, 0) !=
                    cudaSuccess ||
                nb < 1)
                nb = 1;
            per_sm[by] = nb;
        }
        const double waves = (double)(VB_DIV_CEIL(w, 32) * VB_DIV_CEIL(h, by)) / ((double)per_sm[by] * n_sm);
        const double eff = waves / ceil(waves);
        if (eff > best_eff + 1e-9) best_eff = eff, best = by;
    }
    return best;
}

int DepthEM::seed_rng() {
    const dim3 b(32, 8), g(VB_DIV_CEIL(w, 32), VB_DIV_CEIL(h, 8));
    k_seed_rng<<<g, b, 0, stream>>>(rng.ptr, w, h, rng.pitch, rng.layer_elems());
    VB_RETURN_IF_CUDA_ERROR();
    return 0;
}

int DepthEM::ensure(int w_, int h_, int N, int N_dp) {
    if (init_stream()) return (int)cudaErrorUnknown;
    invalidate_smoothing();  // the caller is about to (re)write the maps
    w = w_, h = h_;
    if (rng.ensure(w, h, 6, false)) {
        if (int e = seed_rng()) return e;
    }
    cost.ensure(w, h, 1, false);
    depth.ensure(w, h, 1, false);
    if (N > 0) {
        if (!shared_flows) flows.ensure(w, h, N, true);
        rig.ensure(w, h, N, true);
        rig_s.ensure(w, h, N, true);
    }
    if (N_dp > 0) {
        dp.ensure(w, h, N_dp, true);
        dp_pconf.ensure(w, h, N_dp, true);
        dp_conf.ensure(w, h, N_dp, true);
    }
    const int L = N > N_dp ? N : N_dp;
    if (L > 0) {
        fb_fwd.ensure(w, h, L, true);
        fb_bwd.ensure(w, h, L, true);
    }
    VB_RETURN_IF_CUDA_ERROR();
    return 0;
}

int DepthEM::run(int N, int N_dp, const DepthHyper& hp, bool update_rigidness_only) {
    DepthView A;
    A.N = N, A.N_dp = N_dp, A.w = w, A.h = h;
    A.pitch = depth.pitch, A.plane = depth.layer_elems();
    A.abs_rf = hp.abs_resize_factor, A.basefocal = hp.basefocal, A.lambda = hp.lambda, A.omega = hp.omega;
    A.delta = hp.delta, A.disp_delta = hp.disp_delta, A.range_factor = hp.range_factor;
    const TexStack<float2>& fl = shared_flows ? *shared_flows : flows;
    A.flows_tex = fl.tex;
    A.dp_tex = dp.tex, A.dp_pconf_tex = dp_pconf.tex, A.dp_conf_tex = dp_conf.tex;
    A.rig = rig.ptr, A.depth = depth.ptr, A.cost = cost.ptr, A.rng = rng.ptr;
    A.dp_conf = dp_conf.ptr;
    A.dp_conf_pitch = (int)(dp_conf.pitch / sizeof(float));
    A.dp_conf_plane = (size_t)A.dp_conf_pitch * h;

    KernelProfile none;  // counters of a context that does not profile
    KernelProfile& prof = this->prof ? *this->prof : none;
    cudaStream_t s = stream;
    const dim3 pb(32, 8), pg(VB_DIV_CEIL(w, 32), VB_DIV_CEIL(h, 8));

    // smoothing of the rigidness maps issued on the side stream at the end of the previous call (window pipeline)
    const bool pre_smoothed = smooth_layers >= N && smooth_layers > 0 && smooth_s0 == hp.s0_ems_prob &&
                              smooth_nc == hp.no_change_prob;
    if (smooth_layers > 0) cudaStreamWaitEvent(s, ev_smooth_done, 0);
    smooth_layers = 0;

    if (!update_rigidness_only) {
        if (hp.fb_smooth) {
            if (N > 0) {
                // out of place: the E-step below rewrites every rigidness value, so the smoothed maps are only ever
                // seen as the weights of this M-step (the reference smooths in place, fb_smooth.h:77-107)
                StackView E{rig.ptr, rig.pitch, rig.layer_elems()};
                StackView S{rig_s.ptr, rig_s.pitch, rig_s.layer_elems()};
                StackView F{fb_fwd.ptr, fb_fwd.pitch, fb_fwd.layer_elems()};
                StackView B{fb_bwd.ptr, fb_bwd.pitch, fb_bwd.layer_elems()};
                if (!pre_smoothed) fb_smooth_stack(E, S, F, B, N, w, h, hp.s0_ems_prob, hp.no_change_prob, s);
                A.rig = rig_s.ptr;
            }
            if (N_dp > 0) {
                // prior confidences stay in place: the E-step leaves them untouched where the prior has no depth,
                // so smoothed values can survive (SURVEY §9 Q19)
                StackView E{dp_conf.ptr, A.dp_conf_pitch, A.dp_conf_plane};
                StackView F{fb_fwd.ptr, fb_fwd.pitch, fb_fwd.layer_elems()};
                StackView B{fb_bwd.ptr, fb_bwd.pitch, fb_bwd.layer_elems()};
                fb_smooth_stack(E, E, F, B, N_dp, w, h, hp.s0_ems_prob, hp.no_change_prob, s);
            }
            VB_RETURN_IF_CUDA_ERROR();
        }
        timed(prof, s, prof.search_ms, prof.search_launches, [&] {
            const int by = pick_search_block_y(w, h, n_sm);
            const dim3 sb(32, by), sg(VB_DIV_CEIL(w, 32), VB_DIV_CEIL(h, by));
            k_cost_and_random_search_pruned<<<sg, sb, 0, s>>>(A, cam, pcam, hp.n_rand_samples);
        });
        VB_RETURN_IF_CUDA_ERROR();
        if (hp.global_prop_step > 0) {
            launch_global<DIR_L2R>(A, cam, pcam, hp.global_prop_step, s);
            launch_global<DIR_B2T>(A, cam, pcam, hp.global_prop_step, s);
            launch_global<DIR_R2L>(A, cam, pcam, hp.global_prop_step, s);
            launch_global<DIR_T2B>(A, cam, pcam, hp.global_prop_step, s);
        }
        if (hp.local_prop_width > 0) {
            timed(prof, s, prof.local_ms, prof.local_runs, [&] {
                launch_local<DIR_L2R>(A, cam, pcam, hp.local_prop_width, s);
                launch_local<DIR_B2T>(A, cam, pcam, hp.local_prop_width, s);
                launch_local<DIR_R2L>(A, cam, pcam, hp.local_prop_width, s);
                launch_local<DIR_T2B>(A, cam, pcam, hp.local_prop_width, s);
            });
        }
        VB_RETURN_IF_CUDA_ERROR();
    }
    A.rig = rig.ptr;  // the E-step writes the raw posteriors
    timed(prof, s, prof.estep_ms, prof.estep_launches, [&] { k_update_rigidness<<<pg, pb, 0, s>>>(A, cam, pcam); });
    VB_RETURN_IF_CUDA_ERROR();
    if (overlap_smoothing && hp.fb_smooth && N > 0) {
        // smooth the new rigidness maps for the next M-step on the side stream, concurrently with whatever the
        // caller does next with the raw maps (the camera step of the next EM iteration only reads them)
        VB_CUDA(cudaEventRecord(ev_rig_ready, s));
        VB_CUDA(cudaStreamWaitEvent(side, ev_rig_ready, 0));
        StackView E{rig.ptr, rig.pitch, rig.layer_elems()};
        StackView S{rig_s.ptr, rig_s.pitch, rig_s.layer_elems()};
        StackView F{fb_fwd.ptr, fb_fwd.pitch, fb_fwd.layer_elems()};
        StackView B{fb_bwd.ptr, fb_bwd.pitch, fb_bwd.layer_elems()};
        timed(prof, side, prof.smooth_ms, prof.smooth_runs,
              [&] { fb_smooth_stack(E, S, F, B, N, w, h, hp.s0_ems_prob, hp.no_change_prob, side); });
        VB_CUDA(cudaEventRecord(ev_smooth_done, side));
        smooth_layers = N, smooth_s0 = hp.s0_ems_prob, smooth_nc = hp.no_change_prob;
        VB_RETURN_IF_CUDA_ERROR();
    }
    return 0;
}

}  // namespace vb
