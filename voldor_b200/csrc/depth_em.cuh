// Depth / rigidness EM state and driver (device-resident).
//
// Replaces the reference's optimize_depth.cu file-static GMats + 26-launch host driver
// (reference: gpu-kernels/optimize_depth.cu:24-52 state, :293-520 driver, fb_smooth.h:17-109).
// One DepthEM instance per execution context (context.h; context 0 = the reference's one-per-process state) keeps
// what the reference keeps in file statics, including the per-pixel XORWOW streams that advance across calls and
// windows (optimize_depth.cu:357-361, SURVEY §9 Q1).
#pragma once
#include <mutex>
#include "common.cuh"

namespace vb {

struct DepthHyper {
    float abs_resize_factor, basefocal;
    int n_rand_samples, global_prop_step, local_prop_width;
    float lambda, omega, disp_delta, delta;
    bool fb_smooth;
    float s0_ems_prob, no_change_prob;
    float range_factor;
};

struct KernelProfile;

struct DepthEM {
    KernelProfile* prof = nullptr;  // the owning context's counters
    // geometry of the cached window
    int w = 0, h = 0;
    // device state
    TexStack<float2> flows;      // N layers, bilinear fetched
    Plane<float> rig;            // N layers, rigidness maps W_f (raw E-step posteriors)
    Plane<float> rig_s;          // N layers, forward-backward smoothed copy = the weights of the M-step
    Plane<float> depth, cost;    // 1 layer each
    Plane<uint32_t> rng;         // 6 layers: XORWOW d, v0..v4 (SoA)
    TexStack<float> dp, dp_pconf, dp_conf;  // N_dp layers each, bilinear fetched
    Plane<float> fb_fwd, fb_bwd;            // message scratch, max(N, N_dp) layers
    CamBlock cam;
    PriorCamBlock pcam;
    cudaStream_t stream = nullptr;
    // Side stream for the smoothing of the rigidness maps: in the window pipeline it runs right after the E-step,
    // concurrently with the next camera step (which reads the raw maps).  smooth_layers > 0 <=> rig_s holds (once
    // ev_smooth_done fires) the smoothing of the current `rig` with these parameters.
    cudaStream_t side = nullptr;
    cudaEvent_t ev_rig_ready = nullptr, ev_smooth_done = nullptr;
    bool overlap_smoothing = false;
    int smooth_layers = 0;
    float smooth_s0 = 0.f, smooth_nc = 0.f;
    int n_sm = 148;
    // call before anything else writes `rig` on `stream` (uploads, fills)
    void invalidate_smoothing();
    // when set, kernels fetch flows from this stack instead of `flows` (window pipeline shares one upload)
    TexStack<float2>* shared_flows = nullptr;

    int init_stream();
    // (Re)allocate for a window geometry; mirrors the reference's lazy create() calls
    // (optimize_depth.cu:357-375,391-404,427-458).  Re-seeds the RNG plane iff (w,h) changed.
    int ensure(int w_, int h_, int N, int N_dp);
    int seed_rng();

    void set_K(const float* h_K) { fill_K(cam, h_K); }
    void set_pose(int f, const float* R9, const float* t3) {
        memcpy(cam.R[f], R9, 9 * sizeof(float));
        memcpy(cam.t[f], t3, 3 * sizeof(float));
    }
    void set_prior_pose(int f, const float* R9, const float* t3) {
        memcpy(pcam.R[f], R9, 9 * sizeof(float));
        memcpy(pcam.t[f], t3, 3 * sizeof(float));
    }

    // One M-step (unless rigidness_only) + E-step on the device-resident state.  Asynchronous on `stream`.
    int run(int N, int N_dp, const DepthHyper& hp, bool update_rigidness_only);
};

// Optional in-library timing of the dominant kernel (fused cost + random search), CUDA events on the launching
// stream.  Off by default; bench.py switches it on for the roofline figure (vb_profile_* in voldor_b200.h).
struct KernelProfile {
    bool enabled = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    double search_ms = 0;      // accumulated duration of k_cost_and_random_search_pruned
    long long search_launches = 0;
    double estep_ms = 0;       // k_update_rigidness
    long long estep_launches = 0;
    double smooth_ms = 0;      // one forward-backward smoothing of the N rigidness maps (rows, posterior, cols, posterior)
    long long smooth_runs = 0;
    double local_ms = 0;       // the four local-propagation passes of one depth step
    long long local_runs = 0;
    long long launches = 0;    // all kernel launches issued by the depth step / pose stages since reset
    // fixed-point loops of the pose-mode kernels (always counted; host-side bookkeeping only)
    long long meanshift_runs = 0, meanshift_iters = 0, meanshift_trials = 0;
    long long robust_runs = 0, robust_iters = 0;
};

}  // namespace vb
