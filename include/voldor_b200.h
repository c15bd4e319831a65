/* voldor_b200 — C ABI of the B200-native VOLDOR EM hot path.
 *
 * Plain-C aliases (prefix vb_) of the C++-linkage entry points in gpu_kernels.h / py_export.h, for FFI users
 * (ctypes, cgo, JNI, ...).  Each cites the reference interface it replaces; semantics are identical to the
 * C++ symbols (host pointers, NULL = cached / skip, int return code).  `bool` parameters are `int` here and
 * the C++ reference-to-int output of py_voldor_wrapper is a pointer.
 */
#ifndef VOLDOR_B200_H_
#define VOLDOR_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

/* reference: gpu-kernels/gpu_kernels.h:11-15 (meanshift.cu:34-150) */
int vb_meanshift_gpu(float* h_space, float kernel_var, float* h_io_mean, float* h_o_confidence, int* used_iters,
                     int use_external_init_mean, int N, int dims, float epsilon, int max_iters,
                     int max_init_trials, float good_init_confidence);

/* reference: gpu-kernels/gpu_kernels.h:17-22 (fit_robust_gaussian.cu:101-286) */
int vb_fit_robust_gaussian(float* h_space, float* h_io_mean, float* h_io_covar, float trunc_sigma,
                           float covar_reg_lambda, float* h_o_density, int* used_iters, int N, int dims,
                           float epsilon, int max_iters);

/* reference: gpu-kernels/gpu_kernels.h:24-35 (collect_p3p_instances.cu:147-250) */
int vb_collect_p3p_instances(float** h_flows, float** h_rigidnesses, float* h_depth, float* h_K, float** h_Rs,
                             float** h_ts, float* h_o_p2_map, float* h_o_p3_map, int N, int w, int h,
                             int active_idx, float rigidness_thresh, float rigidness_sum_thresh,
                             float sample_min_depth, float sample_max_depth, int max_trace_on_flow);

/* reference: gpu-kernels/gpu_kernels.h:37-39 (solve_batch_ap3p.cu:387-437) */
int vb_solve_batch_p3p_ap3p_gpu(float* h_p3s, float* h_p2s, float* h_o_rvecs, float* h_o_tvecs, float* h_K,
                                int N_pts, int N_poses);

/* reference: gpu-kernels/gpu_kernels.h:40-42 (solve_batch_lambdatwist.cu:51-102) */
int vb_solve_batch_p3p_lambdatwist_gpu(float* h_p3s, float* h_p2s, float* h_o_rvecs, float* h_o_tvecs, float* h_K,
                                       int N_pts, int N_poses);

/* reference: gpu-kernels/gpu_kernels.h:44-58 (optimize_depth.cu:293-520) */
int vb_optimize_depth_gpu(float** h_flows, float** h_rigidnesses, float** h_o_rigidnesses, float** h_depth_priors,
                          float** h_depth_prior_pconfs, float** h_depth_prior_confs, float** h_o_depth_prior_confs,
                          float* h_depth, float* h_o_depth, float* h_K, float** h_Rs, float** h_ts, float** h_dp_Rs,
                          float** h_dp_ts, float abs_resize_factor, int N, int N_dp, int w, int h, float basefocal,
                          int n_rand_samples, int global_prop_step, int local_prop_width, float lambda, float omega,
                          float disp_delta, float delta, int fb_smooth, float s0_ems_prob, float no_change_prob,
                          float range_factor, int update_rigidness_only);

/* reference: gpu-kernels/gpu_kernels.h:60-66 (align_frame.cu:512-554) */
int vb_align_frame_init_gpu(float** h_images, float** h_depths, float** h_weights, float* h_K, float vbf, float crw,
                            int N, int w, int h);

/* reference: gpu-kernels/gpu_kernels.h:68-74 (align_frame.cu:414-510) */
int vb_align_frame_eval_gpu(int ref_fid, int tar_fid, const float* h_params_ref, const float* h_params_tar,
                            float* h_o_residual, float* h_o_jacobian, int apply_weights);

/* No counterpart in the reference ABI: the same evaluation restricted to the samples its only caller reads — every
 * stride-th pixel in x and y (frame-alignment/align_frame_cost_fun.h:183-229), packed as
 * out[(y/stride) * ceil(w/stride) + x/stride] (x9 for the Jacobian).  slam_py uses stride 4 for local links and 3 for
 * loop closures, which cut the per-evaluation D2H from 40 B/px to 40/16 and 40/9 B/px.  Values are those of
 * vb_align_frame_eval_gpu at the same pixels. */
int vb_align_frame_eval_strided(int ref_fid, int tar_fid, const float* h_params_ref, const float* h_params_tar,
                                float* h_o_residual, float* h_o_jacobian, int apply_weights, int stride);

/* reference: gpu-kernels/gblur.h:6 (gblur.cu:47-72; device-to-device in the reference, host buffers here).
 * src/dst: [depth][h][w] float, ksize odd. */
int vb_gblur_gpu(const float* h_src, float* h_dst, int w, int h, int depth, float sigma, int ksize);

/* reference: voldor/py_export.h:3-11 (py_export.cpp:5-79) — one VO window through the device-resident pipeline */
int vb_py_voldor_wrapper(const float* flows, const float* disparity, const float* disparity_pconf,
                         const float* depth_priors, const float* depth_prior_poses, const float* depth_prior_pconfs,
                         float fx, float fy, float cx, float cy, float basefocal, int N, int N_dp, int w, int h,
                         const char* config, int* n_registered, float* poses, float* poses_covar, float* depth,
                         float* depth_conf);

/* reference: frame-alignment/py_export.h (py_export.cpp, align_frame.cpp) — keyframe alignment with the solver on
 * the device (DESIGN.md §9).  Runs on the calling thread's execution context.  Returns 0, a CUDA error code, or: */
#define VB_FALIGN_EINVAL (-1) /* N outside 2..64, stride < 1, connectivity entry out of range or unterminated */
#define VB_FALIGN_EDEBUG (-2) /* debug != 0 (the reference opens OpenCV windows) */
int vb_py_falign_wrapper(const float* depths, const float* images, const float* weights, const float* poses_init,
                         float* poses_ret, const int* connectivity, float* poses_covar, float* scaling_factor,
                         float* visibility_mat, float* consistency_mat, int N, int w, int h, float fx, float fy,
                         float cx, float cy, float vbf, float crw, int optimize_7dof, int graduated_optmize, int stride,
                         float consistency_residual_bound, int debug);

/* ---- additions that have no counterpart in the reference ---- */

/* Same alignment, also reporting what the solve did.  n_connectivity: length of `connectivity` in ints including
 * the -1 terminator (< 0: scan to the terminator).  iters_run: LM iterations; reason: termination (1 gradient,
 * 2 parameter, 3 function tolerance, 4 minimum trust-region radius, 5 iteration limit, 6 invalid steps);
 * costs[2]: initial and final cost 1/2 sum f^2; stats[4] ms: total, upload + preparation, LM loop, covariance +
 * scores + download.  samples (test hook, may be NULL): the per-sample residuals [pairs][n] and Jacobians
 * [pairs][n][9] of the first evaluation, n = ceil(w/stride) * ceil(h/stride), as vb_align_frame_eval_strided
 * packs them.  Any output pointer except the reference's may be NULL. */
int vb_py_falign_wrapper_ex(const float* depths, const float* images, const float* weights, const float* poses_init,
                            float* poses_ret, const int* connectivity, int n_connectivity, float* poses_covar,
                            float* scaling_factor, float* visibility_mat, float* consistency_mat, int N, int w, int h,
                            float fx, float fy, float cx, float cy, float vbf, float crw, int optimize_7dof,
                            int graduated_optmize, int stride, float consistency_residual_bound, int debug,
                            int* iters_run, int* reason, double* costs, float* stats, float* samples);

/* Monocular bootstrap injection: when set (valid != 0), the next windows that have no depth prior start from
 * this pose (R row-major 3x3, t) and depth map instead of the essential-matrix bootstrap
 * (reference: voldor/voldor.cpp:151-162, geometry.cpp:267-332).  Used by the measurement harness so every
 * series starts from identical state (BASELINE.md §3). */
int vb_set_bootstrap_override(int valid, const float* R9, const float* t3, const float* depth, int w, int h);

/* The monocular bootstrap itself (host code, no GPU needed): relative pose of the first frame pair from one dense
 * flow map (w*h*2 floats) by an LMedS essential-matrix fit, then the closed-form depth map.  Replaces the OpenCV
 * calls of voldor/geometry.cpp:288-332 and :267-285.  R9 row-major, |t| = 1.  Returns 0, or 1 if degenerate. */
int vb_bootstrap_from_flow(const float* flow, int w, int h, const float* K9, float* R9, float* t3, float* depth);

/* Same window call, also reporting the number of EM iterations executed (VOLDOR::solve's return value,
 * voldor/voldor.cpp:148) and per-stage device/host time in ms: stats[0]=total, [1]=cameras, [2]=depth, [3]=io. */
int vb_py_voldor_wrapper_ex(const float* flows, const float* disparity, const float* disparity_pconf,
                            const float* depth_priors, const float* depth_prior_poses,
                            const float* depth_prior_pconfs, float fx, float fy, float cx, float cy, float basefocal,
                            int N, int N_dp, int w, int h, const char* config, int* n_registered, float* poses,
                            float* poses_covar, float* depth, float* depth_conf, int* iters_run, float* stats);

/* ---- execution contexts: several independent windows in flight on one GPU ----
 *
 * The reference keeps its device state in file statics (gpu-kernels/optimize_depth.cu:45-52,
 * collect_p3p_instances.cu:29-34) and gets concurrency from a pool of worker PROCESSES
 * (slam_py/voldor_slam.py:182-191).  Here one process holds up to vb_context_max() execution contexts, each owning
 * what one reference process owns: streams, depth / rigidness / per-pixel RNG state, collector and pose-mode scratch,
 * bootstrap override, profile counters and the start-sample rand() stream.  Every entry point of this library acts on
 * the context selected by the CALLING HOST THREAD (default 0); calls on different contexts run concurrently, calls on
 * one context serialise.  Context 0 draws start samples from the process-wide libc rand() exactly like the reference;
 * contexts >= 1 own a private generator with glibc's rand() sequence (as a fresh process would), seeded 1. */
int vb_context_select(int ctx);           /* bind this host thread to context ctx; returns the previous one, -1 if invalid */
int vb_context_current(void);
int vb_context_max(void);
int vb_context_srand(unsigned int seed);  /* srand() of the current context's start-sample stream */
int vb_context_rand(void);                /* one draw from it (test hook: consumption checks) */

/* Select the CUDA device of this process' state.  CUDA's current device is per host thread (default 0), so every entry
 * point of the library makes this device current first: worker threads need no cudaSetDevice of their own.  Default:
 * the device that was current in the thread that made the first call into the library. */
int vb_set_device(int device);
/* Test hook: the CUDA device an entry point would run on when called from this host thread. */
int vb_debug_thread_device(void);

/* In-library CUDA-event timing of the dominant kernel (fused cost + random depth search), for roofline
 * reporting.  Enabling it adds one event synchronisation per launch, so it is off by default. */
void vb_profile_enable(int on);
void vb_profile_get(double* search_ms, long long* search_launches);
/* also timed while profiling is on: ms3 / counts3 = { E-step kernel, one forward-backward smoothing of the rigidness
 * maps (4 launches), the four local-propagation passes of one depth step } */
void vb_profile_get_more(double* ms3, long long* counts3);
/* Counters of the on-device fixed-point loops since the last vb_profile_enable():
 * out5 = { mean-shift runs, their iterations, start-sample trials, robust-fit runs, their iterations }. */
void vb_profile_counters(long long* out5);

/* Profiling hook: per-phase clock64 totals accumulated since process start, only collected when the environment
 * variable VB_POSE_MODE_PHASES is set before the first call.  out16[0..5]: robust fit (LU, E-step, level-1 sums,
 * exchange barrier, level-2 sums, M-step); out16[8..15]: mean-shift (pool build, staging, weights, level-1 sums,
 * exchange barrier, level-2 sums, mean update, result + pose tail).  Returns 0, or 1 when not collected. */
int vb_debug_pose_mode_phases(long long* out24);

/* Test hook: rotation vector -> matrix through the device and the host instantiation of the same deterministic
 * double-precision routine (csrc/host_math.h); the window pipeline relies on both giving identical bits. */
int vb_debug_rvec_to_matrix(const float* rvecs, int n, float* R_device, float* R_host);

/* Test hook for the speculative use of the libc rand() stream by the fused mean-shift start-sample selection
 * (csrc/libc_rand.h): snapshot, draw `draw` numbers, rewind, draw `keep`.  Afterwards the process-wide stream must
 * be exactly `keep` draws past where it was.  Returns 0, or 1 if the state array could not be captured. */
int vb_debug_rand_speculate(int draw, int keep);

/* Test hook: parse a flag string with this library's flag grammar (csrc/config.h; reference voldor/config.h:110-253,
 * py_export.cpp:15-25) and dump all 56 fields as doubles; returns the number of fields written. */
int vb_debug_config_dump(const char* flags, float fx, float fy, float cx, float cy, float basefocal, double* out);

/* Library self-description: returns a static string "voldor_b200 <version> sm_100a". */
const char* vb_version(void);

#ifdef __cplusplus
}
#endif
#endif /* VOLDOR_B200_H_ */
