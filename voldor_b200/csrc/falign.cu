// Frame alignment (the reference's pyvoldor.falign: frame-alignment/py_export.cpp -> align_frame.cpp) without Ceres:
// the normal equations of every connectivity pair are reduced on the device and a device-resident FP64
// Levenberg-Marquardt loop (falign_math.h) restates the trust-region solve the reference configures.  No per-pixel
// data crosses PCIe during the solve.  DESIGN.md §9 has the contract, the summation tree and the launch counts.
//
// Per LM iteration: k_fa_eval (every pair, one launch), k_fa_pair_sums, k_fa_step, then one 8-byte status readback
// and one stream synchronisation.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <vector>
#include "../../include/py_falign.h"
#include "../../include/voldor_b200.h"
#include "align_pixel.cuh"
#include "context.h"
#include "falign_math.h"

namespace vb {
namespace {

using fa::kBlock;
using fa::kP;
using fa::kQ;

constexpr int kScoreQ = 2;

// Residual, Jacobian (LM mode) or score quantities of every sample of every pair, reduced to one block sum per
// quantity (falign_math.h: halving inside each warp, then over the 8 warps).  blockIdx.y = pair, blockIdx.x = block of
// 256 consecutive packed samples.  xr / xt: the FP64 state read for the ref / target frame of each pair.
// dump (LM mode, optional): the raw per-sample residual and Jacobian, [pair][n] then [pair][n][9].
template <int NQ>
__global__ void __launch_bounds__(kBlock)
    k_fa_eval(AlignView A, const int* __restrict__ pairs, const double* xr, const double* xt, int photo,
              int with_jacobian, int apply_weights, int stride, int use_factor, double bound, double* partial,
              float* dump) {
    __shared__ double sm[kBlock / 32][NQ];
    const int p = blockIdx.y;
    const int ref = pairs[p * 3], tar = pairs[p * 3 + 1];
    const int ow = VB_DIV_CEIL(A.w, stride), n = ow * VB_DIV_CEIL(A.h, stride);
    const int k = blockIdx.x * kBlock + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float f = 0.f, J[kAlignParams];
    for (int i = 0; i < kAlignParams; i++) J[i] = 0.f;
    if (k < n) {
        float pref[kP], ptar[kP];
        fa::params_float(xr + ref * kP, pref);
        fa::params_float(xt + tar * kP, ptar);
        f = align_sample(A, pref, ptar, ref, tar, (k % ow) * stride, (k / ow) * stride, photo, with_jacobian,
                         apply_weights, J);
        if (dump) {
            dump[(size_t)p * n + k] = f;
            float* dj = dump + (size_t)gridDim.y * n + ((size_t)p * n + k) * kP;
            for (int i = 0; i < kP; i++) dj[i] = J[i];
        }
    }
    auto put = [&](int q, double v) {
        for (int h = 16; h >= 1; h >>= 1) v = __dadd_rn(v, __shfl_down_sync(0xffffffffu, v, h));
        if (lane == 0) sm[warp][q] = v;
    };
    if constexpr (NQ == kQ) {
        if (k < n) {
            // NaN residual -> 0 and its Jacobian row -> 0 (align_frame_cost_fun.h:187-207); x2 for a bi-connected pair
            if (!isfinite(f)) {
                f = 0.f;
                for (int i = 0; i < kP; i++) J[i] = 0.f;
            }
            const float factor = use_factor ? (float)pairs[p * 3 + 2] : 1.f;
            for (int i = 0; i < kP; i++) J[i] = __fmul_rn(J[i], factor);
        }
        int q = 0;
        put(q++, __dmul_rn(f, f));
#pragma unroll
        for (int i = 0; i < kP; i++) put(q++, __dmul_rn(J[i], f));
#pragma unroll
        for (int i = 0; i < kP; i++)
#pragma unroll
            for (int j = i; j < kP; j++) put(q++, __dmul_rn(J[i], J[j]));
    } else {
        double v[kScoreQ] = {0.0, 0.0};
        if (k < n) fa::score_quantities(f, bound, v);
        put(0, v[0]);
        put(1, v[1]);
    }
    __syncthreads();
    if (threadIdx.x < NQ) {
        double s[kBlock / 32];
        for (int w = 0; w < kBlock / 32; w++) s[w] = sm[w][threadIdx.x];
        for (int h = kBlock / 64; h >= 1; h >>= 1)
            for (int i = 0; i < h; i++) s[i] = __dadd_rn(s[i], s[i + h]);
        partial[((size_t)p * gridDim.x + blockIdx.x) * NQ + threadIdx.x] = s[0];
    }
}

// block sums of a pair, in block order from +0
__global__ void k_fa_pair_sums(const double* __restrict__ partial, int nblocks, int nq, double* pair_sums) {
    const int p = blockIdx.x, q = threadIdx.x;
    if (q >= nq) return;
    double s = 0.0;
    for (int b = 0; b < nblocks; b++) s = __dadd_rn(s, partial[((size_t)p * nblocks + b) * nq + q]);
    pair_sums[(size_t)p * nq + q] = s;
}

__device__ void frame_sums(const fa::Lm* L, const int* pairs, int npairs, const double* pair_sums, double* fs) {
    for (int i = threadIdx.x; i < L->N * kQ; i += blockDim.x) fs[i] = fa::frame_sum(pair_sums, pairs, npairs, i / kQ, i % kQ);
    __syncthreads();
}

// frame sums in parallel, then the serial LM logic on one thread (iteration zero when start != 0)
__global__ void __launch_bounds__(256)
    k_fa_step(fa::Lm* L, const int* pairs, int npairs, const double* pair_sums, double* fs, int start) {
    frame_sums(L, pairs, npairs, pair_sums, fs);
    if (threadIdx.x != 0) return;
    if (start)
        fa::lm_start(*L, fs);
    else
        fa::lm_candidate(*L, fs);
}

// poses and covariances from the final state, visibility / consistency from the score sums
__global__ void __launch_bounds__(256)
    k_fa_finish(const fa::Lm* L, const int* pairs, int npairs, const double* cov_sums, const double* score_sums,
                double* fs, int optimize_7dof, int w, int h, float* out) {
    frame_sums(L, pairs, npairs, cov_sums, fs);
    const int N = L->N;
    float* vis = out + N * 6 + N * 49;
    float* cons = vis + N * N;
    if (threadIdx.x == 0) {
        fa::finish(*L, fs, optimize_7dof, out, out + N * 6);
        for (int i = 0; i < N * N; i++) vis[i] = cons[i] = __int_as_float(0x7fc00000);  // quiet NaN, as std::nan("")
        for (int p = 0; p < npairs; p++)
            fa::pair_scores(score_sums + p * kScoreQ, w, h, &vis[pairs[p * 3] * N + pairs[p * 3 + 1]],
                            &cons[pairs[p * 3] * N + pairs[p * 3 + 1]]);
    }
}

template <typename T>
int grow(T*& p, size_t& cap, size_t n) {
    if (n <= cap) return 0;
    if (p) cudaFree(p);
    p = nullptr, cap = 0;
    VB_CUDA(cudaMalloc((void**)&p, n * sizeof(T)));
    cap = n;
    return 0;
}

}  // namespace

int falign_run(const float* depths, const float* images, const float* weights, const float* poses_init,
               const int* connectivity, int n_connectivity, float* poses_ret, float* poses_covar,
               float* scaling_factor, float* visibility, float* consistency, int N, int w, int h, float fx, float fy,
               float cx, float cy, float vbf, float crw, bool optimize_7dof, int stride, float bound, bool debug,
               int* iters_run, int* reason, double* costs, float* stats, float* dump) {
    if (debug) {
        printf("falign: debug=True (OpenCV windows) is not supported\n");
        return VB_FALIGN_EDEBUG;
    }
    std::vector<int> pairs;
    if (N < 2 || N > fa::kMaxFrames || w < 1 || h < 1 || stride < 1 || !depths || !poses_ret || !poses_covar ||
        !scaling_factor || !visibility || !consistency || !fa::parse_pairs(connectivity, n_connectivity, N, pairs)) {
        printf("falign: invalid input\n");
        return VB_FALIGN_EINVAL;
    }
    const auto t0 = std::chrono::steady_clock::now();
    enter_device();
    Context& cx_ = current_context();
    std::lock_guard<std::recursive_mutex> lock(cx_.mutex);
    FalignState& S = cx_.fa;
    if (!S.stream) {
        VB_CUDA(cudaStreamCreateWithFlags(&S.stream, cudaStreamNonBlocking));
        for (auto& e : S.ev) VB_CUDA(cudaEventCreate(&e));
        VB_CUDA(cudaMalloc((void**)&S.lm, sizeof(fa::Lm)));
        VB_CUDA(cudaMalloc((void**)&S.frame_sums, fa::kMaxFrames * kQ * sizeof(double)));
        VB_CUDA(cudaMalloc((void**)&S.out, (fa::kMaxFrames * (6 + 49 + 2 * fa::kMaxFrames)) * sizeof(float)));
        VB_CUDA(cudaMallocHost((void**)&S.h_status, 2 * sizeof(int)));
    }
    cudaStream_t s = S.stream;
    VB_CUDA(cudaEventRecord(S.ev[0], s));
    const int npairs = (int)pairs.size() / 3;
    const bool photo = images != nullptr && crw > 0;
    const size_t npx = (size_t)w * h;

    // frames, normals and gradients (the reference's align_frame_init_gpu)
    S.depths.ensure(w, h, N, false), S.ddepths.ensure(w, h, N, false), S.normals.ensure(w, h, N, false);
    S.weights.ensure(w, h, N, false);
    if (photo) S.images.ensure(w, h, N, false), S.dimages.ensure(w, h, N, false);
    if (!S.depths.ptr || !S.normals.ptr || !S.weights.ptr || (photo && !S.images.ptr)) return (int)cudaErrorMemoryAllocation;
    std::vector<float> ones;
    if (!weights) ones.assign(npx, 1.f);
    for (int i = 0; i < N; i++) {
        VB_CUDA(S.depths.upload_layer(depths + i * npx, i, s));
        VB_CUDA(S.weights.upload_layer(weights ? weights + i * npx : ones.data(), i, s));
        if (photo) VB_CUDA(S.images.upload_layer(images + i * npx, i, s));
    }
    AlignView A;
    A.w = w, A.h = h, A.vbf = vbf, A.crw = crw;
    A.K.fx = fx, A.K.cx = cx, A.K.fy = fy, A.K.cy = cy;
    A.K.fxi = 1.f / fx, A.K.cxi = -cx / fx, A.K.fyi = 1.f / fy, A.K.cyi = -cy / fy;
    A.images = S.images.tex, A.depths = S.depths.tex, A.dimages = S.dimages.tex, A.normals = S.normals.tex;
    A.images_raw = S.images.ptr, A.images_pitch = S.images.pitch;
    A.depths_raw = S.depths.ptr, A.depths_pitch = S.depths.pitch;
    A.weights = S.weights.ptr, A.wpitch = S.weights.pitch, A.wplane = S.weights.layer_elems();
    A.residual = nullptr, A.jacobian = nullptr;
    k_align_prepare<<<dim3(VB_DIV_CEIL(w, 32), VB_DIV_CEIL(h, 4), N), dim3(32, 4), 0, s>>>(
        A, S.normals.ptr, S.normals.pitch, S.ddepths.ptr, S.ddepths.pitch, S.dimages.ptr, S.dimages.pitch, photo ? 1 : 0);

    // pair table, solver state, scratch
    if (npairs > S.pair_cap) {
        if (S.pairs) cudaFree(S.pairs), cudaFree(S.pair_sums);
        S.pairs = nullptr, S.pair_sums = nullptr, S.pair_cap = 0;
        VB_CUDA(cudaMalloc((void**)&S.pairs, (size_t)npairs * 3 * sizeof(int)));
        VB_CUDA(cudaMalloc((void**)&S.pair_sums, (size_t)npairs * (kQ + kScoreQ) * sizeof(double)));
        S.pair_cap = npairs;
    }
    VB_CUDA(cudaMemcpyAsync(S.pairs, pairs.data(), pairs.size() * sizeof(int), cudaMemcpyHostToDevice, s));
    std::vector<int> is_ref(N, 0);
    for (int p = 0; p < npairs; p++) is_ref[pairs[p * 3]] = 1;
    std::unique_ptr<fa::Lm> L(new fa::Lm);
    fa::lm_init(*L, N, optimize_7dof, photo, poses_init, is_ref.data());
    VB_CUDA(cudaMemcpyAsync(S.lm, L.get(), sizeof(fa::Lm), cudaMemcpyHostToDevice, s));
    const int n_lm = VB_DIV_CEIL(w, stride) * VB_DIV_CEIL(h, stride), nb_lm = VB_DIV_CEIL(n_lm, kBlock);
    const int nb_sc = VB_DIV_CEIL((int)npx, kBlock);
    if (grow(S.partial, S.partial_cap, (size_t)npairs * std::max(nb_lm * kQ, nb_sc * kScoreQ))) return (int)cudaErrorMemoryAllocation;
    if (dump && grow(S.dump, S.dump_cap, (size_t)npairs * n_lm * (1 + kP))) return (int)cudaErrorMemoryAllocation;
    VB_CUDA(cudaEventRecord(S.ev[1], s));

    // the LM loop: one evaluation of every pair, its reduction and one step per iteration
    const double* x = &S.lm->x[0][0];
    const double* xc = &S.lm->xc[0][0];
    for (int it = 0;; it++) {
        k_fa_eval<kQ><<<dim3(nb_lm, npairs), kBlock, 0, s>>>(A, S.pairs, it == 0 ? x : xc, x, photo ? 1 : 0, 1, 1,
                                                             stride, 1, 0.0, S.partial, it == 0 && dump ? S.dump : nullptr);
        k_fa_pair_sums<<<npairs, 64, 0, s>>>(S.partial, nb_lm, kQ, S.pair_sums);
        k_fa_step<<<1, 256, 0, s>>>(S.lm, S.pairs, npairs, S.pair_sums, S.frame_sums, it == 0 ? 1 : 0);
        VB_CUDA(cudaMemcpyAsync(S.h_status, &S.lm->iter, 2 * sizeof(int), cudaMemcpyDeviceToHost, s));
        VB_CUDA(cudaStreamSynchronize(s));
        VB_RETURN_IF_CUDA_ERROR();
        if (S.h_status[1] != fa::kRunning) break;
    }
    VB_CUDA(cudaEventRecord(S.ev[2], s));

    // covariance (un-doubled Jacobian at the final state) and scores (full resolution, unweighted)
    double* cov_sums = S.pair_sums;
    double* score_sums = S.pair_sums + (size_t)npairs * kQ;
    k_fa_eval<kQ><<<dim3(nb_lm, npairs), kBlock, 0, s>>>(A, S.pairs, x, x, photo ? 1 : 0, 1, 1, stride, 0, 0.0,
                                                         S.partial, nullptr);
    k_fa_pair_sums<<<npairs, 64, 0, s>>>(S.partial, nb_lm, kQ, cov_sums);
    k_fa_eval<kScoreQ><<<dim3(nb_sc, npairs), kBlock, 0, s>>>(A, S.pairs, x, x, photo ? 1 : 0, 0, 0, 1, 0,
                                                              (double)bound, S.partial, nullptr);
    k_fa_pair_sums<<<npairs, 64, 0, s>>>(S.partial, nb_sc, kScoreQ, score_sums);
    k_fa_finish<<<1, 256, 0, s>>>(S.lm, S.pairs, npairs, cov_sums, score_sums, S.frame_sums, optimize_7dof ? 1 : 0, w,
                                  h, S.out);
    VB_RETURN_IF_CUDA_ERROR();
    const int C = optimize_7dof ? 7 : 6;
    std::vector<float> out((size_t)N * (6 + 49 + 2 * N));
    VB_CUDA(cudaMemcpyAsync(out.data(), S.out, out.size() * sizeof(float), cudaMemcpyDeviceToHost, s));
    VB_CUDA(cudaMemcpyAsync(L.get(), S.lm, sizeof(fa::Lm), cudaMemcpyDeviceToHost, s));
    if (dump)
        VB_CUDA(cudaMemcpyAsync(dump, S.dump, (size_t)npairs * n_lm * (1 + kP) * sizeof(float), cudaMemcpyDeviceToHost,
                                s));
    VB_CUDA(cudaEventRecord(S.ev[3], s));
    VB_CUDA(cudaStreamSynchronize(s));
    VB_RETURN_IF_CUDA_ERROR();

    memcpy(poses_ret, out.data(), (size_t)N * 6 * sizeof(float));
    memcpy(poses_covar, out.data() + N * 6, (size_t)N * C * C * sizeof(float));
    memcpy(visibility, out.data() + N * 55, (size_t)N * N * sizeof(float));
    memcpy(consistency, out.data() + N * 55 + N * N, (size_t)N * N * sizeof(float));
    for (int f = 0; f < N; f++) scaling_factor[f] = optimize_7dof ? (float)std::exp(L->x[f][6]) : 1.f;
    if (iters_run) *iters_run = L->iter;
    if (reason) *reason = L->reason;
    if (costs) costs[0] = L->cost0, costs[1] = L->cost;
    if (stats) {
        stats[0] = (float)std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        for (int i = 0; i < 3; i++) VB_CUDA(cudaEventElapsedTime(&stats[1 + i], S.ev[i], S.ev[i + 1]));
    }
    return 0;
}

}  // namespace vb

int py_falign_wrapper(const float* depths, const float* images, const float* weights, float* poses_init,
                      float* poses_ret, const int* connectivity, float* poses_covar, float* scaling_factor,
                      float* visibility_mat, float* consistency_mat, const int N, const int w, const int h,
                      const float fx, const float fy, const float cx, const float cy, const float vbf, const float crw,
                      const bool optimize_7dof, const bool graduated_optmize, const int stride,
                      const float consistency_residual_bound, const bool debug) {
    (void)graduated_optmize;  // accepted and unused, as in the reference
    return vb::falign_run(depths, images, weights, poses_init, connectivity, -1, poses_ret, poses_covar,
                          scaling_factor, visibility_mat, consistency_mat, N, w, h, fx, fy, cx, cy, vbf, crw,
                          optimize_7dof, stride, consistency_residual_bound, debug, nullptr, nullptr, nullptr, nullptr,
                          nullptr);
}

extern "C" {

VB_EXPORT int vb_py_falign_wrapper(const float* depths, const float* images, const float* weights,
                                   const float* poses_init, float* poses_ret, const int* connectivity,
                                   float* poses_covar, float* scaling_factor, float* visibility_mat,
                                   float* consistency_mat, int N, int w, int h, float fx, float fy, float cx, float cy,
                                   float vbf, float crw, int optimize_7dof, int graduated_optmize, int stride,
                                   float consistency_residual_bound, int debug) {
    (void)graduated_optmize;
    return vb::falign_run(depths, images, weights, poses_init, connectivity, -1, poses_ret, poses_covar,
                          scaling_factor, visibility_mat, consistency_mat, N, w, h, fx, fy, cx, cy, vbf, crw,
                          optimize_7dof != 0, stride, consistency_residual_bound, debug != 0, nullptr, nullptr,
                          nullptr, nullptr, nullptr);
}

VB_EXPORT int vb_py_falign_wrapper_ex(const float* depths, const float* images, const float* weights,
                                      const float* poses_init, float* poses_ret, const int* connectivity,
                                      int n_connectivity, float* poses_covar, float* scaling_factor,
                                      float* visibility_mat, float* consistency_mat, int N, int w, int h, float fx,
                                      float fy, float cx, float cy, float vbf, float crw, int optimize_7dof,
                                      int graduated_optmize, int stride, float consistency_residual_bound, int debug,
                                      int* iters_run, int* reason, double* costs, float* stats, float* samples) {
    (void)graduated_optmize;
    return vb::falign_run(depths, images, weights, poses_init, connectivity, n_connectivity, poses_ret, poses_covar,
                          scaling_factor, visibility_mat, consistency_mat, N, w, h, fx, fy, cx, cy, vbf, crw,
                          optimize_7dof != 0, stride, consistency_residual_bound, debug != 0, iters_run, reason, costs,
                          stats, samples);
}

}  // extern "C"
