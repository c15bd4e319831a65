// Frame-alignment residual / Jacobian kernels (the two GPU entry points the reference's Ceres cost function
// calls) and the separable Gaussian blur, for sm_100a.
//
// Behavioural source: reference gpu-kernels/align_frame.cu:414-554 (host entry points); gblur.cu:12-72.  The
// per-pixel arithmetic (align_frame.cu:47-411) lives in align_pixel.cuh, shared with the solver in falign.cu.
// Restructured: residual, Jacobian and robust loss are ONE kernel (the reference: 2 memsets + 2 kernels per
// evaluation), all layered images live in stacked textures like the EM path.
// Parity target for these two entry points is 1e-4 relative with identical NaN pattern (SURVEY §8c).
#include "../../include/gpu_kernels.h"
#include "../../include/voldor_b200.h"
#include "align_pixel.cuh"
#include "common.cuh"
#include "context.h"
#include <cfloat>
#include <cmath>
#include <mutex>

namespace vb {
namespace {

struct AlignState {
    int N = 0, w = 0, h = 0;
    bool photo = false;
    float vbf = 0, crw = 0;
    AlignIntr K;
    TexStack<float> images, depths;
    TexStack<float2> dimages, ddepths;
    TexStack<float4> normals;
    Plane<float> weights;
    float* residual = nullptr;
    float* jacobian = nullptr;
    size_t cap = 0;
    cudaStream_t stream = nullptr;
    float params_ref[kAlignParams] = {0}, params_tar[kAlignParams] = {0};
};
AlignState g_align;
std::mutex g_align_mutex;

struct AlignParams {
    float ref[kAlignParams], tar[kAlignParams];
};

// residual + Jacobian + weighted sqrt-Cauchy loss, one thread per reference pixel (align_frame.cu:205-411)
__global__ void __launch_bounds__(128)
    k_align_eval(AlignView A, const AlignParams P, int f_ref, int f_tar, int photo, int with_jacobian,
                 int apply_weights, int stride) {
    // stride 1: every pixel, outputs at (y, x).  stride s > 1: only the pixels the reference's cost function reads
    // (x % s == 0, y % s == 0; frame-alignment/align_frame_cost_fun.h:183-185), outputs packed at
    // (y/s) * ceil(w/s) + x/s.  The per-pixel arithmetic does not depend on the mode.
    const int gx = blockIdx.x * blockDim.x + threadIdx.x;
    const int gy = blockIdx.y * blockDim.y + threadIdx.y;
    const int x = gx * stride, y = gy * stride;
    if (x >= A.w || y >= A.h) return;
    const size_t pix = stride == 1 ? (size_t)y * A.w + x : (size_t)gy * ((A.w + stride - 1) / stride) + gx;
    float* jac = A.jacobian + pix * kAlignParams;
    float J[kAlignParams];
    const float residual = align_sample(A, P.ref, P.tar, f_ref, f_tar, x, y, photo, with_jacobian, apply_weights, J);
    A.residual[pix] = residual;
    if (with_jacobian)
        for (int i = 0; i < kAlignParams; i++) jac[i] = J[i];
}

// separable Gaussian with border renormalisation (gblur.cu:12-44); vertical then horizontal like the reference.
// Rounding points as in the reference build: the tap products are fused into the running sum.
template <int VERTICAL>
__global__ void __launch_bounds__(256) k_gblur(const float* __restrict__ src, float* __restrict__ dst, int w, int h,
                                               const float* __restrict__ gk, int hw) {
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    const int d = blockIdx.z;
    if (x >= w || y >= h) return;
    const float* s = src + (size_t)d * w * h;
    float sum = __fmul_rn(gk[0], s[(size_t)y * w + x]);
    float sum_w = gk[0];
    for (int k = 1; k < hw; k++) {
        const float g = gk[k];
        if (VERTICAL) {
            if (y + k < h) sum = __fmaf_rn(g, s[(size_t)(y + k) * w + x], sum), sum_w = __fadd_rn(sum_w, g);
            if (y - k >= 0) sum = __fmaf_rn(g, s[(size_t)(y - k) * w + x], sum), sum_w = __fadd_rn(sum_w, g);
        } else {
            if (x + k < w) sum = __fmaf_rn(g, s[(size_t)y * w + x + k], sum), sum_w = __fadd_rn(sum_w, g);
            if (x - k >= 0) sum = __fmaf_rn(g, s[(size_t)y * w + x - k], sum), sum_w = __fadd_rn(sum_w, g);
        }
    }
    dst[(size_t)d * w * h + (size_t)y * w + x] = __fdiv_rn(sum, sum_w);
}

AlignView make_view(AlignState& S) {
    AlignView A;
    A.w = S.w, A.h = S.h, A.K = S.K, A.vbf = S.vbf, A.crw = S.crw;
    A.images = S.images.tex, A.depths = S.depths.tex, A.dimages = S.dimages.tex, A.normals = S.normals.tex;
    A.images_raw = S.images.ptr, A.images_pitch = S.images.pitch;
    A.depths_raw = S.depths.ptr, A.depths_pitch = S.depths.pitch;
    A.weights = S.weights.ptr, A.wpitch = S.weights.pitch, A.wplane = S.weights.layer_elems();
    A.residual = S.residual, A.jacobian = S.jacobian;
    return A;
}

}  // namespace
}  // namespace vb

int align_frame_init_gpu(float* h_images[], float* h_depths[], float* h_weights[], float* h_K, float vbf, float crw,
                         int N, int w, int h) {
    using namespace vb;
    enter_device();
    std::lock_guard<std::mutex> lock(g_align_mutex);
    AlignState& S = g_align;
    if (!S.stream) VB_CUDA(cudaStreamCreateWithFlags(&S.stream, cudaStreamNonBlocking));
    cudaStream_t s = S.stream;
    S.N = N, S.w = w, S.h = h, S.vbf = vbf, S.crw = crw;
    S.photo = (h_images != nullptr && crw > 0);
    if (S.photo) {
        S.images.ensure(w, h, N, false);
        for (int i = 0; i < N; i++) VB_CUDA(S.images.upload_layer(h_images[i], i, s));
        S.dimages.ensure(w, h, N, false);
    }
    S.depths.ensure(w, h, N, false);
    for (int i = 0; i < N; i++) VB_CUDA(S.depths.upload_layer(h_depths[i], i, s));
    S.weights.ensure(w, h, N, false);
    for (int i = 0; i < N; i++) VB_CUDA(S.weights.upload_layer(h_weights[i], i, s));
    S.ddepths.ensure(w, h, N, false);
    S.normals.ensure(w, h, N, false);
    const size_t npx = (size_t)w * h;
    if (npx > S.cap) {
        if (S.residual) cudaFree(S.residual), cudaFree(S.jacobian);
        VB_CUDA(cudaMalloc((void**)&S.residual, npx * sizeof(float)));
        VB_CUDA(cudaMalloc((void**)&S.jacobian, npx * kAlignParams * sizeof(float)));
        S.cap = npx;
    }
    if (h_K) {  // NULL keeps the cached intrinsics, like the other entry points of this library
        S.K.fx = h_K[0], S.K.cx = h_K[2], S.K.fy = h_K[4], S.K.cy = h_K[5];
        S.K.fxi = 1.f / h_K[0], S.K.cxi = -h_K[2] / h_K[0], S.K.fyi = 1.f / h_K[4], S.K.cyi = -h_K[5] / h_K[4];
    }
    VB_RETURN_IF_CUDA_ERROR();
    const dim3 b(32, 4), g(VB_DIV_CEIL(w, 32), VB_DIV_CEIL(h, 4), N);
    k_align_prepare<<<g, b, 0, s>>>(make_view(S), S.normals.ptr, S.normals.pitch, S.ddepths.ptr, S.ddepths.pitch,
                                    S.dimages.ptr, S.dimages.pitch, S.photo ? 1 : 0);
    VB_CUDA(cudaStreamSynchronize(s));
    VB_RETURN_IF_CUDA_ERROR();
    return 0;
}

int align_frame_eval_gpu(int ref_fid, int tar_fid, const float* h_params_ref, const float* h_params_tar,
                         float* h_o_residual, float* h_o_jacobian, const bool apply_weights) {
    using namespace vb;
    enter_device();
    std::lock_guard<std::mutex> lock(g_align_mutex);
    AlignState& S = g_align;
    if (!S.stream || S.w == 0) return (int)cudaErrorNotReady;
    cudaStream_t s = S.stream;
    if (h_params_ref) memcpy(S.params_ref, h_params_ref, sizeof(S.params_ref));
    if (h_params_tar) memcpy(S.params_tar, h_params_tar, sizeof(S.params_tar));
    AlignParams P;
    memcpy(P.ref, S.params_ref, sizeof(P.ref));
    memcpy(P.tar, S.params_tar, sizeof(P.tar));
    const dim3 b(32, 4), g(VB_DIV_CEIL(S.w, 32), VB_DIV_CEIL(S.h, 4));
    k_align_eval<<<g, b, 0, s>>>(make_view(S), P, ref_fid, tar_fid, S.photo ? 1 : 0, h_o_jacobian != nullptr,
                                 apply_weights ? 1 : 0, 1);
    VB_RETURN_IF_CUDA_ERROR();
    const size_t npx = (size_t)S.w * S.h;
    if (h_o_residual) VB_CUDA(cudaMemcpyAsync(h_o_residual, S.residual, npx * sizeof(float), cudaMemcpyDefault, s));
    if (h_o_jacobian)
        VB_CUDA(cudaMemcpyAsync(h_o_jacobian, S.jacobian, npx * kAlignParams * sizeof(float), cudaMemcpyDefault, s));
    VB_CUDA(cudaStreamSynchronize(s));
    VB_RETURN_IF_CUDA_ERROR();
    return 0;
}

// Strided / packed evaluation: what the only caller of align_frame_eval_gpu actually consumes.  The reference's cost
// function downloads the full residual (4 B/px) and Jacobian (36 B/px) of every evaluation and then reads every
// `stride`-th sample of both (frame-alignment/align_frame_cost_fun.h:169-229; slam_py uses stride 4 for local links and 3 for loop closures); here only those
// samples are computed and copied: ceil(h/stride) x ceil(w/stride) residuals and 9x as many Jacobian entries, in the
// cost function's own index order.  Same per-pixel arithmetic as the full evaluation.
static int align_frame_eval_strided(int ref_fid, int tar_fid, const float* h_params_ref, const float* h_params_tar,
                                    float* h_o_residual, float* h_o_jacobian, bool apply_weights, int stride) {
    using namespace vb;
    enter_device();
    std::lock_guard<std::mutex> lock(g_align_mutex);
    AlignState& S = g_align;
    if (!S.stream || S.w == 0) return (int)cudaErrorNotReady;
    if (stride < 1) return (int)cudaErrorInvalidValue;
    cudaStream_t s = S.stream;
    if (h_params_ref) memcpy(S.params_ref, h_params_ref, sizeof(S.params_ref));
    if (h_params_tar) memcpy(S.params_tar, h_params_tar, sizeof(S.params_tar));
    AlignParams P;
    memcpy(P.ref, S.params_ref, sizeof(P.ref));
    memcpy(P.tar, S.params_tar, sizeof(P.tar));
    const int ow = VB_DIV_CEIL(S.w, stride), oh = VB_DIV_CEIL(S.h, stride);
    const dim3 b(32, 4), g(VB_DIV_CEIL(ow, 32), VB_DIV_CEIL(oh, 4));
    k_align_eval<<<g, b, 0, s>>>(make_view(S), P, ref_fid, tar_fid, S.photo ? 1 : 0, h_o_jacobian != nullptr,
                                 apply_weights ? 1 : 0, stride);
    VB_RETURN_IF_CUDA_ERROR();
    const size_t n = (size_t)ow * oh;
    if (h_o_residual) VB_CUDA(cudaMemcpyAsync(h_o_residual, S.residual, n * sizeof(float), cudaMemcpyDefault, s));
    if (h_o_jacobian)
        VB_CUDA(cudaMemcpyAsync(h_o_jacobian, S.jacobian, n * kAlignParams * sizeof(float), cudaMemcpyDefault, s));
    VB_CUDA(cudaStreamSynchronize(s));
    VB_RETURN_IF_CUDA_ERROR();
    return 0;
}

extern "C" {

DLL_EXPORT int vb_align_frame_init_gpu(float** h_images, float** h_depths, float** h_weights, float* h_K, float vbf,
                                       float crw, int N, int w, int h) {
    return align_frame_init_gpu(h_images, h_depths, h_weights, h_K, vbf, crw, N, w, h);
}
DLL_EXPORT int vb_align_frame_eval_gpu(int ref_fid, int tar_fid, const float* h_params_ref, const float* h_params_tar,
                                       float* h_o_residual, float* h_o_jacobian, int apply_weights) {
    return align_frame_eval_gpu(ref_fid, tar_fid, h_params_ref, h_params_tar, h_o_residual, h_o_jacobian,
                                apply_weights != 0);
}

DLL_EXPORT int vb_align_frame_eval_strided(int ref_fid, int tar_fid, const float* h_params_ref,
                                           const float* h_params_tar, float* h_o_residual, float* h_o_jacobian,
                                           int apply_weights, int stride) {
    return align_frame_eval_strided(ref_fid, tar_fid, h_params_ref, h_params_tar, h_o_residual, h_o_jacobian,
                                    apply_weights != 0, stride);
}

// reference gblur_gpu(GMatf src, GMatf& dst, sigma, ksize) (gblur.cu:47-72) on host/device buffers [depth][h][w]
DLL_EXPORT int vb_gblur_gpu(const float* h_src, float* h_dst, int w, int h, int depth, float sigma, int ksize) {
    vb::enter_device();
    static std::mutex m;
    std::lock_guard<std::mutex> lock(m);
    // grow-only scratch: two image stacks + the half kernel (the reference allocates and frees a GMat per call)
    static cudaStream_t s = nullptr;
    static float *a = nullptr, *b = nullptr, *gk = nullptr;
    static size_t cap = 0;
    if (w <= 0 || h <= 0 || depth <= 0 || !h_src || !h_dst) return (int)cudaErrorInvalidValue;
    if (!s) VB_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    if (ksize == 0) ksize = std::max((int)std::ceil(6 * sigma), 3);
    const int half = ksize / 2 + 1;
    if (half > 128) return (int)cudaErrorInvalidFilterSetting;  // GBLUR_MAXIMUM_HALF_KWIDTH
    float hk[128];
    for (int i = 0; i < half; i++) hk[i] = expf(-(float)(i * i) / (float)(2 * sigma * sigma));
    const size_t n = (size_t)w * h * depth;
    if (!gk) VB_CUDA(cudaMalloc((void**)&gk, 128 * sizeof(float)));
    if (n > cap) {
        if (a) cudaFree(a), cudaFree(b);
        a = b = nullptr, cap = 0;
        VB_CUDA(cudaMalloc((void**)&a, n * sizeof(float)));
        if (cudaMalloc((void**)&b, n * sizeof(float)) != cudaSuccess) {
            cudaFree(a), a = nullptr;
            return (int)cudaErrorMemoryAllocation;
        }
        cap = n;
    }
    VB_CUDA(cudaMemcpyAsync(gk, hk, half * sizeof(float), cudaMemcpyHostToDevice, s));
    VB_CUDA(cudaMemcpyAsync(a, h_src, n * sizeof(float), cudaMemcpyDefault, s));
    const dim3 bl(32, 8), gr(VB_DIV_CEIL(w, 32), VB_DIV_CEIL(h, 8), depth);
    vb::k_gblur<1><<<gr, bl, 0, s>>>(a, b, w, h, gk, half);
    vb::k_gblur<0><<<gr, bl, 0, s>>>(b, a, w, h, gk, half);
    VB_CUDA(cudaMemcpyAsync(h_dst, a, n * sizeof(float), cudaMemcpyDefault, s));
    VB_CUDA(cudaStreamSynchronize(s));
    VB_RETURN_IF_CUDA_ERROR();
    return 0;
}

}  // extern "C"
