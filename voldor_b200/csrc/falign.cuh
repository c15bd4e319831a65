// Per-context state of the frame-alignment solver (falign.cu).  Data only, so that context.h can hold it.
#pragma once
#include "common.cuh"

namespace vb {

struct AlignIntr {
    float fx, cx, fy, cy, fxi, cxi, fyi, cyi;
};

namespace fa {
struct Lm;
}

// Device state of one falign() call, grow-only across calls on the same context: the frame stacks with their
// normals and gradients, the pair table, the reduction scratch, the FP64 solver state and a pinned status word.
struct FalignState {
    TexStack<float> images, depths;
    TexStack<float2> dimages, ddepths;
    TexStack<float4> normals;
    Plane<float> weights;
    int* pairs = nullptr;        // [npairs][3]: ref, tar, Jacobian factor (2 when the reverse pair is connected)
    int pair_cap = 0;
    double* partial = nullptr;   // [npairs][blocks][kQ] block sums
    size_t partial_cap = 0;
    double* pair_sums = nullptr; // [npairs][kQ]
    double* frame_sums = nullptr;  // [kMaxFrames][kQ]
    float* out = nullptr;        // poses (N*6) + covariances (N*49) + visibility (N*N) + consistency (N*N)
    fa::Lm* lm = nullptr;
    int* h_status = nullptr;     // pinned: [0] iterations, [1] termination reason
    float* dump = nullptr;       // optional per-sample residual + Jacobian of the last evaluation (test hook)
    size_t dump_cap = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
};

}  // namespace vb
