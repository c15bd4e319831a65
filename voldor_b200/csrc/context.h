// Execution contexts: everything the reference keeps in file statics, bundled per context.
//
// The reference's device state is process-wide (file statics in optimize_depth.cu:45-52, collect_p3p_instances.cu:29-34,
// per-call buffers elsewhere) and its callers get concurrency by running SEVERAL PROCESSES (the 6-worker pool of
// slam_py/voldor_slam.py:182-187); on one GPU those processes time-slice.  Here one process can hold several
// contexts — each with its own streams, depth/rigidness state, per-pixel XORWOW planes, collector, pose-mode scratch,
// start-sample stream and profile counters, i.e. the state of one reference process — so that independent windows
// run concurrently on one GPU and fill the SMs that a single window's latency-bound stages (camera chain, local
// propagation) leave idle.
//
// Context 0 is what every reference-ABI entry point uses unless the calling host thread selected another one
// (vb_context_select): a program that never selects a context sees exactly the single-process behaviour, including
// the process-wide libc rand() stream.  Contexts >= 1 draw their start samples from a private generator that
// reproduces glibc's rand() sequence (libc_rand.h), like a worker process of their own.
#pragma once
#include <memory>
#include <mutex>
#include <vector>
#include "depth_em.cuh"
#include "falign.cuh"
#include "libc_rand.h"
#include "pose_mode.cuh"
#include "pose_sampler.cuh"

namespace vb {

constexpr int kMaxContexts = 16;

// grow-only device scratch
struct DevBuf {
    float* ptr = nullptr;
    size_t cap = 0;
    int ensure(size_t n) {
        if (n <= cap) return 0;
        if (ptr) cudaFree(ptr);
        ptr = nullptr, cap = 0;
        VB_CUDA(cudaMalloc((void**)&ptr, n * sizeof(float)));
        cap = n;
        return 0;
    }
};

// staging of the host-pointer ABI entry points (abi.cu)
struct AbiScratch {
    DevBuf p2, p3, rv, tv;       // batched P3P
    float K4[4] = {0, 0, 0, 0};  // fx, fy, cx, cy survive a NULL h_K like the reference's __constant__ copies
    cudaStream_t p3p_stream = nullptr;
    DevBuf ms_space, rg_space;   // pose pools of meanshift_gpu / fit_robust_gaussian
};

// scratch of the device-resident window (window.cu)
struct WindowScratch {
    float *rvecs = nullptr, *tvecs = nullptr, *pool = nullptr;
    int* d_used = nullptr;
    int pose_cap = 0;
    double *sum_partial = nullptr, *sums = nullptr;
    double* h_sums = nullptr;
    int* h_counts = nullptr;  // pinned: [0]=n_points, [1]=pool_used
    float* d_out = nullptr;
    size_t out_cap = 0;
    float* d_disp = nullptr;
    size_t disp_cap = 0;
    CamBlock* d_cams = nullptr;  // device-resident poses of the pipelined camera loop
    CamBlock* h_cams = nullptr;  // pinned staging
};

struct BootstrapOverride {
    bool valid = false;
    float R[9], t[3];
    std::vector<float> depth;
    int w = 0, h = 0;
};

struct Context {
    const int id;
    // every entry point that touches this context holds it: calls from different host threads on ONE context
    // serialise (the reference relies on the GIL for that), calls on different contexts run concurrently
    std::recursive_mutex mutex;
    KernelProfile prof;
    DepthEM E;
    Collector C;
    PoseMode M;
    AbiScratch abi;
    WindowScratch ws;
    BootstrapOverride boot;
    FalignState fa;  // frame alignment (falign.cu); the reference-ABI align_frame_* entry points keep their own state
    std::unique_ptr<RandStream> rnd;

    explicit Context(int id_) : id(id_) {
        if (id == 0)
            rnd.reset(new LibcStream());
        else
            rnd.reset(new PrivateStream());
        E.prof = &prof, M.prof = &prof, M.rnd = rnd.get();
    }
};

// The CUDA device of this process' state.  CUDA's current device is a PER-THREAD setting that defaults to device 0, so
// a worker thread created after the main thread chose a device would silently land on GPU 0: every entry point makes
// the library's device current first (enter_device).  It is the device passed to vb_set_device(), else the device that
// was current in the thread that made the first call into the library.
void enter_device();
int set_library_device(int device);

// context `id` (created on first use); nullptr when id is out of range
Context* context_at(int id);
// the context the calling host thread selected (default 0)
Context& current_context();
// returns the previous selection, or -1 when id is out of range
int select_context(int id);

}  // namespace vb
