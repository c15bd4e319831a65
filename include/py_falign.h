// voldor_b200 — drop-in boundary of frame alignment (Python-binding level).
//
// py_falign_wrapper has the C++-linkage signature of the reference's frame-alignment/py_export.h, which the Cython
// module slam_py/install/pyvoldor_full.pyx declares via `cdef extern`.  It aligns N keyframes by their depth maps
// (and images) and fills the outputs as reference frame-alignment/py_export.cpp does, without Ceres: the solver runs
// on the device (voldor_b200/csrc/falign.cu, DESIGN.md §9).  Parameter names and documentation are this project's.
// Returns 0, a CUDA error code, or VB_FALIGN_EINVAL / VB_FALIGN_EDEBUG (include/voldor_b200.h) where the reference
// would exit(1) or open OpenCV windows.
#pragma once
#include "py_export.h"

extern VB_EXPORT int py_falign_wrapper(
    const float* depths,                 // [N][rows][cols]
    const float* images,                 // [N][rows][cols] or NULL (no photo consistency)
    const float* weights,                // [N][rows][cols] or NULL (= 1)
    float* poses_init,                   // [N][6] rvec, tvec camera -> world, or NULL (= 0)
    float* poses_ret,                    // [N][6]
    const int* connectivity,             // ref, tar, ref, tar, ..., -1; NULL = every ordered pair
    float* poses_covar,                  // [N][6][6], or [N][7][7] with optimize_7dof
    float* scaling_factor,               // [N] exp(log depth scale), 1 without optimize_7dof
    float* visibility_mat,               // [N][N], NaN where not connected
    float* consistency_mat,              // [N][N], NaN where not connected
    const int N,                         // 2 .. 64
    const int cols,
    const int rows,
    const float focal_x,
    const float focal_y,
    const float centre_x,
    const float centre_y,
    const float virtual_basefocal,
    const float colour_weight,           // photo consistency is on when images != NULL and colour_weight > 0
    const bool optimize_7dof,
    const bool graduated_optimize,       // accepted, no effect (as in the reference)
    const int stride,                    // sample every stride-th pixel in x and y
    const float consistency_residual_bound,
    const bool debug);                   // must be false
