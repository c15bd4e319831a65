"""Python binding of frame alignment, drop-in for the reference's `pyvoldor.falign`.

Mirrors reference slam_py/install/pyvoldor_full.pyx (falign): same argument names, defaults and returned dict
(`poses_ret (N,6)`, `poses_covar (N,6,6)` or `(N,7,7)` with optimize_7dof, `scaling_factor (N,)`,
`visibility_mat (N,N)`, `consistency_mat (N,N)`), so slam_py/voldor_slam.py can pass the same kwargs.  The solve
runs on the device (csrc/falign.cu) on the calling thread's execution context (select_context)."""
import ctypes as C

import numpy as np

from .pyvoldor_vo import load_library

FP = C.POINTER(C.c_float)
IP = C.POINTER(C.c_int)
DP = C.POINTER(C.c_double)

REASONS = {1: "gradient_tolerance", 2: "parameter_tolerance", 3: "function_tolerance", 4: "min_trust_region_radius",
           5: "max_iterations", 6: "invalid_steps"}
_EINVAL, _EDEBUG = -1, -2


def _bind():
    lib = load_library()
    f = lib.vb_py_falign_wrapper_ex
    if f.argtypes is None:
        f.restype = C.c_int
        f.argtypes = [FP, FP, FP, FP, FP, IP, C.c_int, FP, FP, FP, FP, C.c_int, C.c_int, C.c_int] + \
            [C.c_float] * 6 + [C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, IP, IP, DP, FP, FP]
    return f


def _stack(a, name, shape):
    if a is None:
        return None
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.shape != shape:
        raise ValueError(f"{name}: expected shape {shape}, got {a.shape}")
    return a


def _p(a, t=FP):
    return None if a is None else a.ctypes.data_as(t)


def falign_ex(depths, fx, fy, cx, cy, weights=None, images=None, poses_init=None, connectivity=None, vbf=1000,
              crw=10, optimize_7dof=False, graduated_optmize=False, stride=4, consistency_residual_bound=1.0,
              debug=False, samples=False):
    """falign() plus `iters` (LM iterations), `reason` (termination, see REASONS), `cost_init` / `cost_final`
    (1/2 sum of squared residuals), `stats_ms` = [total, upload + preparation, LM loop, covariance + scores +
    download]; with samples=True also `samples_res (pairs, n)` and `samples_jac (pairs, n, 9)`: the per-sample
    residuals and Jacobians of the first evaluation, n = ceil(w/stride) * ceil(h/stride)."""
    if debug:
        raise ValueError("falign: debug=True (OpenCV windows) is not supported")
    depths = np.ascontiguousarray(depths, dtype=np.float32)
    if depths.ndim != 3:
        raise ValueError(f"depths: expected (N, h, w), got shape {depths.shape}")
    N, h, w = depths.shape
    if not 2 <= N <= 64:
        raise ValueError(f"falign needs 2..64 frames, got {N}")
    if int(stride) < 1:
        raise ValueError(f"stride must be >= 1, got {stride}")
    weights = _stack(weights, "weights", (N, h, w))
    images = _stack(images, "images", (N, h, w))
    poses_init = _stack(poses_init, "poses_init", (N, 6))
    n_conn = -1
    npairs = N * (N - 1)
    if connectivity is not None:
        connectivity = np.ascontiguousarray(connectivity, dtype=np.int32).reshape(-1)
        n_conn = connectivity.size
        if n_conn == 0 or connectivity[-1] != -1 or (n_conn - 1) % 2 != 0 or np.any(connectivity[:-1] == -1):
            raise ValueError("connectivity must be ref, tar, ref, tar, ..., -1")
        if np.any(connectivity[:-1] < 0) or np.any(connectivity[:-1] >= N):
            raise ValueError(f"connectivity entry out of range 0..{N - 1}")
        if n_conn > 1:
            npairs = (n_conn - 1) // 2
    C7 = 7 if optimize_7dof else 6
    poses_ret = np.zeros((N, 6), np.float32)
    poses_covar = np.zeros((N, C7, C7), np.float32)
    scaling = np.zeros((N,), np.float32)
    vis = np.zeros((N, N), np.float32)
    cons = np.zeros((N, N), np.float32)
    iters, reason = C.c_int(0), C.c_int(0)
    costs = np.zeros(2, np.float64)
    stats = np.zeros(4, np.float32)
    n = -(-w // int(stride)) * -(-h // int(stride))
    dump = np.zeros(npairs * n * 10, np.float32) if samples else None
    rc = _bind()(_p(depths), _p(images), _p(weights), _p(poses_init), _p(poses_ret), _p(connectivity, IP), n_conn,
                 _p(poses_covar), _p(scaling), _p(vis), _p(cons), N, w, h, fx, fy, cx, cy, vbf, crw,
                 int(bool(optimize_7dof)), int(bool(graduated_optmize)), int(stride), consistency_residual_bound, 0,
                 C.byref(iters), C.byref(reason), _p(costs, DP), _p(stats), _p(dump))
    if rc in (_EINVAL, _EDEBUG):
        raise ValueError(f"falign: invalid input (code {rc})")
    if rc != 0:
        raise RuntimeError(f"falign failed with CUDA error {rc}")
    out = {"poses_ret": poses_ret, "poses_covar": poses_covar, "scaling_factor": scaling, "visibility_mat": vis,
           "consistency_mat": cons, "iters": iters.value, "reason": reason.value, "cost_init": float(costs[0]),
           "cost_final": float(costs[1]), "stats_ms": stats}
    if samples:
        out["samples_res"] = dump[:npairs * n].reshape(npairs, n)
        out["samples_jac"] = dump[npairs * n:].reshape(npairs, n, 9)
    return out


def falign(depths, fx, fy, cx, cy, weights=None, images=None, poses_init=None, connectivity=None, vbf=1000, crw=10,
           optimize_7dof=False, graduated_optmize=False, stride=4, consistency_residual_bound=1.0, debug=False):
    """Align N keyframes (camera -> world rvec/tvec poses) by their depth maps and, with images and crw > 0, their
    intensities.  Returns the reference's dict; see falign_ex for the solver report."""
    r = falign_ex(depths, fx, fy, cx, cy, weights, images, poses_init, connectivity, vbf, crw, optimize_7dof,
                  graduated_optmize, stride, consistency_residual_bound, debug)
    return {k: r[k] for k in ("poses_ret", "poses_covar", "scaling_factor", "visibility_mat", "consistency_mat")}
