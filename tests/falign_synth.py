"""Synthetic keyframes for the frame-alignment tests: depth rendered analytically from the planes of a room (floor,
ceiling, three walls: no two parallel planes carry the whole view, so all 6 degrees of freedom are constrained),
a smooth texture for the images, known camera -> world poses; plus the ctypes front-end of
oracle/liboracle_falign.so (the host restatement of falign)."""
import ctypes as C
import os

import numpy as np

import ffi

ORACLE = os.path.join(ffi.ROOT, "oracle", "liboracle_falign.so")
CPU = os.path.join(ffi.ROOT, "oracle", "libvoldor_oracle.so")
FP = C.POINTER(C.c_float)
IP = C.POINTER(C.c_int)
DP = C.POINTER(C.c_double)

# n . X = c, world frame
PLANES = [((0, 1, 0), 1.2), ((0, -1, 0), 1.5), ((1, 0, 0), 2.0), ((-1, 0, 0), 2.5), ((0, 0.3, 1), 6.0)]


def rodrigues(r):
    r = np.asarray(r, np.float64)
    th = np.linalg.norm(r)
    if th < 1e-12:
        return np.eye(3)
    k = r / th
    Kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.eye(3) + np.sin(th) * Kx + (1 - np.cos(th)) * Kx @ Kx


def rvec_of(R):
    c = np.clip((np.trace(R) - 1) / 2, -1, 1)
    th = np.arccos(c)
    if th < 1e-12:
        return np.zeros(3)
    v = np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]]) / (2 * np.sin(th))
    return v * th


def texture(X, freq=1.0):
    """smooth intensity in [0, 1]; freq scales the spatial frequency (fine texture for large images, where a coarse
    one leaves the photometric term nearly flat per pixel)"""
    a = freq * X
    return 0.5 + 0.25 * np.sin(1.3 * a[..., 0] + 0.7 * a[..., 2]) + 0.25 * np.cos(1.1 * a[..., 1] - 0.9 * a[..., 2])


def render(pose, w, h, fx, fy, cx, cy, freq=1.0):
    """depth and image of a camera with camera -> world pose (rvec, t)"""
    R, t = rodrigues(pose[:3]), np.asarray(pose[3:], np.float64)
    xs, ys = np.meshgrid(np.arange(w, dtype=np.float64), np.arange(h, dtype=np.float64))
    d = np.stack([(xs - cx) / fx, (ys - cy) / fy, np.ones_like(xs)], -1)
    dw = d @ R.T
    depth = np.full((h, w), np.inf)
    for n, c in PLANES:
        n = np.asarray(n, np.float64)
        den = dw @ n
        with np.errstate(divide="ignore", invalid="ignore"):
            s = (c - n @ t) / den
        s = np.where((den > 1e-9) & (s > 0), s, np.inf)
        depth = np.minimum(depth, s)
    X = t + depth[..., None] * dw
    return depth.astype(np.float32), texture(X, freq).astype(np.float32)


def scene(N, w, h, seed=0, step=0.15, freq=1.0):
    """N keyframes along a short arc: poses (N,6) camera -> world, depths, images, intrinsics"""
    rng = np.random.default_rng(seed)
    fx = fy = 0.9 * w
    cx, cy = (w - 1) / 2.0, (h - 1) / 2.0
    poses = np.zeros((N, 6))
    for i in range(N):
        poses[i, :3] = np.array([0.02, -0.04, 0.015]) * i + rng.normal(0, 0.005, 3)
        poses[i, 3:] = np.array([step, -0.3 * step, 0.5 * step]) * i + rng.normal(0, 0.01, 3)
    dep, img = zip(*[render(p, w, h, fx, fy, cx, cy, freq) for p in poses])
    return dict(poses=poses.astype(np.float32), depths=np.stack(dep), images=np.stack(img), fx=fx, fy=fy, cx=cx,
                cy=cy, w=w, h=h)


def perturb(poses, seed=1, rot=0.01, trans=0.03):
    rng = np.random.default_rng(seed)
    p = poses.astype(np.float64).copy()
    p[:, :3] += rng.normal(0, rot, (len(p), 3))
    p[:, 3:] += rng.normal(0, trans, (len(p), 3))
    return p.astype(np.float32)


def relative(poses, i, j=0):
    """pose of camera i in camera j's frame: (R, t)"""
    Ri, ti = rodrigues(poses[i, :3]), np.asarray(poses[i, 3:], np.float64)
    Rj, tj = rodrigues(poses[j, :3]), np.asarray(poses[j, 3:], np.float64)
    return Rj.T @ Ri, Rj.T @ (ti - tj)


def relative_error(est, gt, i, j=0, scale=1.0):
    """rotation error (rad) and translation error of camera i relative to camera j; scale multiplies the estimate's
    translation (7-DoF: the estimate's world scale)"""
    Re, te = relative(est, i, j)
    Rg, tg = relative(gt, i, j)
    return float(np.linalg.norm(rvec_of(Re.T @ Rg))), float(np.linalg.norm(te * scale - tg))


# ---- oracle front-end -------------------------------------------------------------------------------------------
_lib = None


def oracle():
    global _lib
    if _lib is None:
        _lib = C.CDLL(ORACLE)
        _lib.oracle_falign_bind.argtypes = [C.c_char_p, C.c_char_p, C.c_int]
        _lib.oracle_falign.argtypes = [FP, FP, FP, FP, FP, IP, C.c_int, FP, FP, FP, FP, C.c_int, C.c_int, C.c_int] + \
            [C.c_float] * 6 + [C.c_int, C.c_int, C.c_float, IP, IP, DP, FP]
        _lib.oracle_falign_frame_step.argtypes = [DP, DP, DP, IP, C.c_int, C.c_double, DP, DP]
        _lib.oracle_falign_lm_rules.argtypes = [DP, DP]
    return _lib


def _p(a, t=FP):
    return None if a is None else a.ctypes.data_as(t)


def run_oracle(backend, depths, fx, fy, cx, cy, weights=None, images=None, poses_init=None, connectivity=None,
               vbf=1000, crw=10, optimize_7dof=False, stride=4, consistency_residual_bound=1.0, strided=True):
    """backend: "cpu" (CPU port) or "vb" (this library's evaluation); same dict as voldor_b200.falign_ex"""
    L = oracle()
    path, prefix = {"cpu": (CPU, b"cpu_"), "vb": (ffi.OURS, b"vb_"), "ref": (ffi.REF, b"ref_")}[backend]
    assert L.oracle_falign_bind(path.encode(), prefix, int(strided)) == 0
    f32 = lambda a: None if a is None else np.ascontiguousarray(a, np.float32)  # noqa: E731
    depths, weights, images, poses_init = f32(depths), f32(weights), f32(images), f32(poses_init)
    N, h, w = depths.shape
    n_conn = -1
    if connectivity is not None:
        connectivity = np.ascontiguousarray(connectivity, np.int32)
        n_conn = connectivity.size
    C7 = 7 if optimize_7dof else 6
    out = dict(poses_ret=np.zeros((N, 6), np.float32), poses_covar=np.zeros((N, C7, C7), np.float32),
               scaling_factor=np.zeros(N, np.float32), visibility_mat=np.zeros((N, N), np.float32),
               consistency_mat=np.zeros((N, N), np.float32))
    it, rs = C.c_int(0), C.c_int(0)
    costs = np.zeros(2)
    stats = np.zeros(4, np.float32)
    rc = L.oracle_falign(_p(depths), _p(images), _p(weights), _p(poses_init), _p(out["poses_ret"]),
                         _p(connectivity, IP), n_conn, _p(out["poses_covar"]), _p(out["scaling_factor"]),
                         _p(out["visibility_mat"]), _p(out["consistency_mat"]), N, w, h, fx, fy, cx, cy, vbf, crw,
                         int(optimize_7dof), stride, consistency_residual_bound, C.byref(it), C.byref(rs),
                         _p(costs, DP), _p(stats))
    assert rc == 0, rc
    out.update(iters=it.value, reason=rs.value, cost_init=float(costs[0]), cost_final=float(costs[1]),
               stats_ms=stats)
    return out
