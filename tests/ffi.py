"""ctypes front-end over the library-level boundary (gpu_kernels.h) of either build:
   ours   : voldor_b200/libvoldor_b200.so, C symbols prefixed vb_
   oracle : oracle/_ref/libgpu_kernels_ref.so (the reference's own .cu files for sm_100a), prefix ref_
Both expose the same argument lists, so the parity tests drive them with identical call histories."""
import ctypes as C
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OURS = os.path.join(ROOT, "voldor_b200", "libvoldor_b200.so")
REF = os.path.join(ROOT, "oracle", "_ref", "libgpu_kernels_ref.so")

FP = C.POINTER(C.c_float)
FPP = C.POINTER(FP)
IP = C.POINTER(C.c_int)


def _fp(a):
    if a is None:
        return None
    assert a.dtype == np.float32 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(FP)


def _table(arrs):
    """array of row pointers (float* h_x[]) or NULL"""
    if arrs is None:
        return None, None
    keep = [np.ascontiguousarray(a, np.float32) for a in arrs]
    t = (FP * len(keep))(*[k.ctypes.data_as(FP) for k in keep])
    return t, keep


class GpuKernels:
    def __init__(self, path, prefix):
        self.lib = C.CDLL(path, mode=C.RTLD_LOCAL)
        self.prefix = prefix
        f = self._f("optimize_depth_gpu")
        f.restype = C.c_int
        f.argtypes = [FPP] * 7 + [FP, FP, FP] + [FPP] * 4 + [C.c_float] + [C.c_int] * 4 + [C.c_float] + \
            [C.c_int] * 3 + [C.c_float] * 4 + [C.c_int, C.c_float, C.c_float, C.c_float, C.c_int]
        f = self._f("collect_p3p_instances")
        f.restype = C.c_int
        f.argtypes = [FPP, FPP, FP, FP, FPP, FPP, FP, FP] + [C.c_int] * 4 + [C.c_float] * 4 + [C.c_int]
        for n in ("solve_batch_p3p_lambdatwist_gpu", "solve_batch_p3p_ap3p_gpu"):
            f = self._f(n)
            f.restype = C.c_int
            f.argtypes = [FP] * 5 + [C.c_int] * 2
        f = self._f("meanshift_gpu")
        f.restype = C.c_int
        f.argtypes = [FP, C.c_float, FP, FP, IP, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.c_float]
        f = self._f("fit_robust_gaussian")
        f.restype = C.c_int
        f.argtypes = [FP, FP, FP, C.c_float, C.c_float, FP, IP, C.c_int, C.c_int, C.c_float, C.c_int]
        try:
            f = self._f("align_frame_init_gpu")
            f.restype = C.c_int
            f.argtypes = [FPP, FPP, FPP, FP, C.c_float, C.c_float, C.c_int, C.c_int, C.c_int]
            f = self._f("align_frame_eval_gpu")
            f.restype = C.c_int
            f.argtypes = [C.c_int, C.c_int, FP, FP, FP, FP, C.c_int]
        except AttributeError:
            pass
        try:
            f = self._f("gblur_gpu")
            f.restype = C.c_int
            f.argtypes = [FP, FP, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int]
        except AttributeError:
            pass

    def _f(self, name):
        return getattr(self.lib, self.prefix + name)

    # ------------------------------------------------------------------------------------------
    def optimize_depth(self, w, h, N, N_dp=0, flows=None, rig=None, depth=None, K=None, Rs=None, ts=None,
                       priors=None, pconfs=None, confs=None, dp_Rs=None, dp_ts=None, out_depth=True, out_rig=True,
                       out_confs=True, abs_rf=1.0, basefocal=0.0, n_rand=10, gstep=8, lwidth=32, lam=0.15,
                       omega=0.15, disp_delta=-1.0, delta=0.5, fb_smooth=True, fb_emm=0.5, fb_nc=0.9,
                       range_factor=1.0, rigidness_only=False):
        t_fl, k1 = _table(flows)
        t_rg, k2 = _table(rig)
        t_R, k3 = _table(Rs)
        t_t, k4 = _table(ts)
        t_dp, k5 = _table(priors)
        t_pc, k6 = _table(pconfs)
        t_cf, k7 = _table(confs)
        t_dR, k8 = _table(dp_Rs)
        t_dt, k9 = _table(dp_ts)
        o_depth = np.zeros((h, w), np.float32) if out_depth else None
        o_rig = np.zeros((N, h, w), np.float32) if (out_rig and N > 0) else None
        o_conf = np.zeros((N_dp, h, w), np.float32) if (out_confs and N_dp > 0) else None
        t_or = (FP * N)(*[o_rig[f].ctypes.data_as(FP) for f in range(N)]) if o_rig is not None else None
        t_oc = (FP * N_dp)(*[o_conf[f].ctypes.data_as(FP) for f in range(N_dp)]) if o_conf is not None else None
        d = None if depth is None else np.ascontiguousarray(depth, np.float32)
        Kc = None if K is None else np.ascontiguousarray(K, np.float32)
        rc = self._f("optimize_depth_gpu")(
            t_fl, t_rg, t_or, t_dp, t_pc, t_cf, t_oc, _fp(d), _fp(o_depth), _fp(Kc), t_R, t_t, t_dR, t_dt,
            abs_rf, N, N_dp, w, h, basefocal, n_rand, gstep, lwidth, lam, omega, disp_delta, delta,
            int(fb_smooth), fb_emm, fb_nc, range_factor, int(rigidness_only))
        return rc, o_depth, o_rig, o_conf

    def collect(self, w, h, N, active_idx, flows=None, rig=None, depth=None, K=None, Rs=None, ts=None,
                rig_thresh=0.5, rig_sum_thresh=1.0, min_depth=0.1, max_depth=1000.0, max_trace=3):
        t_fl, k1 = _table(flows)
        t_rg, k2 = _table(rig)
        t_R, k3 = _table(Rs)
        t_t, k4 = _table(ts)
        d = None if depth is None else np.ascontiguousarray(depth, np.float32)
        Kc = None if K is None else np.ascontiguousarray(K, np.float32)
        p2 = np.zeros((h, w, 2), np.float32)
        p3 = np.zeros((h, w, 3), np.float32)
        rc = self._f("collect_p3p_instances")(t_fl, t_rg, _fp(d), _fp(Kc), t_R, t_t, _fp(p2), _fp(p3), N, w, h,
                                              active_idx, rig_thresh, rig_sum_thresh, min_depth, max_depth,
                                              max_trace)
        return rc, p2, p3

    def solve_p3p(self, p3s, p2s, K, n_poses, ap3p=False):
        p3s = np.ascontiguousarray(p3s, np.float32)
        p2s = np.ascontiguousarray(p2s, np.float32)
        Kc = np.ascontiguousarray(K, np.float32)
        rv = np.zeros((n_poses, 3), np.float32)
        tv = np.zeros((n_poses, 3), np.float32)
        name = "solve_batch_p3p_ap3p_gpu" if ap3p else "solve_batch_p3p_lambdatwist_gpu"
        rc = self._f(name)(_fp(p3s), _fp(p2s), _fp(rv), _fp(tv), _fp(Kc), p3s.shape[0], n_poses)
        return rc, rv, tv

    def meanshift(self, space, kernel_var, mean, external_init, eps=1e-5, max_iters=100, max_trials=20,
                  good_conf=0.5):
        space = np.ascontiguousarray(space, np.float32)
        io_mean = np.ascontiguousarray(mean, np.float32).copy()
        conf = C.c_float(0)
        used = C.c_int(0)
        rc = self._f("meanshift_gpu")(_fp(space), kernel_var, _fp(io_mean), C.byref(conf), C.byref(used),
                                      int(external_init), space.shape[0], space.shape[1], eps, max_iters,
                                      max_trials, good_conf)
        return rc, io_mean, conf.value, used.value

    def fit_robust_gaussian(self, space, mean, covar, trunc_sigma=3.0, reg_lambda=0.001, eps=1e-5, max_iters=100):
        space = np.ascontiguousarray(space, np.float32)
        io_mean = np.ascontiguousarray(mean, np.float32).copy()
        io_cov = np.ascontiguousarray(covar, np.float32).copy()
        dens = C.c_float(-1)
        used = C.c_int(-1)
        rc = self._f("fit_robust_gaussian")(_fp(space), _fp(io_mean), _fp(io_cov), trunc_sigma, reg_lambda,
                                            C.byref(dens), C.byref(used), space.shape[0], space.shape[1], eps,
                                            max_iters)
        return rc, io_mean, io_cov, dens.value, used.value

    def align_init(self, images, depths, weights, K, vbf, crw):
        N, h, w = images.shape
        t_i, k1 = _table(list(images))
        t_d, k2 = _table(list(depths))
        t_w, k3 = _table(list(weights))
        Kc = np.ascontiguousarray(K, np.float32)
        return self._f("align_frame_init_gpu")(t_i, t_d, t_w, _fp(Kc), vbf, crw, N, w, h)

    def align_eval(self, ref_fid, tar_fid, p_ref, p_tar, w, h, apply_weights=True):
        pr = np.ascontiguousarray(p_ref, np.float32)
        pt = np.ascontiguousarray(p_tar, np.float32)
        res = np.zeros((h, w), np.float32)
        jac = np.zeros((h, w, 9), np.float32)
        rc = self._f("align_frame_eval_gpu")(ref_fid, tar_fid, _fp(pr), _fp(pt), _fp(res), _fp(jac),
                                             int(apply_weights))
        return rc, res, jac


    def gblur(self, src, sigma, ksize=0):
        """src: [depth, h, w] float32 -> (rc, blurred)"""
        src = np.ascontiguousarray(src, np.float32)
        d, h, w = src.shape
        dst = np.full_like(src, -7.0)
        rc = self._f("gblur_gpu")(_fp(src), _fp(dst), w, h, d, sigma, ksize)
        return rc, dst


def ours():
    return GpuKernels(OURS, "vb_")


def reference():
    return GpuKernels(REF, "ref_")


def libc_srand(seed):
    """both builds draw the mean-shift start samples from the process-wide libc rand() (SURVEY §9 Q13)"""
    C.CDLL(None).srand(C.c_uint(seed))


def bits_equal(a, b):
    """b: an array, or a reference result kept as a digest (tests/refgold.py)"""
    if hasattr(b, "matches"):
        return b.matches(a)
    a = np.ascontiguousarray(a)
    b = np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def mismatch_report(a, b, name=""):
    a = np.asarray(a)
    if hasattr(b, "matches"):  # digest of a reference result: equal or not, no per-element figures
        same = b.matches(a)
        return dict(name=name, n=int(a.size), bit_mismatch=0 if same else None, against="golden digest",
                    nan_pattern_equal=b.nan_matches(a), max_rel=0.0 if same else None,
                    frac_within_1e4=1.0 if same else None)
    b = np.asarray(b)
    neq = a.view(np.uint32) != b.view(np.uint32)
    n = int(neq.sum())
    both_nan = np.isnan(a) & np.isnan(b)
    with np.errstate(all="ignore"):
        rel = np.abs(a.astype(np.float64) - b) / np.maximum(np.abs(b.astype(np.float64)), 1e-30)
    rel = np.where(both_nan, 0, rel)
    rel = np.where(np.isnan(rel), np.inf, rel)
    return dict(name=name, n=int(a.size), bit_mismatch=n, frac_bit_mismatch=n / max(1, a.size),
                nan_pattern_equal=bool(np.array_equal(np.isnan(a), np.isnan(b))),
                max_rel=float(rel.max()) if rel.size else 0.0,
                frac_within_1e4=float((rel <= 1e-4).mean()) if rel.size else 1.0)
