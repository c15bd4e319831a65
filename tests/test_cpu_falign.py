"""Frame alignment without a GPU: the host restatement (oracle/host_falign.cpp) over the CPU port recovers known
relative poses of synthetic keyframes, its covariance and scores match numpy, the shared LM step header matches
numpy, and the library refuses invalid arguments before touching the device.

Tolerances, chosen from these runs (160x120, stride 2, vbf 500, perturbation ~0.017 rad / 0.045):
rotation error of every relative pose < 3e-3 rad, translation error < 1.2e-2 (scene depth 2..6); with 7-DoF, where
the depth scales add a gauge freedom, translation error < 2e-2 and the recovered scale ratio within 1 %."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import falign_synth as fs
import ffi

W, H, STRIDE, VBF = 160, 120, 2, 500.0
ROT_TOL, TRANS_TOL, TRANS_TOL_7DOF = 3e-3, 1.2e-2, 2e-2

pytestmark = pytest.mark.skipif(not (os.path.exists(fs.ORACLE) and os.path.exists(fs.CPU)),
                                reason="oracle not built (make -C oracle all; make falign-oracle)")


@pytest.fixture(scope="module")
def scene():
    S = fs.scene(3, W, H, seed=0)
    S["init"] = fs.perturb(S["poses"])
    return S


def _run(S, **kw):
    kw.setdefault("poses_init", S["init"])
    return fs.run_oracle("cpu", S.pop("depths_override", S["depths"]), S["fx"], S["fy"], S["cx"], S["cy"],
                         stride=STRIDE, vbf=VBF, **kw)


def _check_relative(r, S, frames, scale=1.0, trans_tol=TRANS_TOL):
    for i in frames:
        e_rot, e_t = fs.relative_error(r["poses_ret"], S["poses"], i, scale=scale)
        e0_rot, e0_t = fs.relative_error(S["init"], S["poses"], i)
        assert e_rot < ROT_TOL and e_t < trans_tol, (i, e_rot, e_t, "from", e0_rot, e0_t)
        assert e_rot < e0_rot and e_t < e0_t


@pytest.mark.parametrize("photo", [False, True])
def test_converges_6dof_default_connectivity(scene, photo):
    r = _run(dict(scene), images=scene["images"] if photo else None)
    assert r["reason"] in (1, 2, 3), r["reason"]
    assert r["cost_final"] < 0.1 * r["cost_init"]
    _check_relative(r, scene, (1, 2))
    np.testing.assert_array_equal(r["scaling_factor"], 1)
    assert np.isnan(np.diag(r["visibility_mat"])).all() and (r["visibility_mat"][~np.eye(3, dtype=bool)] > 0.8).all()
    assert r["poses_covar"].shape == (3, 6, 6) and np.abs(r["poses_covar"]).max() > 0


def test_converges_7dof_and_recovers_a_depth_scale(scene):
    factor = 1.25
    S = dict(scene)
    S["depths_override"] = scene["depths"] * np.array([1, factor, 1], np.float32)[:, None, None]
    r = _run(S, optimize_7dof=True)
    s = r["scaling_factor"]
    assert abs(s[1] / s[0] * factor - 1) < 0.01 and abs(s[2] / s[0] - 1) < 0.01, s
    _check_relative(r, scene, (1, 2), scale=1.0 / s[0], trans_tol=TRANS_TOL_7DOF)
    assert r["poses_covar"].shape == (3, 7, 7)
    assert (r["poses_covar"][:, 6, :6] == 0).all() and (r["poses_covar"][:, 6, 6] > 0).all()


def test_one_directional_pair_keeps_the_other_pose_and_zero_covariance(scene):
    r = _run(dict(scene), connectivity=np.array([1, 0, -1], np.int32))
    np.testing.assert_array_equal(r["poses_ret"][0], scene["init"][0])
    np.testing.assert_array_equal(r["poses_ret"][2], scene["init"][2])
    e_rot, e_t = fs.relative_error(r["poses_ret"], scene["poses"], 1)
    assert e_rot < ROT_TOL and e_t < TRANS_TOL
    assert (r["poses_covar"] == 0).all()  # frames 0 and 2 have no parameter block: Covariance::Compute fails
    vis = r["visibility_mat"]
    assert np.isfinite(vis[1, 0]) and np.isnan(np.delete(vis.ravel(), 1 * 3 + 0)).all()


def _cpu_eval(S, params, stride, weights=True, photo=False):
    """per-pair per-sample residuals and Jacobians from the CPU port at the given per-frame parameters"""
    k = ffi.GpuKernels(fs.CPU, "cpu_")
    N = len(S["depths"])
    K = np.array([[S["fx"], 0, S["cx"], 0, S["fy"], S["cy"], 0, 0, 1]], np.float32)
    imgs = S["images"] if photo else np.zeros_like(S["depths"])
    assert k.align_init(imgs, S["depths"], np.ones_like(S["depths"]), K, VBF, 10.0 if photo else 0.0) == 0
    out = {}
    for ref in range(N):
        for tar in range(N):
            if ref != tar:
                rc, res, jac = k.align_eval(ref, tar, params[ref], params[tar], W, H, weights)
                out[ref, tar] = res[::stride, ::stride].reshape(-1), jac[::stride, ::stride].reshape(-1, 9)
    return out


def test_covariance_is_the_inverse_of_each_frame_block(scene):
    r = _run(dict(scene))
    p = np.zeros((3, 9), np.float32)
    p[:, :6] = r["poses_ret"]
    ev = _cpu_eval(scene, p, STRIDE)
    for f in range(3):
        Hm = np.zeros((6, 6))
        for (ref, tar), (res, jac) in ev.items():
            if ref == f:
                J = np.where(np.isfinite(res)[:, None], jac, 0).astype(np.float64)[:, :6]
                Hm += J.T @ J
        want = np.linalg.inv(Hm)
        np.testing.assert_allclose(r["poses_covar"][f], want, rtol=2e-6, atol=1e-7 * np.abs(want).max())


def test_scores_match_numpy_over_the_full_evaluation(scene):
    r = _run(dict(scene), consistency_residual_bound=0.5)
    p = np.zeros((3, 9), np.float32)
    p[:, :6] = r["poses_ret"]
    ev = _cpu_eval(scene, p, 1, weights=False)
    for (ref, tar), (res, _) in ev.items():
        fin = np.isfinite(res)
        n = int(fin.sum())
        vis = n / res.size
        b = 0.5
        cons = np.sum(1.0 - np.minimum(res[fin].astype(np.float64) ** 2, b) / b) / max(n, 1)
        assert r["visibility_mat"][ref, tar] == np.float32(vis)
        np.testing.assert_allclose(r["consistency_mat"][ref, tar], cons, rtol=1e-6)


# ---- the shared step header (voldor_b200/csrc/falign_math.h) -------------------------------------------------------
def _tri(i, j):
    return i * 9 - i * (i - 1) // 2 + (j - i)


@pytest.mark.parametrize("P", [6, 7, 9])
def test_damped_scaled_step_matches_numpy(P):
    L = fs.oracle()
    rng = np.random.default_rng(P)
    act = np.array(list(range(P)), np.int32)
    for trial in range(20):
        A = rng.normal(size=(9, 9)) * rng.uniform(0.1, 10, 9)
        Hf = A.T @ A + 1e-3 * np.eye(9)
        g = rng.normal(size=9)
        D = 1.0 / (1.0 + np.sqrt(np.diag(Hf)))
        radius = 10.0 ** rng.uniform(-3, 4)
        Hp = np.array([Hf[i, j] for i in range(9) for j in range(i, 9)])
        delta, m = np.zeros(9), C.c_double(0)
        ok = L.oracle_falign_frame_step(Hp.ctypes.data_as(fs.DP), g.ctypes.data_as(fs.DP), D.ctypes.data_as(fs.DP),
                                        act.ctypes.data_as(fs.IP), P, radius, delta.ctypes.data_as(fs.DP),
                                        C.byref(m))
        assert ok == 1
        Hs = (D[:P, None] * Hf[:P, :P]) * D[None, :P]
        gs = D[:P] * g[:P]
        Ad = Hs + np.diag(np.clip(np.diag(Hs), 1e-6, 1e32) / radius)
        ds = np.linalg.solve(Ad, -gs)
        np.testing.assert_allclose(delta[:P], D[:P] * ds, rtol=1e-8, atol=1e-12 * np.abs(ds).max())
        np.testing.assert_allclose(m.value, gs @ ds + 0.5 * ds @ Hs @ ds, rtol=1e-8)
    # a block that is not positive definite makes the step invalid
    Hp = np.zeros(45)
    Hp[_tri(0, 0)] = -1.0
    assert L.oracle_falign_frame_step(Hp.ctypes.data_as(fs.DP), np.ones(9).ctypes.data_as(fs.DP),
                                      np.ones(9).ctypes.data_as(fs.DP), act.ctypes.data_as(fs.IP), P, 1.0,
                                      np.zeros(9).ctypes.data_as(fs.DP), C.byref(C.c_double())) == 0


def test_trust_region_rules_and_tolerances():
    L = fs.oracle()

    def rules(cost, model, radius, dfac, cand):
        i = np.array([cost, model, radius, dfac, cand], np.float64)
        o = np.zeros(4)
        rc = L.oracle_falign_lm_rules(i.ctypes.data_as(fs.DP), o.ctypes.data_as(fs.DP))
        return rc, o

    # accepted: rho = 0.9 -> radius / max(1/3, 1 - (2 rho - 1)^3), decrease factor back to 2
    rc, o = rules(10.0, 1.0, 3.0, 8.0, 9.1)
    rho = 0.9 / 1.0
    assert o[2] == 1 and o[1] == 2.0 and o[3] == 1
    np.testing.assert_allclose(o[0], 3.0 / max(1 / 3, 1 - (2 * rho - 1) ** 3), rtol=1e-13)
    # accepted with rho ~ 0.5: radius unchanged
    rc, o = rules(10.0, 2.0, 3.0, 2.0, 9.0)
    np.testing.assert_allclose(o[0], 3.0, rtol=1e-13)
    # rejected (rho <= 1e-3): radius / decrease factor, decrease factor doubles
    rc, o = rules(10.0, 1.0, 3.0, 4.0, 10.5)
    assert o[2] == 0 and o[0] == 0.75 and o[1] == 8.0
    # function tolerance: |cost - candidate| <= 1e-6 cost stops before the step is judged
    rc, o = rules(10.0, 1.0, 3.0, 2.0, 10.0 - 5e-6)
    assert rc == 3 and o[3] == 0
    # minimum radius after a rejection
    rc, o = rules(10.0, 1.0, 1e-32, 2.0, 11.0)
    assert rc == 4


# ---- argument handling ---------------------------------------------------------------------------------------------
def _c_call(lib, N=3, conn=None, n_conn=-1, stride=4, debug=0):
    d = np.ones((max(N, 1), 8, 8), np.float32)
    outs = [np.zeros(64 * 64, np.float32) for _ in range(5)]
    f = lib.vb_py_falign_wrapper_ex
    P = lambda a: a.ctypes.data_as(fs.FP)  # noqa: E731
    c = None if conn is None else np.asarray(conn, np.int32)
    return f(P(d), None, None, None, P(outs[0]), None if c is None else c.ctypes.data_as(fs.IP), C.c_int(n_conn),
             P(outs[1]), P(outs[2]), P(outs[3]), P(outs[4]), N, 8, 8, C.c_float(5), C.c_float(5), C.c_float(4),
             C.c_float(4), C.c_float(100), C.c_float(0), 0, 0, stride, C.c_float(1), debug, None, None, None, None,
             None)


@pytest.mark.skipif(not os.path.exists(ffi.OURS), reason="libvoldor_b200.so not built (make lib)")
def test_invalid_arguments_are_refused_before_the_device():
    lib = C.CDLL(ffi.OURS)
    assert _c_call(lib, conn=[0, 3, -1], n_conn=3) == -1        # out of range
    assert _c_call(lib, conn=[0, -2, -1], n_conn=3) == -1
    assert _c_call(lib, conn=[0, 1, 1, 0], n_conn=4) == -1      # no terminator
    assert _c_call(lib, conn=[0, 1, 2], n_conn=3) == -1         # half a pair, no terminator
    assert _c_call(lib, N=1) == -1
    assert _c_call(lib, N=65) == -1
    assert _c_call(lib, stride=0) == -1
    assert _c_call(lib, debug=1) == -2


def test_python_binding_refuses_invalid_arguments():
    import voldor_b200

    d = np.ones((3, 8, 8), np.float32)
    for kw in (dict(connectivity=np.array([0, 3, -1])), dict(connectivity=np.array([0, 1, 1, 0])),
               dict(debug=True), dict(stride=0)):
        with pytest.raises(ValueError):
            voldor_b200.falign(d, 5, 5, 4, 4, **kw)
    with pytest.raises(ValueError):
        voldor_b200.falign(d[:1], 5, 5, 4, 4)


@pytest.mark.skipif(not os.path.exists(ffi.OURS), reason="libvoldor_b200.so not built (make lib)")
def test_py_falign_wrapper_has_the_reference_mangled_name():
    """frame-alignment/py_export.h declares it with C++ linkage; this is g++'s name for that declaration"""
    out = subprocess.check_output(["nm", "-D", "--defined-only", ffi.OURS], text=True)
    assert re.search(r"\b_Z17py_falign_wrapperPKfS0_S0_PfS1_PKiS1_S1_S1_S1_iiiffffffbbifb\b", out)
