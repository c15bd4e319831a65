"""GPU parity, function level: every library entry point of ours against the reference's own kernels
(oracle/_ref, rebuilt for sm_100a) driven with identical call histories through the same ABI.
Bar (north_star): bit-exact P3P instance maps / indices; <= 1e-4 relative on depth/rigidness/pose floats.
We assert the stronger bit-exact property wherever the pipeline is decision-driven."""
import json
import os

import numpy as np
import pytest

import ffi
import refgold
import synth

pytestmark = pytest.mark.gpu

OUT = os.path.join(ffi.ROOT, "gpurun_out")


@pytest.fixture(scope="module")
def libs():
    """(ours, the reference kernels); the second is None where oracle/_ref is absent (refgold)"""
    return ffi.ours(), (ffi.reference() if refgold.LIVE else None)


@pytest.fixture(autouse=True)
def _fresh_depth_rng():
    refgold.reseed_depth_rng()


def _report(rep):
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, "parity_report.jsonl"), "a") as f:
        f.write(json.dumps(rep) + "\n")


def _depth_sequence(lib, win, depth0, Rs, ts, n_calls=3, **kw):
    """call history of the host: first call uploads everything, later calls pass NULL (cached) inputs
    except the poses (reference: voldor/voldor.cpp:250-290)"""
    w, h, N = win["w"], win["h"], win["N"]
    outs = []
    ones = np.ones((N, h, w), np.float32)
    rc, d, r, _ = lib.optimize_depth(w, h, N, flows=list(win["flows"]), rig=list(ones), depth=depth0, K=win["K"],
                                     Rs=list(Rs), ts=list(ts), **kw)
    assert rc == 0
    outs.append((d, r))
    for it in range(1, n_calls):
        rc, d, r, _ = lib.optimize_depth(w, h, N, Rs=list(Rs), ts=list(ts), **kw)
        assert rc == 0
        outs.append((d, r))
    return outs


@pytest.mark.parametrize("w,h,N", [(64, 48, 3), (160, 120, 4), (320, 240, 4)])
def test_optimize_depth_bit_exact(libs, w, h, N):
    mine, ref = libs
    win = synth.make_window(w, h, N, seed=w)
    depth0 = synth.noisy_depth(win)
    Rs, ts = synth.perturbed_poses(win)
    a = _depth_sequence(mine, win, depth0, Rs, ts)
    b = refgold.reference(lambda: _depth_sequence(ref, win, depth0, Rs, ts))
    for it, ((da, ra), (db, rb)) in enumerate(zip(a, b)):
        rep_d = ffi.mismatch_report(da, db, f"optimize_depth[{w}x{h}x{N}] call{it} depth")
        rep_r = ffi.mismatch_report(ra, rb, f"optimize_depth[{w}x{h}x{N}] call{it} rigidness")
        _report(rep_d), _report(rep_r)
        assert rep_d["bit_mismatch"] == 0, rep_d
        assert rep_r["bit_mismatch"] == 0, rep_r


def test_optimize_depth_variants(libs):
    """no fb-smoothing, step-1 global propagation, odd sizes, rigidness-only update"""
    mine, ref = libs
    win = synth.make_window(75, 53, 2, seed=5)
    depth0 = synth.noisy_depth(win)
    Rs, ts = synth.perturbed_poses(win)
    for kw in (dict(fb_smooth=False), dict(gstep=1, lwidth=7), dict(n_rand=3, gstep=0), dict(lwidth=0),
               dict(rigidness_only=True), dict(abs_rf=0.5, lam=0.3, range_factor=2.0)):
        a = _depth_sequence(mine, win, depth0, Rs, ts, n_calls=2, **kw)
        b = refgold.reference(lambda: _depth_sequence(ref, win, depth0, Rs, ts, n_calls=2, **kw))
        for it, ((da, ra), (db, rb)) in enumerate(zip(a, b)):
            rep_d = ffi.mismatch_report(da, db, f"optimize_depth variant {kw} call{it} depth")
            rep_r = ffi.mismatch_report(ra, rb, f"optimize_depth variant {kw} call{it} rigidness")
            _report(rep_d), _report(rep_r)
            assert rep_d["bit_mismatch"] == 0, rep_d
            assert rep_r["bit_mismatch"] == 0, rep_r


def _route_sequence(lib, route):
    """depth steps whose likelihood-term counts pick the different launch shapes of the search and the propagation"""
    if route == "no_terms":
        # a step with neither flows nor priors (every cost INF: the depth must stay, the random streams advance),
        # then a two-flow step continuing on the same streams and the cached depth
        win = synth.make_window(56, 40, 2, seed=21)
        rc, d0, _, _ = lib.optimize_depth(56, 40, 0, depth=synth.noisy_depth(win), K=win["K"])
        assert rc == 0
        Rs, ts = synth.perturbed_poses(win)
        rc, d1, r1, _ = lib.optimize_depth(56, 40, 2, flows=list(win["flows"]), rig=list(np.ones((2, 40, 56))),
                                           Rs=list(Rs), ts=list(ts))
        assert rc == 0
        return d0, d1, r1
    if route in ("one_flow", "eight_flows_gstep1"):
        N, kw = (1, {}) if route == "one_flow" else (8, dict(gstep=1))
        win = synth.make_window(68, 44, N, seed=22 + N)
        Rs, ts = synth.perturbed_poses(win)
        return [x for dr in _depth_sequence(lib, win, synth.noisy_depth(win), Rs, ts, n_calls=2, **kw) for x in dr]
    assert route == "sixteen_flows_sixteen_priors"
    w, h, N = 36, 28, 16
    win = synth.make_window(w, h, N, seed=23)
    Rs, ts = synth.perturbed_poses(win)
    priors = [synth.noisy_depth(win, 0.02, seed=30 + p) for p in range(N)]
    for p, prior in enumerate(priors):
        prior[p:p + 3, 2 * p:2 * p + 5] = 0
    pconfs = [np.full((h, w), 0.5 + 0.03 * p, np.float32) for p in range(N)]
    confs = [np.ones((h, w), np.float32)] * N
    dp_Rs, dp_ts = synth.perturbed_poses(win, 0.001, 0.01, seed=31)
    kw = dict(basefocal=50.0, disp_delta=1.0)
    rc, d1, r1, c1 = lib.optimize_depth(w, h, N, N, flows=list(win["flows"]), rig=list(np.ones((N, h, w), np.float32)),
                                        depth=synth.noisy_depth(win), K=win["K"], Rs=list(Rs), ts=list(ts),
                                        priors=priors, pconfs=pconfs, confs=confs, dp_Rs=list(dp_Rs),
                                        dp_ts=list(dp_ts), **kw)
    assert rc == 0
    rc, d2, r2, c2 = lib.optimize_depth(w, h, N, N, Rs=list(Rs), ts=list(ts), **kw)
    assert rc == 0
    return d1, r1, c1, d2, r2, c2


@pytest.mark.parametrize("route", ["no_terms", "one_flow", "eight_flows_gstep1", "sixteen_flows_sixteen_priors"])
def test_optimize_depth_term_counts(libs, route):
    """no likelihood term at all, one, eight with step-1 global propagation, and the most a step takes (16 + 16)"""
    mine, ref = libs
    a = _route_sequence(mine, route)
    b = refgold.reference(lambda: _route_sequence(ref, route))
    assert len(a) == len(b)
    for k, (x, y) in enumerate(zip(a, b)):
        rep = ffi.mismatch_report(x, y, f"optimize_depth {route} out{k}")
        _report(rep)
        assert rep["bit_mismatch"] == 0, rep


def test_optimize_depth_with_priors(libs):
    mine, ref = libs
    w, h, N = 96, 64, 3
    win = synth.make_window(w, h, N, seed=9)
    Rs, ts = synth.perturbed_poses(win)
    prior = synth.noisy_depth(win, 0.02, seed=4)
    prior[5:9, 7:30] = 0  # holes: confidence must stay untouched there (Q19)
    pconf = np.full((h, w), 0.8, np.float32)
    conf = np.ones((h, w), np.float32)
    I = np.eye(3, dtype=np.float32)
    z = np.zeros(3, np.float32)

    def run(lib, disp_delta):
        # prior-only fusion first (N = 0; reference: voldor/voldor.cpp:116), then the full step twice
        rc, d0, _, c0 = lib.optimize_depth(w, h, 0, 1, depth=prior, K=win["K"], priors=[prior], pconfs=[pconf],
                                           confs=[conf], dp_Rs=[I], dp_ts=[z], basefocal=50.0,
                                           disp_delta=disp_delta)
        assert rc == 0
        ones = np.ones((N, h, w), np.float32)
        rc, d1, r1, c1 = lib.optimize_depth(w, h, N, 1, flows=list(win["flows"]), rig=list(ones), depth=d0,
                                            K=win["K"], Rs=list(Rs), ts=list(ts), priors=[prior],
                                            pconfs=[pconf], confs=list(c0), dp_Rs=[I], dp_ts=[z],
                                            basefocal=50.0, disp_delta=disp_delta)
        assert rc == 0
        rc, d2, r2, c2 = lib.optimize_depth(w, h, N, 1, Rs=list(Rs), ts=list(ts), basefocal=50.0,
                                            disp_delta=disp_delta)
        assert rc == 0
        return d0, c0, d1, r1, c1, d2, r2, c2

    for disp_delta in (-1.0, 1.0):
        outs = [run(mine, disp_delta), refgold.reference(lambda: run(ref, disp_delta))]
        for k, (x, y) in enumerate(zip(*outs)):
            rep = ffi.mismatch_report(x, y, f"optimize_depth priors disp_delta={disp_delta} out{k}")
            _report(rep)
            assert rep["bit_mismatch"] == 0, rep


def _collect_inputs(w, h, N, seed):
    win = synth.make_window(w, h, N, seed=seed)
    rng = np.random.default_rng(seed + 100)
    rig = rng.uniform(0.2, 1.0, (N, h, w)).astype(np.float32)
    depth = synth.noisy_depth(win, 0.01)
    return win, rig, depth


@pytest.mark.parametrize("w,h,N", [(64, 48, 3), (320, 240, 5)])
def test_collect_p3p_bit_exact(libs, w, h, N):
    mine, ref = libs
    win, rig, depth = _collect_inputs(w, h, N, 3)
    Rs, ts = synth.perturbed_poses(win)

    def run(lib, active):
        if active == 0:
            rc, p2, p3 = lib.collect(w, h, N, active, flows=list(win["flows"]), rig=list(rig), depth=depth,
                                     K=win["K"], Rs=list(Rs), ts=list(ts))
        else:  # cached inputs, only the poses travel (reference: voldor/geometry.cpp:51-58)
            rc, p2, p3 = lib.collect(w, h, N, active, Rs=list(Rs), ts=list(ts))
        assert rc == 0
        return p2, p3

    for active in range(N):
        outs = [run(mine, active), refgold.reference(lambda: run(ref, active))]
        for k, (x, y) in enumerate(zip(*outs)):
            rep = ffi.mismatch_report(x, y, f"collect[{w}x{h}x{N}] active={active} map{k}")
            _report(rep)
            assert rep["bit_mismatch"] == 0, rep
        assert np.isfinite(outs[0][0]).any(), "collector found no instances at all"


def _instance_maps(lib, w, h, N, seed, active):
    win, rig, depth = _collect_inputs(w, h, N, seed)
    rc, p2, p3 = lib.collect(w, h, N, active, flows=list(win["flows"]), rig=list(rig), depth=depth, K=win["K"],
                             Rs=list(win["Rs"]), ts=list(win["ts"]))
    assert rc == 0
    return win, p2, p3


@pytest.mark.parametrize("ap3p", [False, True])
def test_solve_batch_p3p(libs, ap3p):
    mine, ref = libs
    # the instances the reference collects (ours collects the same bits)
    win, p2, p3 = _instance_maps(mine, 160, 120, 3, 7, 1)
    p2_ref, p3_ref = refgold.reference(lambda: _instance_maps(ref, 160, 120, 3, 7, 1)[1:])
    assert ffi.bits_equal(p2, p2_ref) and ffi.bits_equal(p3, p3_ref)
    ok = np.isfinite(p2.sum(-1) + p3.sum(-1))
    p2s, p3s = p2[ok], p3[ok]
    assert p2s.shape[0] > 1000
    n_poses = 4096
    rc1, rv1, tv1 = mine.solve_p3p(p3s, p2s, win["K"], n_poses, ap3p)
    rc2, rv2, tv2 = refgold.reference(lambda: ref.solve_p3p(p3s, p2s, win["K"], n_poses, ap3p),
                                      sample=(512 if ap3p else 128, 1))
    assert rc1 == 0 and rc2 == 0
    name = "ap3p" if ap3p else "lambdatwist"
    rep_r = ffi.mismatch_report(rv1, rv2, f"solve_batch_{name} rvec")
    rep_t = ffi.mismatch_report(tv1, tv2, f"solve_batch_{name} tvec")
    _report(rep_r), _report(rep_t)
    assert rep_r["nan_pattern_equal"] and rep_t["nan_pattern_equal"]
    (rv1, rv2), (tv1, tv2) = refgold.sampled(rv1, rv2), refgold.sampled(tv1, tv2)
    assert np.isfinite(rv2).all(axis=1).mean() > 0.5
    # north_star tolerance: 1e-4 relative on pose floats (measured against the pose magnitude)
    fin = np.isfinite(rv2).all(1) & np.isfinite(tv2).all(1)
    scale_r = np.maximum(np.linalg.norm(rv2[fin], axis=1, keepdims=True), 1e-3)
    scale_t = np.maximum(np.linalg.norm(tv2[fin], axis=1, keepdims=True), 1e-3)
    assert (np.abs(rv1[fin] - rv2[fin]) / scale_r).max() <= 1e-4
    assert (np.abs(tv1[fin] - tv2[fin]) / scale_t).max() <= 1e-4
    if not ap3p:
        assert rep_r["bit_mismatch"] == 0 and rep_t["bit_mismatch"] == 0, (rep_r, rep_t)


def _pose_pool(n, seed, outliers=0.3):
    rng = np.random.default_rng(seed)
    mode = np.array([0.05, -0.1, 0.02, 0.02, 0.01, 0.25], np.float32)
    pool = mode + rng.normal(0, 0.02, (n, 6)).astype(np.float32)
    k = int(outliers * n)
    pool[:k] = rng.uniform(-1, 1, (k, 6)).astype(np.float32)
    rng.shuffle(pool)
    return pool.astype(np.float32), mode


@pytest.mark.parametrize("n", [1, 7, 300, 512, 513, 5000, 8192])
def test_meanshift_bit_exact(libs, n):
    mine, ref = libs
    pool, mode = _pose_pool(n, n)
    for external in (True, False):
        init = (mode + 0.05).astype(np.float32)
        ffi.libc_srand(1234)
        res = [mine.meanshift(pool, 0.1, init, external)]
        ffi.libc_srand(1234)
        res.append(refgold.reference(lambda: ref.meanshift(pool, 0.1, init, external)))
        (rc1, m1, c1, u1), (rc2, m2, c2, u2) = res
        assert rc1 == 0 and rc2 == 0
        rep = ffi.mismatch_report(m1, m2, f"meanshift n={n} external={external} mean")
        rep["iters"] = (u1, u2)
        rep["conf"] = (c1, c2)
        _report(rep)
        assert u1 == u2, rep
        assert rep["bit_mismatch"] == 0, rep
        assert np.float32(c1).view(np.uint32) == np.float32(c2).view(np.uint32), rep


@pytest.mark.parametrize("n", [300, 5000, 8192])
def test_fit_robust_gaussian_bit_exact(libs, n):
    mine, ref = libs
    pool, mode = _pose_pool(n, n + 1)
    pool = (pool * 100).astype(np.float32)
    mean0 = (mode * 100).astype(np.float32)
    cov0 = (np.eye(6) * 0.1 * 100 * 100).astype(np.float32)
    res = [mine.fit_robust_gaussian(pool, mean0, cov0),
           refgold.reference(lambda: ref.fit_robust_gaussian(pool, mean0, cov0))]
    (rc1, m1, v1, d1, u1), (rc2, m2, v2, d2, u2) = res
    assert rc1 == rc2
    rep_m = ffi.mismatch_report(m1, m2, f"robust_fit n={n} mean")
    rep_v = ffi.mismatch_report(v1, v2, f"robust_fit n={n} covar")
    rep_m["iters"] = (u1, u2)
    rep_m["density"] = (d1, d2)
    _report(rep_m), _report(rep_v)
    assert u1 == u2 and d1 == d2
    assert rep_m["bit_mismatch"] == 0 and rep_v["bit_mismatch"] == 0, (rep_m, rep_v)


def test_fit_robust_gaussian_unreliable(libs):
    """singular start covariance -> both report 'unreliable' (1) and leave the outputs untouched (Q15)"""
    mine, ref = libs
    pool, mode = _pose_pool(200, 3)
    cov0 = np.zeros((6, 6), np.float32)
    for rc, m, v, d, u in (mine.fit_robust_gaussian(pool, mode, cov0),
                           refgold.reference(lambda: ref.fit_robust_gaussian(pool, mode, cov0))):
        assert rc == 1
        assert ffi.bits_equal(mode, m) and ffi.bits_equal(cov0, v)


def _align_inputs(w, h, N, seed):
    rng = np.random.default_rng(seed)
    win = synth.make_window(w, h, N, seed=seed)
    depths = np.stack([win["depth_gt"] * (1 + 0.02 * i) for i in range(N)]).astype(np.float32)
    yy, xx = np.mgrid[0:h, 0:w]
    images = np.stack([0.5 + 0.3 * np.sin(xx / 9.0 + i) * np.cos(yy / 7.0) for i in range(N)]).astype(np.float32)
    weights = rng.uniform(0.5, 1.0, (N, h, w)).astype(np.float32)
    return win, images, depths, weights


@pytest.mark.parametrize("crw", [0.0, 0.5])
def test_align_frame_parity(libs, crw):
    """frame-alignment residual/Jacobian (SURVEY §8a row 10): identical NaN pattern, <= 1e-4 relative"""
    mine, ref = libs
    w, h, N = 96, 64, 3
    win, images, depths, weights = _align_inputs(w, h, N, 13)
    p_ref = np.array([0.01, -0.02, 0.005, 0.05, 0.02, 0.1, 0.01, 0.02, -0.01], np.float32)
    p_tar = np.array([-0.005, 0.01, 0.0, 0.0, 0.01, -0.05, 0.0, -0.01, 0.02], np.float32)

    def run(lib):
        assert lib.align_init(images, depths, weights, win["K"], 40.0, crw) == 0
        rc, res, jac = lib.align_eval(0, 1, p_ref, p_tar, w, h, True)
        assert rc == 0
        rc, res2, jac2 = lib.align_eval(2, 0, np.zeros(9, np.float32), p_tar, w, h, False)
        assert rc == 0
        return res, jac, res2, jac2

    outs = [run(mine), refgold.reference(lambda: run(ref), sample=(256, 2))]
    for k, (a, b) in enumerate(zip(*outs)):
        rep = ffi.mismatch_report(a, b, f"align_frame crw={crw} out{k}")
        _report(rep)
        assert rep["nan_pattern_equal"], rep
        a, b = refgold.sampled(a, b)
        fin = np.isfinite(b)
        scale = np.maximum(np.abs(b[fin]), 1e-3 * np.abs(b[fin]).max())
        assert (np.abs(a[fin] - b[fin]) / scale).max() <= 1e-4, rep
    assert refgold.isfinite(outs[1][0]).mean() > 0.5


@pytest.mark.parametrize("w,h,depth,sigma,ksize", [
    (96, 64, 3, 1.5, 0),      # default kernel size = max(ceil(6 sigma), 3)
    (75, 53, 2, 0.8, 0),      # odd image sizes
    (33, 17, 1, 2.0, 7),      # explicit kernel size, image narrower than two blocks
    (40, 300, 1, 40.0, 0),    # half width 121: taps reach far past both borders (renormalisation)
    (5, 4, 2, 3.0, 0),        # kernel wider than the image
])
def test_gblur_bit_exact(libs, w, h, depth, sigma, ksize):
    """separable border-renormalised Gaussian (reference gpu-kernels/gblur.cu:12-72, reached through
    oracle/ref_shim/ref_gblur.cu): same taps, same accumulation order, IEEE division -> identical bits"""
    mine, ref = libs
    rng = np.random.default_rng(w * 1000 + h)
    src = rng.uniform(-2, 5, (depth, h, w)).astype(np.float32)
    rc1, a = mine.gblur(src, sigma, ksize)
    rc2, b = refgold.reference(lambda: ref.gblur(src, sigma, ksize))
    assert rc1 == 0 and rc2 == 0
    rep = ffi.mismatch_report(a, b, f"gblur {w}x{h}x{depth} sigma={sigma} ksize={ksize}")
    _report(rep)
    assert rep["bit_mismatch"] == 0, rep
    # and it is a blur: constant images are fixed points, the mean is roughly preserved
    rc, c = mine.gblur(np.full((1, h, w), 3.25, np.float32), sigma, ksize)
    assert rc == 0 and np.abs(c - 3.25).max() < 1e-5


def test_gblur_rejects_oversized_kernel(libs):
    """half width > 128 -> cudaErrorInvalidFilterSetting on both sides (gblur.cu:56-57)"""
    mine, ref = libs
    src = np.zeros((1, 8, 8), np.float32)
    rc1, _ = mine.gblur(src, 50.0, 0)
    rc2, _ = refgold.reference(lambda: ref.gblur(src, 50.0, 0))
    assert rc1 == rc2 != 0


def test_align_frame_strided_output_equals_the_full_evaluation(libs):
    """packed every-stride-th-sample mode (what frame-alignment/align_frame_cost_fun.h:183-229 consumes) against the
    full evaluation of the reference kernels subsampled on the host the way the cost function does it"""
    import ctypes as C
    mine, ref = libs
    w, h, N = 100, 70, 3
    win, images, depths, weights = _align_inputs(w, h, N, 17)
    p_ref = np.array([0.01, -0.02, 0.005, 0.05, 0.02, 0.1, 0.01, 0.02, -0.01], np.float32)
    p_tar = np.array([-0.005, 0.01, 0.0, 0.0, 0.01, -0.05, 0.0, -0.01, 0.02], np.float32)
    assert mine.align_init(images, depths, weights, win["K"], 40.0, 0.5) == 0
    rc, res_full, jac_full = mine.align_eval(0, 1, p_ref, p_tar, w, h, True)
    assert rc == 0
    f = mine.lib.vb_align_frame_eval_strided
    f.argtypes = [C.c_int, C.c_int, ffi.FP, ffi.FP, ffi.FP, ffi.FP, C.c_int, C.c_int]
    for stride in (1, 4, 16):
        ow, oh = -(-w // stride), -(-h // stride)
        res = np.full((oh, ow), -7, np.float32)
        jac = np.full((oh, ow, 9), -7, np.float32)
        assert f(0, 1, ffi._fp(p_ref), ffi._fp(p_tar), ffi._fp(res), ffi._fp(jac), 1, stride) == 0
        assert ffi.bits_equal(res, res_full[::stride, ::stride])
        assert ffi.bits_equal(jac, jac_full[::stride, ::stride])
    # and the full evaluation itself is the reference's (tolerance level, see test_align_frame_parity)
    def run_ref():
        assert ref.align_init(images, depths, weights, win["K"], 40.0, 0.5) == 0
        return ref.align_eval(0, 1, p_ref, p_tar, w, h, True)

    rc, res_r, jac_r = refgold.reference(run_ref)
    assert ffi.mismatch_report(res_full, res_r)["nan_pattern_equal"]


def test_rvec_to_matrix_identical_on_host_and_device():
    """the pipelined camera loop converts poses on the device, the oracle orchestration on the host: same source,
    every operation individually rounded, own sin/cos -> identical bits (csrc/host_math.h)"""
    import ctypes as C
    lib = C.CDLL(ffi.OURS)
    rng = np.random.default_rng(0)
    r = np.concatenate([rng.normal(0, s, (4000, 3)) for s in (1e-20, 1e-6, 0.01, 0.3, 1.5, 10.0)]).astype(np.float32)
    r[0] = 0
    n = r.shape[0]
    Rd, Rh = np.zeros((n, 9), np.float32), np.zeros((n, 9), np.float32)
    fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))
    assert lib.vb_debug_rvec_to_matrix(fp(r), n, fp(Rd), fp(Rh)) == 0
    assert ffi.bits_equal(Rd, Rh)
    # and it is a rotation by |r| about r
    R = Rh.reshape(n, 3, 3).astype(np.float64)
    assert np.abs(R @ R.transpose(0, 2, 1) - np.eye(3)).max() < 1e-6
    k = 5000
    want = synth.rodrigues(r[k].astype(np.float64))
    assert np.abs(R[k] - want).max() < 1e-6


@pytest.mark.parametrize("crw", [0.0, 0.5])
def test_cpu_align_frame_port_against_the_reference_kernels(libs, crw):
    """pins the CPU restatement of the frame alignment (oracle/cpu_kernels.cpp) to the reference's own kernels:
    same NaN pattern away from the validity borders, 1e-3 relative on residual and Jacobian (libm vs libdevice,
    emulated 8-bit texture weights)"""
    import oracle_host

    _, ref = libs
    cpu = ffi.GpuKernels(oracle_host.CPU, "cpu_")
    w, h, N = 96, 64, 3
    win, images, depths, weights = _align_inputs(w, h, N, 13)
    p_ref = np.array([0.01, -0.02, 0.005, 0.05, 0.02, 0.1, 0.01, 0.02, -0.01], np.float32)
    p_tar = np.array([-0.005, 0.01, 0.0, 0.0, 0.01, -0.05, 0.0, -0.01, 0.02], np.float32)

    def run(lib):
        assert lib.align_init(images, depths, weights, win["K"], 40.0, crw) == 0
        rc, res, jac = lib.align_eval(0, 1, p_ref, p_tar, w, h, True)
        assert rc == 0
        return res, jac

    (res_c, jac_c), (res_r, jac_r) = run(cpu), refgold.reference(lambda: run(ref), sample=(1024, 2))
    (res_c, res_r), (jac_c, jac_r) = refgold.sampled(res_c, res_r), refgold.sampled(jac_c, jac_r)
    assert (np.isnan(res_c) != np.isnan(res_r)).mean() < 0.01
    fin = np.isfinite(res_c) & np.isfinite(res_r)
    assert fin.mean() > 0.5
    assert (np.abs(res_c[fin] - res_r[fin]) <= 1e-3 * np.maximum(np.abs(res_r[fin]), 1e-3)).mean() > 0.99
    scale = np.maximum(np.abs(jac_r[fin]), 1e-3 * np.abs(jac_r[fin]).max())
    assert (np.abs(jac_c[fin] - jac_r[fin]) / scale <= 1e-3).mean() > 0.99
