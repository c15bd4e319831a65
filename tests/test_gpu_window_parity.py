"""GPU parity, window level: our device-resident pipeline (vb_py_voldor_wrapper) against the reference's own
kernels driven by the reference's host orchestration restated over the ABI (oracle/host_voldor.cpp), and
against our ABI entry points under that same orchestration.  Identical seeds, identical libc rand() stream."""
import json
import os

import numpy as np
import pytest

import ffi
import oracle_host
import refgold
import synth
import voldor_b200

pytestmark = pytest.mark.gpu
OUT = os.path.join(ffi.ROOT, "gpurun_out")


@pytest.fixture(autouse=True)
def _fresh_depth_rng():
    refgold.reseed_depth_rng()


def _report(rep):
    os.makedirs(OUT, exist_ok=True)
    with open(os.path.join(OUT, "parity_report.jsonl"), "a") as f:
        f.write(json.dumps(rep) + "\n")


def _compare(tag, a, b, exact=True):
    assert a["n_registered"] == b["n_registered"], (tag, a["n_registered"], b["n_registered"])
    assert a["iters"] == b["iters"]
    reps = []
    for k in ("poses", "poses_covar", "depth", "depth_conf"):
        rep = ffi.mismatch_report(a[k], b[k], f"{tag} {k}")
        _report(rep)
        reps.append(rep)
    for rep in reps:
        if exact:
            assert rep["bit_mismatch"] == 0, reps
        else:
            assert rep["frac_within_1e4"] > 0.99, reps


def _mono_case(w, h, N, iters, seed):
    win = synth.make_window(w, h, N, seed=seed)
    boot = (win["Rs"][0], win["ts"][0], synth.noisy_depth(win, 0.05))
    cfg = f"--silent --max_iters {iters} --no_trunc_iters 1000 --n_poses_to_sample 2048"
    return win, boot, cfg


@pytest.mark.parametrize("w,h,N,iters", [(96, 64, 3, 3), (160, 120, 4, 4)])
def test_mono_window_bit_exact(w, h, N, iters):
    win, boot, cfg = _mono_case(w, h, N, iters, seed=11)
    args = (win["flows"], win["fx"], win["fy"], win["cx"], win["cy"])
    # The per-pixel RNG streams of each library continue across windows (SURVEY §9 Q1) and our ABI path and our
    # resident path share one stream, so the three series are interleaved to keep both libraries at the same
    # point of their history: (ref#1, ours-abi#1) then (ref#2, ours-resident#2).
    ffi.libc_srand(77)
    ref1 = refgold.reference(lambda: oracle_host.run_window("ref", *args, config=cfg, boot=boot))
    ffi.libc_srand(77)
    abi1 = oracle_host.run_window("ours_abi", *args, config=cfg, boot=boot)
    assert ref1["n_registered"] == N
    _compare(f"window mono {w}x{h}x{N} abi-vs-ref", abi1, ref1)
    ffi.libc_srand(78)
    ref2 = refgold.reference(lambda: oracle_host.run_window("ref", *args, config=cfg, boot=boot))
    voldor_b200.set_bootstrap_override(*boot)
    ffi.libc_srand(78)
    mine2 = voldor_b200.voldor_ex(*args, config=cfg)
    voldor_b200.set_bootstrap_override()
    _compare(f"window mono {w}x{h}x{N} resident-vs-ref", mine2, ref2)


def test_prior_window_bit_exact():
    """depth-prior window (previous VOLDOR result as prior), default truncation behaviour"""
    w, h, N = 128, 96, 4
    win = synth.make_window(w, h, N, seed=21)
    prior = synth.noisy_depth(win, 0.02)[None]
    pose = np.zeros((1, 6), np.float32)
    cfg = "--silent --max_iters 4 --n_poses_to_sample 2048"
    args = (win["flows"], win["fx"], win["fy"], win["cx"], win["cy"])
    kw = dict(depth_priors=prior, depth_prior_poses=pose, config=cfg)
    ffi.libc_srand(5)
    ref = refgold.reference(lambda: oracle_host.run_window("ref", *args, **kw))
    ffi.libc_srand(5)
    mine = voldor_b200.voldor_ex(*args, **kw)
    assert ref["n_registered"] > 0
    _compare("window prior 128x96x4 resident-vs-ref", mine, ref)


def test_disparity_window_bit_exact():
    """stereo window: disparity prior 0 with disp_delta weighting (BASELINE config 3 shape, reduced)"""
    w, h, N = 207, 62, 3
    win = synth.make_window(w, h, N, seed=31)
    basefocal = float(0.54 * win["fx"])
    rng = np.random.default_rng(3)
    disp = (basefocal / win["depth_gt"] * (1 + rng.normal(0, 0.02, (h, w)))).astype(np.float32)
    disp[10:14, 20:60] = 0  # missing stereo matches
    cfg = "--silent --max_iters 3 --n_poses_to_sample 2048"
    args = (win["flows"], win["fx"], win["fy"], win["cx"], win["cy"])
    kw = dict(basefocal=basefocal, disparity=disp, config=cfg)
    ffi.libc_srand(6)
    ref = refgold.reference(lambda: oracle_host.run_window("ref", *args, **kw))
    ffi.libc_srand(6)
    mine = voldor_b200.voldor_ex(*args, **kw)
    assert ref["n_registered"] > 0
    _compare("window disparity 207x62x3 resident-vs-ref", mine, ref)


def test_mono_window_self_bootstrap_converges():
    """no override: the product's own essential-matrix bootstrap (reference geometry.cpp:267-332, OpenCV there)
    followed by the EM; functional check against the synthetic ground truth (poses up to the world scale)."""
    w, h, N = 320, 240, 5
    win = synth.make_window(w, h, N, seed=21)
    voldor_b200.set_bootstrap_override()
    r = voldor_b200.voldor(win["flows"], win["fx"], win["fy"], win["cx"], win["cy"],
                           config="--silent --max_iters 12 --no_trunc_iters 1000")
    assert r["n_registered"] == N
    t_gt = win["ts"].astype(np.float64)
    scale = N / np.linalg.norm(t_gt, axis=1).sum()  # voldor.cpp:309-317 world-scale normalisation
    for i in range(N):
        R = synth.rodrigues(r["poses"][i, :3])
        assert np.abs(R - win["Rs"][i]).max() < 3e-3, i
        assert np.linalg.norm(r["poses"][i, 3:] - t_gt[i] * scale) < 0.05, (i, r["poses"][i, 3:], t_gt[i] * scale)
    d_gt = win["depth_gt"] * scale
    rigid = r["depth_conf"] > 0.5
    assert rigid.mean() > 0.5
    assert np.median(np.abs(r["depth"][rigid] - d_gt[rigid]) / d_gt[rigid]) < 0.03


@pytest.mark.parametrize("name,w,h,N,iters,poses,kind", [
    ("C2", 640, 480, 8, 4, 8192, "mono"),
    ("C3", 1242, 375, 6, 3, 8192, "stereo"),
    ("C5", 1280, 960, 12, 2, 4096, "prior"),
])
def test_baseline_config_shapes_bit_exact(name, w, h, N, iters, poses, kind):
    """BASELINE.json configs[1], [2], [4] at their full image size / window length / hypothesis count (iteration
    count reduced so the reference kernels finish in seconds); resident pipeline vs reference kernels."""
    win = synth.make_window(w, h, N, seed=41)
    cfg = f"--silent --max_iters {iters} --no_trunc_iters 1000 --n_poses_to_sample {poses}"
    args = (win["flows"], win["fx"], win["fy"], win["cx"], win["cy"])
    kw, boot = dict(config=cfg), None
    if kind == "mono":
        boot = (win["Rs"][0], win["ts"][0], synth.noisy_depth(win, 0.05))
    elif kind == "stereo":
        basefocal = float(0.54 * win["fx"])
        rng = np.random.default_rng(3)
        disp = (basefocal / win["depth_gt"] * (1 + rng.normal(0, 0.02, (h, w)))).astype(np.float32)
        kw.update(basefocal=basefocal, disparity=disp)
    else:
        kw.update(depth_priors=synth.noisy_depth(win, 0.01)[None], depth_prior_poses=np.zeros((1, 6), np.float32))
    ffi.libc_srand(9)
    ref = refgold.reference(lambda: oracle_host.run_window("ref", *args, boot=boot, **kw))
    if boot:
        voldor_b200.set_bootstrap_override(*boot)
    ffi.libc_srand(9)
    mine = voldor_b200.voldor_ex(*args, **kw)
    voldor_b200.set_bootstrap_override()
    assert ref["n_registered"] == N
    _compare(f"window {name} {w}x{h}x{N} resident-vs-ref", mine, ref)


def test_c2_benchmarked_configuration_30_iterations_bit_exact():
    """exactly what bench.py times (BASELINE.json configs[1]: 640x480, 8 flows, 30 EM iterations, 8192 hypotheses,
    bench.py's seeds and flags): resident pipeline vs the reference kernels under the reference orchestration"""
    import bench

    win, boot = bench.make_inputs(0)
    args = (win["flows"], win["fx"], win["fy"], win["cx"], win["cy"])
    ffi.libc_srand(1000)
    ref = refgold.reference(lambda: oracle_host.run_window("ref", *args, config=bench.CONFIG, boot=boot))
    voldor_b200.set_bootstrap_override(*boot)
    ffi.libc_srand(1000)
    mine = voldor_b200.voldor_ex(*args, config=bench.CONFIG)
    voldor_b200.set_bootstrap_override()
    assert ref["n_registered"] == bench.NFLOWS and ref["iters"] == bench.EM_ITERS
    _compare("window C2 640x480x8 30 iterations (bench.py workload) resident-vs-ref", mine, ref)


@pytest.mark.parametrize("name", ["C3", "C5"])
def test_benchmarked_extra_configurations_full_iterations_bit_exact(name):
    """the `extra` lines of bench.py (BASELINE.json configs[2] and configs[4]) exactly as timed: full image size,
    window length, hypothesis count AND iteration count (C5: 1280x960, 12 flows, 50 EM iterations, depth prior)"""
    import bench

    win, kw, boot, cfg = bench.make_case(name)
    assert boot is None
    args = (win["flows"], win["fx"], win["fy"], win["cx"], win["cy"])
    ffi.libc_srand(2000)
    ref = refgold.reference(lambda: oracle_host.run_window("ref", *args, config=cfg, **kw))
    ffi.libc_srand(2000)
    mine = voldor_b200.voldor_ex(*args, config=cfg, **kw)
    c = bench.CASES[name]
    assert ref["n_registered"] == c["N"] and ref["iters"] == c["iters"]
    _compare(f"window {name} {c['w']}x{c['h']}x{c['N']} {c['iters']} iterations (bench.py extra) resident-vs-ref", mine, ref)


def test_c1_configuration_bit_exact():
    """BASELINE.json configs[0]: single 320x240 frame, 4 flows, 10 EM iterations, monocular"""
    w, h, N, iters = 320, 240, 4, 10
    win = synth.make_window(w, h, N, seed=43)
    boot = (win["Rs"][0], win["ts"][0], synth.noisy_depth(win, 0.05))
    cfg = f"--silent --max_iters {iters} --no_trunc_iters 1000 --n_poses_to_sample 8192"
    args = (win["flows"], win["fx"], win["fy"], win["cx"], win["cy"])
    ffi.libc_srand(12)
    ref = refgold.reference(lambda: oracle_host.run_window("ref", *args, config=cfg, boot=boot))
    voldor_b200.set_bootstrap_override(*boot)
    ffi.libc_srand(12)
    mine = voldor_b200.voldor_ex(*args, config=cfg)
    voldor_b200.set_bootstrap_override()
    assert ref["n_registered"] == N and ref["iters"] == iters
    _compare("window C1 320x240x4 10 iterations resident-vs-ref", mine, ref)


def test_vo_sequence_chained_windows_bit_exact():
    """A 10-flow sequence through the VO front-end (sliding windows, keyframe depth priors, covisibility steps):
    identical trajectories and identical per-window outputs from the product and from the reference kernels under
    the reference orchestration — covers RNG persistence across windows and priors built from own outputs."""
    from voldor_b200 import vo_frontend

    w, h, F = 160, 120, 10
    win = synth.make_window(w, h, F, seed=51)
    boot = (win["Rs"][0], win["ts"][0], synth.noisy_depth(win, 0.05))
    user = "--no_trunc_iters 1000 --n_poses_to_sample 2048 "
    outs = {"ref": [], "mine": []}

    def ref_solver(flows, fx, fy, cx, cy, **kw):
        first = kw.get("depth_priors") is None
        r = oracle_host.run_window("ref", flows, fx, fy, cx, cy, boot=boot if first else None, **kw)
        outs["ref"].append(r)
        return r

    def my_solver(flows, fx, fy, cx, cy, **kw):
        if kw.get("depth_priors") is None:
            voldor_b200.set_bootstrap_override(*boot)
        r = voldor_b200.voldor_ex(flows, fx, fy, cx, cy, **kw)
        voldor_b200.set_bootstrap_override()
        outs["mine"].append(r)
        return r

    def run_ref():
        ffi.libc_srand(31)
        vo_ref = vo_frontend.VisualOdometry(win["fx"], win["fy"], win["cx"], win["cy"], winsize=4, user_config=user,
                                            solver=ref_solver)
        return vo_ref.run(list(win["flows"])), outs["ref"]

    T_ref, outs["ref"] = refgold.reference(run_ref)
    ffi.libc_srand(31)
    vo_mine = vo_frontend.VisualOdometry(win["fx"], win["fy"], win["cx"], win["cy"], winsize=4, user_config=user,
                                         solver=my_solver)
    T_mine = vo_mine.run(list(win["flows"]))
    assert len(outs["ref"]) == len(outs["mine"]) >= 3
    for k, (a, b) in enumerate(zip(outs["mine"], outs["ref"])):
        _compare(f"vo sequence window {k}", a, b)
    assert len(T_ref) == len(T_mine) == F + 1
    for a, b in zip(T_mine, T_ref):
        assert ffi.bits_equal(a, b)
    # and the trajectory is the ground truth up to the monocular scale (loose: the point of this test is parity)
    gt = np.stack([np.concatenate([vo_frontend.matrix_to_rvec(win["Rs"][i]), win["ts"][i]]) for i in range(F)])
    T_gt = vo_frontend.formats.accumulate_poses(gt)
    scale = np.linalg.norm(T_mine[-1][:3, 3]) / np.linalg.norm(T_gt[-1][:3, 3])
    for a, b in zip(T_mine, T_gt):
        assert np.abs(a[:3, :3] - b[:3, :3]).max() < 5e-2
        assert np.linalg.norm(a[:3, 3] - b[:3, 3] * scale) < 0.25 * np.linalg.norm(T_mine[-1][:3, 3])


@pytest.mark.parametrize("flags", [
    "--lambdatwist 0",
    "--fb_smooth 0",
    "--optimize_depth 0",
    "--rg_refine_last_only 0",
    "--rg_refine 0",
    "--meanshift_max_init_trials 40",
    "--meanshift_max_init_trials 1 --meanshift_good_init_confidence 0.0001",
    "--norm_world_scale 0",
    "--depth_rand_samples 3 --depth_global_prop_step 1 --depth_local_prop_width 8",
    "--depth_global_prop_step 0 --depth_local_prop_width 0",
    "--no_trunc_iters 1 --trunc_rigidness_density 0.93",
    "--no_trunc_iters 1 --trunc_sample_density 0.02",
    "--exclusive_gpu_context 0",
    "--max_trace_on_flow 1 --rigidness_threshold 0.8",
    "--abs_resize_factor 0.5 --lambda 0.2 --meanshift_kernel_var 0.2",
    "--pose_sample_min_depth 6 --pose_sample_max_depth 9",
    "--meanshift_max_iters 3 --rg_max_iters 4",
    # beyond the exchange-free pool build (16384 hypotheses): cluster-wide compaction of the pose pool
    "--n_poses_to_sample 20000",
    # beyond 32768: the level-1 partial sums are exchanged through global memory instead of DSMEM
    "--n_poses_to_sample 40000",
])
def test_mono_window_flag_variants_bit_exact(flags):
    """configuration flags that switch code paths (solver, smoothing, truncation, start-sample fallbacks, ...)"""
    w, h, N, iters = 112, 80, 4, 4
    win, boot, _ = _mono_case(w, h, N, iters, seed=61)
    cfg = f"--silent --max_iters {iters} --n_poses_to_sample 1536 {flags}"
    args = (win["flows"], win["fx"], win["fy"], win["cx"], win["cy"])
    libc = __import__("ctypes").CDLL(None)
    ffi.libc_srand(90)
    ref, next_ref = refgold.reference(lambda: (oracle_host.run_window("ref", *args, config=cfg, boot=boot),
                                               libc.rand()))
    voldor_b200.set_bootstrap_override(*boot)
    ffi.libc_srand(90)
    mine = voldor_b200.voldor_ex(*args, config=cfg)
    next_mine = libc.rand()
    voldor_b200.set_bootstrap_override()
    _compare(f"window flags [{flags}]", mine, ref)
    # both sides must also have consumed the same number of libc rand() draws
    assert next_mine == next_ref


def test_mono_window_with_nonfinite_flow_pixels_bit_exact():
    """NaN / inf in the input flows (failed optical-flow regions): every kernel must degrade exactly like the
    reference's (NaN through the bilinear fetch, fmaxf/fminf clamps, strict comparisons)"""
    w, h, N, iters = 112, 80, 4, 3
    win, boot, _ = _mono_case(w, h, N, iters, seed=71)
    flows = win["flows"].copy()
    flows[0, 10:15, 20:26, :] = np.nan
    flows[1, 40, 50, 0] = np.inf
    flows[2, 60:62, 70:75, 1] = -np.inf
    flows[3, 5, 5, :] = 1e30
    cfg = f"--silent --max_iters {iters} --no_trunc_iters 1000 --n_poses_to_sample 1536"
    args = (flows, win["fx"], win["fy"], win["cx"], win["cy"])
    ffi.libc_srand(91)
    ref = refgold.reference(lambda: oracle_host.run_window("ref", *args, config=cfg, boot=boot))
    voldor_b200.set_bootstrap_override(*boot)
    ffi.libc_srand(91)
    mine = voldor_b200.voldor_ex(*args, config=cfg)
    voldor_b200.set_bootstrap_override()
    assert ref["n_registered"] >= 1  # the reference itself drops the cameras whose pose pool is poisoned
    _compare("window mono with non-finite flow pixels", mine, ref)


def test_reference_cython_module_over_this_library_bit_exact():
    """The reference's own, unmodified pyvoldor_vo.pyx (built by integration/build_cython_binding.py against
    libvoldor_b200.so) called exactly like slam_py/voldor_slam.py:447-457 does, against the reference kernels under
    the reference orchestration."""
    import glob
    import sys

    built = glob.glob(os.path.join(ffi.ROOT, "integration", "_build", "pyvoldor_vo*.so"))
    if not built:
        pytest.skip("integration/_build/pyvoldor_vo*.so not built (needs the reference checkout at build time)")
    sys.path.insert(0, os.path.dirname(built[0]))
    import pyvoldor_vo

    w, h, N, iters = 128, 96, 4, 3
    win, boot, _ = _mono_case(w, h, N, iters, seed=81)
    cfg = f"--silent --max_iters {iters} --no_trunc_iters 1000 --n_poses_to_sample 2048"
    ffi.libc_srand(92)
    ref = refgold.reference(lambda: oracle_host.run_window("ref", win["flows"], win["fx"], win["fy"], win["cx"],
                                                           win["cy"], config=cfg, boot=boot))
    voldor_b200.set_bootstrap_override(*boot)
    ffi.libc_srand(92)
    py_voldor_kwargs = {"flows": win["flows"], "fx": float(win["fx"]), "fy": float(win["fy"]), "cx": float(win["cx"]),
                        "cy": float(win["cy"]), "basefocal": 0.0, "disparity": None, "depth_priors": None,
                        "depth_prior_pconfs": None, "depth_prior_poses": None, "config": cfg}
    mine = pyvoldor_vo.voldor(**py_voldor_kwargs)
    voldor_b200.set_bootstrap_override()
    assert mine["n_registered"] == ref["n_registered"] == N
    for k in ("poses", "poses_covar", "depth", "depth_conf"):
        assert ffi.bits_equal(np.asarray(mine[k]), ref[k]), k
