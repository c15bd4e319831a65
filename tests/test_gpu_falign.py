"""Frame alignment on the device (voldor_b200.falign, csrc/falign.cu) against its host restatement
(oracle/host_falign.cpp) driven by this library's own per-sample evaluation: bit for bit, over 6/7-DoF, photo
consistency on/off, strides 1/3/4, 2/3/5 keyframes, default and partial connectivity, with and without weights and
initial poses.  Plus the per-sample bits of the solver's evaluation, determinism, execution contexts and a
slam_py-shaped call.  Needs no reference checkout."""
import ctypes as C
import itertools
import os
import threading

import numpy as np
import pytest

import falign_synth as fs
import ffi

pytestmark = pytest.mark.gpu
W, H = 64, 48
KEYS = ("poses_ret", "poses_covar", "scaling_factor", "visibility_mat", "consistency_mat")


@pytest.fixture(scope="module")
def vb():
    import voldor_b200

    voldor_b200.load_library()
    return voldor_b200


def _problem(N, seed, weights, init, partial):
    S = fs.scene(N, W, H, seed=seed, step=0.12)
    rng = np.random.default_rng(seed + 100)
    kw = dict(images=S["images"])
    kw["weights"] = rng.uniform(0.3, 1.0, S["depths"].shape).astype(np.float32) if weights else None
    kw["poses_init"] = fs.perturb(S["poses"], seed=seed) if init else None
    if partial:  # a chain, one link each way, plus one one-directional link back to frame 0
        conn = [0, 1, 1, 0] + sum([[i, i + 1] for i in range(1, N - 1)], []) + ([N - 1, 0] if N > 2 else []) + [-1]
        kw["connectivity"] = np.array(conn, np.int32)
    return S, kw


def _same(a, b, what):
    for k in KEYS:
        assert ffi.bits_equal(a[k], b[k]), f"{what}: {k} differs\n{a[k]}\n{b[k]}"
    assert a["iters"] == b["iters"] and a["reason"] == b["reason"], (what, a["iters"], b["iters"], a["reason"],
                                                                     b["reason"])


GRID = list(itertools.product([False, True], [False, True], [1, 3, 4], [2, 3, 5]))


@pytest.mark.parametrize("dof7,photo,stride,N", GRID)
def test_falign_equals_the_host_restatement(vb, dof7, photo, stride, N):
    i = GRID.index((dof7, photo, stride, N))
    weights, init, partial = bool(i & 1), bool(i & 2), bool(i & 4) or i % 3 == 0
    S, kw = _problem(N, i, weights, init, partial)
    if not photo:
        kw["images"] = None
    args = (S["depths"], S["fx"], S["fy"], S["cx"], S["cy"])
    opts = dict(vbf=60.0, crw=10.0, optimize_7dof=dof7, stride=stride, consistency_residual_bound=0.8, **kw)
    mine = vb.falign_ex(*args, **opts)
    want = fs.run_oracle("vb", *args, **opts)
    _same(mine, want, (dof7, photo, stride, N, weights, init, partial))
    assert mine["cost_init"] == want["cost_init"] and mine["cost_final"] == want["cost_final"]
    assert mine["iters"] >= 1


@pytest.mark.parametrize("stride,photo", list(itertools.product([1, 3, 4], [False, True])))
def test_solver_samples_equal_the_strided_evaluation(vb, stride, photo):
    N = 3
    S, kw = _problem(N, 7, True, True, False)
    args = (S["depths"], S["fx"], S["fy"], S["cx"], S["cy"])
    r = vb.falign_ex(*args, vbf=60.0, crw=10.0, stride=stride, samples=True, weights=kw["weights"],
                     poses_init=kw["poses_init"], images=S["images"] if photo else None)
    lib = ffi.ours()
    K = np.array([S["fx"], 0, S["cx"], 0, S["fy"], S["cy"], 0, 0, 1], np.float32)
    t_i, k1 = ffi._table(list(S["images"]))
    t_d, k2 = ffi._table(list(S["depths"]))
    t_w, k3 = ffi._table(list(kw["weights"]))
    assert lib.lib.vb_align_frame_init_gpu(t_i if photo else None, t_d, t_w, ffi._fp(K), C.c_float(60.0),
                                           C.c_float(10.0 if photo else 0.0), N, W, H) == 0
    ow, oh = -(-W // stride), -(-H // stride)
    p = 0
    for ref in range(N):
        for tar in range(N):
            if ref == tar:
                continue
            pr = np.zeros(9, np.float32)
            pt = np.zeros(9, np.float32)
            pr[:6], pt[:6] = kw["poses_init"][ref], kw["poses_init"][tar]
            res = np.zeros(ow * oh, np.float32)
            jac = np.zeros(ow * oh * 9, np.float32)
            assert lib.lib.vb_align_frame_eval_strided(ref, tar, ffi._fp(pr), ffi._fp(pt), ffi._fp(res), ffi._fp(jac),
                                                       1, stride) == 0
            assert ffi.bits_equal(r["samples_res"][p], res), (ref, tar)
            assert ffi.bits_equal(r["samples_jac"][p], jac.reshape(-1, 9)), (ref, tar)
            p += 1


def test_repeated_calls_give_identical_bits(vb):
    S, kw = _problem(3, 3, True, True, False)
    args = (S["depths"], S["fx"], S["fy"], S["cx"], S["cy"])
    a = vb.falign_ex(*args, vbf=60.0, stride=3, optimize_7dof=True, **kw)
    for _ in range(2):
        _same(vb.falign_ex(*args, vbf=60.0, stride=3, optimize_7dof=True, **kw), a, "repeat")


def test_four_contexts_run_concurrently_with_the_bits_of_a_sequential_run(vb):
    probs = [_problem(2 + (i % 3), 20 + i, i % 2 == 0, True, i == 3) for i in range(4)]

    def run(i):
        S, kw = probs[i]
        return vb.falign_ex(S["depths"], S["fx"], S["fy"], S["cx"], S["cy"], vbf=60.0, stride=3, **kw)

    seq = [run(i) for i in range(4)]
    got = [None] * 4

    def worker(i):
        vb.select_context(1 + i)
        got[i] = run(i)

    ts = [threading.Thread(target=worker, args=(i,)) for i in range(4)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    for i in range(4):
        _same(got[i], seq[i], f"context {1 + i}")


def test_window_after_falign_on_the_same_context_is_unchanged(vb):
    """the smoke() window, checked against its stored reference digests, after an alignment on context 0"""
    import oracle_host
    import refgold
    import synth

    S, kw = _problem(3, 5, True, True, False)
    vb.select_context(0)
    vb.falign(S["depths"], S["fx"], S["fy"], S["cx"], S["cy"], vbf=60.0, **kw)
    w, h, N = 96, 64, 3
    win = synth.make_window(w, h, N, seed=1)
    boot = (win["Rs"][0], win["ts"][0], synth.noisy_depth(win, 0.05))
    cfg = "--silent --max_iters 2 --no_trunc_iters 1000 --n_poses_to_sample 1024"
    args = (win["flows"], win["fx"], win["fy"], win["cx"], win["cy"])
    vb.set_bootstrap_override(*boot)
    ffi.libc_srand(1)
    mine = vb.voldor_ex(*args, config=cfg)
    vb.set_bootstrap_override()
    ffi.libc_srand(1)
    ref = refgold.reference(lambda: oracle_host.run_window("ref", *args, config=cfg, boot=boot), key="smoke")
    for k in ("poses", "depth", "depth_conf"):
        assert ffi.bits_equal(mine[k], ref[k]), k


def test_reference_abi_evaluation_is_untouched_by_falign(vb):
    S, kw = _problem(3, 9, True, True, False)
    lib = ffi.ours()
    K = np.array([S["fx"], 0, S["cx"], 0, S["fy"], S["cy"], 0, 0, 1], np.float32)
    assert lib.align_init(S["images"], S["depths"], kw["weights"], K, 40.0, 0.5) == 0
    p_ref = np.zeros(9, np.float32)
    p_tar = np.zeros(9, np.float32)
    p_tar[:6] = kw["poses_init"][1] - kw["poses_init"][0]
    before = lib.align_eval(0, 1, p_ref, p_tar, W, H, True)
    S2, kw2 = _problem(5, 11, False, True, False)
    vb.falign(S2["depths"], S2["fx"], S2["fy"], S2["cx"], S2["cy"], vbf=60.0, **kw2)
    after = lib.align_eval(0, 1, p_ref, p_tar, W, H, True)
    assert ffi.bits_equal(before[1], after[1]) and ffi.bits_equal(before[2], after[2])


def test_slam_py_shaped_call_converges(vb):
    """two keyframes at 640x480, stride 4, 7-DoF, images, crw=10, vbf = 5 * basefocal (as voldor_slam.py passes
    them); tolerances of tests/test_cpu_falign.py for 7-DoF.  The texture is fine enough to give the photometric term
    a slope at this resolution (with the coarse one the solve stops on the parameter tolerance ~0.011 rad away)."""
    S = fs.scene(2, 640, 480, seed=4, step=0.15, freq=10.0)
    init = fs.perturb(S["poses"], seed=4)
    basefocal = 0.1 * S["fx"]
    r = vb.falign_ex(S["depths"], S["fx"], S["fy"], S["cx"], S["cy"], weights=np.ones_like(S["depths"]),
                     poses_init=init, images=S["images"], optimize_7dof=True, stride=4, vbf=5 * basefocal, crw=10)
    s = r["scaling_factor"]
    e_rot, e_t = fs.relative_error(r["poses_ret"], S["poses"], 1, scale=1.0 / s[0])
    assert e_rot < 3e-3 and e_t < 2e-2, (e_rot, e_t, r["iters"], r["reason"])
    assert abs(s[1] / s[0] - 1) < 0.01
    assert r["poses_covar"].shape == (2, 7, 7) and np.all(np.linalg.matrix_rank(r["poses_covar"]) == 7)
