"""Contraction sites of the quad-lane minimal solvers, settled ON THE DEVICE against the reference kernels.

Reading the reference's PTX leaves a handful of multi-use products next to an add/sub undecided (would ptxas fold a
copy of the product into an FFMA?  p3p_quad_math.cuh).  tests/p3p_device_probe.cu builds the product's solver headers
with those sites switchable at run time; here every assignment is run against the reference's own solve kernels on
8192 hypotheses: exactly one assignment may reproduce all of them bit for bit, and it must be the shipped one."""
import ctypes as C
import os

import numpy as np
import pytest

import ffi
import refgold
import synth

pytestmark = pytest.mark.gpu
PROBE = os.path.join(ffi.ROOT, "tests", "_build", "libp3p_probe.so")
FP = C.POINTER(C.c_float)


def _instances(w=160, h=120, N=4, seed=23):
    """the instances of camera 2 of a seeded window and the hypotheses the reference's solve kernels draw from them,
    as tests/make_golden.py stored them (p3p_hypotheses_160x120.npz) on the same inputs"""
    g = np.load(os.path.join(ffi.ROOT, "tests", "golden", "p3p_hypotheses_160x120.npz"))
    win = synth.make_window(w, h, N, seed=seed)
    assert int(g["seed"]) == seed and np.array_equal(g["K"], win["K"])
    return g


def _probe(lib, solver, mask, p2s, p3s, K, n_poses):
    rv = np.zeros((n_poses, 3), np.float32)
    tv = np.zeros((n_poses, 3), np.float32)
    rc = lib.probe_solve(solver, C.c_uint(mask), p2s.ctypes.data_as(FP), p3s.ctypes.data_as(FP), p2s.shape[0], n_poses,
                         C.c_float(K[0, 0]), C.c_float(K[1, 1]), C.c_float(K[0, 2]), C.c_float(K[1, 2]),
                         rv.ctypes.data_as(FP), tv.ctypes.data_as(FP))
    assert rc == 0
    return rv, tv


@pytest.mark.skipif(not os.path.exists(PROBE), reason="tests/_build/libp3p_probe.so not built (make probes)")
@pytest.mark.parametrize("solver,n_sites,exclusive", [(0, 9, ((2, 3), (5, 6))), (1, 10, ())])
def test_exactly_the_shipped_site_assignment_reproduces_the_reference(solver, n_sites, exclusive):
    lib = C.CDLL(PROBE)
    lib.probe_default_sites.restype = C.c_uint
    g = _instances()
    K, p2s, p3s = g["K"], np.ascontiguousarray(g["p2s"]), np.ascontiguousarray(g["p3s"])
    name = "ap3p" if solver == 1 else "lambdatwist"
    rv_ref, tv_ref = g[f"rvecs_{name}"], g[f"tvecs_{name}"]
    n_poses = rv_ref.shape[0]
    assert n_poses == 8192 and np.isfinite(tv_ref).all(1).sum() > 6000
    if refgold.LIVE:  # the stored hypotheses are what the reference's solve kernels draw
        rc, rv, tv = ffi.reference().solve_p3p(p3s, p2s, K, n_poses, ap3p=(solver == 1))
        assert rc == 0 and ffi.bits_equal(rv, rv_ref) and ffi.bits_equal(tv, tv_ref)
    shipped = lib.probe_default_sites(solver)
    perfect, best = [], (-1, None)
    for mask in range(1 << n_sites):
        if any((mask >> a) & 1 and (mask >> b) & 1 for a, b in exclusive):
            continue
        rv, tv = _probe(lib, solver, mask, p2s, p3s, K, n_poses)
        same = int(((rv.view(np.uint32) == rv_ref.view(np.uint32)) & (tv.view(np.uint32) == tv_ref.view(np.uint32))).all(1).sum())
        if same == n_poses:
            perfect.append(mask)
        if same > best[0]:
            best = (same, mask)
    os.makedirs(os.path.join(ffi.ROOT, "gpurun_out"), exist_ok=True)
    with open(os.path.join(ffi.ROOT, "gpurun_out", f"p3p_site_search_solver{solver}.txt"), "w") as f:
        f.write(f"solver {solver}: shipped {shipped:#x}, perfect assignments {[hex(m) for m in perfect]}, best {best}\n")
    assert perfect == [shipped], (solver, [hex(m) for m in perfect], hex(shipped), best)
