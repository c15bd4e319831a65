"""The flag grammar and every default of this library's Config (csrc/config.h) against the reference's OWN struct Config:
voldor/config.h compiled unmodified (oracle/ref_shim/ref_config_probe.cpp against the OpenCV stand-in oracle/ref_shim/cv_min)
and driven exactly like voldor/py_export.cpp:15-25 drives it.  Covers the defaults, every flag one at a time, the
str_to_arg fall-through (fractional values given to integer fields), the value-less switches and realistic strings."""
import ctypes as C
import os

import numpy as np
import pytest

import ffi
import refgold

REF = os.path.join(ffi.ROOT, "oracle", "_ref", "libref_config.so")
LIVE = os.path.exists(REF)  # else the reference's values come from tests/golden (refgold)
pytestmark = pytest.mark.skipif(not os.path.exists(ffi.OURS), reason="libvoldor_b200.so not built")

NUMERIC = ["basefocal", "omega", "disp_delta", "delta", "rg_refine", "rg_refine_last_only", "rg_trunc_sigma",
           "rg_covar_reg_lambda", "rg_epsilon", "rg_max_iters", "rg_pose_scaling", "resize_factor", "abs_resize_factor",
           "fx", "fy", "cx", "cy", "viz_img_per_row", "viz_depth_scale", "exclusive_gpu_context", "lambda",
           "meanshift_kernel_var", "meanshift_rvec_scale", "norm_world_scale", "cpu_p3p", "lambdatwist",
           "max_trace_on_flow", "n_poses_to_sample", "pose_sample_min_depth", "pose_sample_max_depth",
           "rigidness_threshold", "rigidness_sum_threshold", "trunc_rigidness_density", "trunc_sample_density",
           "max_iters", "no_trunc_iters", "min_iters_after_trunc", "fb_smooth", "fb_emm", "fb_no_change_prob",
           "optimize_depth", "depth_rand_samples", "depth_global_prop_step", "depth_local_prop_width",
           "depth_range_factor", "meanshift_max_iters", "meanshift_max_init_trials", "meanshift_good_init_confidence",
           "meanshift_epsilon", "kitti_estimate_ground", "kitti_ground_holo_width", "kitti_ground_roi",
           "kitti_ground_meanshift_kernel_var"]


def _dump(lib, name, flags, intr=(400.0, 410.0, 320.5, 239.5, 216.0)):
    f = getattr(lib, name)
    f.restype = C.c_int
    f.argtypes = [C.c_char_p] + [C.c_float] * 5 + [C.POINTER(C.c_double)]
    out = np.full(80, np.nan)
    n = f(flags.encode(), *intr, out.ctypes.data_as(C.POINTER(C.c_double)))
    return out[:n]


@pytest.fixture(scope="module")
def libs():
    return C.CDLL(ffi.OURS), (C.CDLL(REF) if LIVE else None)


def _same(libs, flags):
    a = _dump(libs[0], "vb_debug_config_dump", flags)
    b = refgold.reference(lambda: _dump(libs[1], "ref_config_dump", flags), live=LIVE)
    assert len(a) == len(b) == 56
    if not LIVE:
        assert ffi.bits_equal(a, b), (flags, a)
        return
    assert np.array_equal(a, b), (flags, np.nonzero(a != b)[0], a[a != b], b[a != b])


def test_defaults_and_intrinsics(libs):
    _same(libs, "")
    _same(libs, "   ")


def test_every_numeric_flag_alone(libs):
    for k, name in enumerate(NUMERIC):
        for value in ("7", "0", "2.75", "-3.5", "1e-3"):  # fractional values reach integer fields through stod (Q16)
            _same(libs, f"--{name} {value}")


def test_switches_and_realistic_strings(libs):
    for flags in ("--silent", "--debug --silent", "--save_everything",
                  "--silent --meanshift_kernel_var 0.2 --delta 1.5 --max_iters 5",                    # voldor_slam.py:153
                  "--silent --meanshift_kernel_var 0.1 --disp_delta 1 --delta 0.2 --max_iters 4",      # voldor_slam.py:145
                  "--silent --max_iters 30 --no_trunc_iters 1000 --n_poses_to_sample 8192",           # bench.py
                  "--pose_sample_min_depth 0.54 --pose_sample_max_depth 54 --abs_resize_factor 0.5",  # set_cam_params
                  "--lambdatwist 0 --rg_refine_last_only 0 --fb_smooth 0 --optimize_depth 0 --norm_world_scale 0"):
        _same(libs, flags)
