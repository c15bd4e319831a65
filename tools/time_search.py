"""Search-kernel timing through the library's own CUDA-event profile (vb_profile_*), one C2 window."""
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import synth  # noqa: E402
import voldor_b200  # noqa: E402
from voldor_b200.pyvoldor_vo import load_library  # noqa: E402

win = synth.make_window(640, 480, 8, seed=100)
boot = (win["Rs"][0], win["ts"][0], synth.noisy_depth(win, 0.05, seed=7))
voldor_b200.set_bootstrap_override(*boot)
cfg = "--silent --max_iters 10 --no_trunc_iters 1000 --n_poses_to_sample 8192"
lib = load_library()
args = (win["flows"], win["fx"], win["fy"], win["cx"], win["cy"])
voldor_b200.voldor_ex(*args, config=cfg)
lib.vb_profile_enable(1)
r = voldor_b200.voldor_ex(*args, config=cfg)
ms, n = C.c_double(0), C.c_longlong(0)
lib.vb_profile_get(C.byref(ms), C.byref(n))
print("search ms/launch", ms.value / n.value, "launches", n.value,
      "window ms", r["stats_ms"][0])
