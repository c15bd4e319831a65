"""Time voldor_b200.falign on the three call shapes of slam_py's mapping thread, against the reference's data flow
in the same run: the host restatement (oracle/host_falign.cpp) driving the full-resolution align_frame_eval_gpu with
the full residual and Jacobian downloaded per evaluation (this library's kernel, and the reference's own kernels
when oracle/_ref is built).

    python tools/time_falign.py [--reps 5] [--out results/time_falign.json]

Prints one JSON object: GPU name and power limit, then per shape and path the median ms per call and the LM
iterations."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import falign_synth as fs  # noqa: E402
import ffi  # noqa: E402
import voldor_b200  # noqa: E402


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                      text=True).strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})", "unknown"


def shapes():
    w, h = 640, 480
    two = fs.scene(2, w, h, seed=4, step=0.15, freq=10.0)
    five = fs.scene(5, w, h, seed=5, step=0.1, freq=10.0)
    bf = 0.1 * two["fx"]
    local = dict(S=two, init=fs.perturb(two["poses"], seed=4),
                 calls=[dict(images=True, optimize_7dof=True, stride=4, vbf=5 * bf, crw=10)])
    loop = dict(S=two, init=fs.perturb(two["poses"], seed=6, rot=0.02, trans=0.06),
                calls=[dict(images=False, optimize_7dof=True, stride=3, vbf=5 * bf, crw=10),
                       dict(images=True, optimize_7dof=True, stride=3, vbf=5 * bf, crw=10)])
    multi = dict(S=five, init=fs.perturb(five["poses"], seed=5),
                 calls=[dict(images=True, optimize_7dof=False, stride=4, vbf=5 * bf, crw=10)])
    return {"local_link_2kf_s4_7dof_img": local, "loop_closure_2kf_s3_then_img": loop,
            "default_conn_5kf_s4_img": multi}


def run(path, shape):
    """one slam_py call sequence; returns (ms, iterations per call)"""
    S = shape["S"]
    poses = shape["init"]
    iters = []
    t0 = time.perf_counter()
    for c in shape["calls"]:
        kw = dict(c)
        kw["images"] = S["images"] if kw["images"] else None
        args = (S["depths"], S["fx"], S["fy"], S["cx"], S["cy"])
        if path == "falign":
            r = voldor_b200.falign_ex(*args, weights=np.ones_like(S["depths"]), poses_init=poses, **kw)
        else:
            backend, strided = {"oracle_full_vb": ("vb", False), "oracle_full_ref": ("ref", False)}[path]
            r = fs.run_oracle(backend, *args, weights=np.ones_like(S["depths"]), poses_init=poses, strided=strided,
                              **kw)
        poses = r["poses_ret"]
        iters.append(r["iters"])
    return (time.perf_counter() - t0) * 1e3, iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch

    torch.cuda.init()
    name, power = gpu_info()
    paths = ["falign", "oracle_full_vb"] + (["oracle_full_ref"] if os.path.exists(ffi.REF) else [])
    res = {"gpu": name, "power_limit": power, "reps": a.reps, "shapes": {}}
    for sname, shape in shapes().items():
        row = {}
        for p in paths:
            run(p, shape)  # warm-up: allocations, module load
            ms = []
            for _ in range(a.reps):
                t, iters = run(p, shape)
                ms.append(t)
            row[p] = {"ms_median": float(np.median(ms)), "ms_min": float(np.min(ms)), "iters": iters}
        res["shapes"][sname] = row
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(a.out), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
