#!/usr/bin/env python
"""bench.py — VOLDOR EM hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|cpu-port|abi-dropin]
                  [--inflight M] [--no-extras] [--no-cpu-baseline] [--dump-outputs DIR]

Workload (both arms, `config.workload`): BASELINE.json configs[1] — a single 640x480 frame with 8 flows, 30 EM
iterations, monocular (bootstrap pose/depth injected, BASELINE.md §3), 8192 pose hypotheses per camera, window
truncation disabled.  metric = EM iterations per second, whole job (all ranks).

One "step" = M independent VO windows solved concurrently on one GPU, one per execution context of the library
(csrc/context.h: each context owns what one reference worker process owns — the reference gets its concurrency from
a 6-worker process pool, slam_py/voldor_slam.py:182-191).  M = --inflight (default 8: the reference pool holds 6 workers; with 32
hardware work queues 8 windows are 3 % faster than 6 and 10 add nothing); `latency` in the JSON line reports the per-window latency in that regime and with one window in flight.  With N > 1 ranks each rank runs its own
independent windows (window-per-GPU, SURVEY §8e) and contributes the poses of its context-0 window to ONE NCCL
all_gather per step; "scaling": "weak".

  value : windows whose inputs already live in HBM when the timed region starts (device pointers are passed to the
          same C-ABI call; every bulk copy in the library is cudaMemcpyDefault)
  e2e   : the same call with pinned HOST buffers: H2D of the flows and D2H of poses/covariances/depth/confidence are
          inside the timed region.  `e2e_pageable`: one window at a time through the reference-facing C++ symbol
          py_voldor_wrapper (what pyvoldor_vo.pyx binds) with pageable numpy buffers, exactly like slam_py calls it.
  roofline : dominant kernel = fused cost + random depth search, algorithmic bytes W*H*(12N+60) per launch (flows
             8N, rigidness weights 4N, depth r/w 8, cost w 4, XORWOW state r/w 48; DESIGN.md) over its CUDA-event
             duration measured live in the library (vb_profile_*), against MEASURED_PEAKS.json
  cpu_baseline : the CPU port (oracle/cpu_kernels.cpp, OpenMP) under the restated reference orchestration on a
             bounded sample (same window, 2 EM iterations)
  parity_checked : outside the timed region the first window of context 0 is bit-compared with the reference kernels
             (oracle/_ref) run on the same input from the same fresh state
  extra : the other single-GPU BASELINE configs (C1 with the CPU restatement timed beside it, C3, C5), one window in
          flight, each with its own roofline figures

--dump-outputs DIR writes what the last timed step returned for each window in flight (rank 0), as float32
DIR/ctx<k>_{poses,poses_covar,depth,depth_conf}.npy: the arrays voldor() returns, poses cut to the registered frames.
The inputs are seeded, so two builds run with the same arguments can be compared output for output.

--impl reference runs the REFERENCE arm: the reference's own CUDA kernels (oracle/_ref, its unmodified .cu files
rebuilt for sm_100a) driven by the reference's host orchestration restated OpenCV-free over the ABI
(oracle/host_voldor.cpp) — i.e. voldor.cpp's geometry loop on the host cores calling its gpu-kernels library, which
is the only implementation of this path the reference has (SURVEY §0: there is no CPU E/M step in the reference).
--impl cpu-port times the CPU port instead; --impl abi-dropin times the same reference host orchestration over THIS
library's gpu_kernels.h entry points (what a maintainer gets by only re-linking).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# hardware work queues for the windows in flight (voldor_b200/csrc/context.cu); must be set before CUDA is initialised
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# the benchmarked configuration (BASELINE.json configs[1])
W, H, NFLOWS, EM_ITERS, NPOSES = 640, 480, 8, 30, 8192
CONFIG = f"--silent --max_iters {EM_ITERS} --no_trunc_iters 1000 --n_poses_to_sample {NPOSES}"
WORKLOAD = (f"BASELINE configs[1]: single {W}x{H} frame, {NFLOWS} flows, {EM_ITERS} EM iters, monocular (injected "
            f"bootstrap), {NPOSES} hypotheses/camera, truncation off")

# the other single-GPU configurations of BASELINE.json (extra lines; C4 = the --gpus 8 run of C2)
CASES = {
    "C1": dict(w=320, h=240, N=4, iters=10, P=8192, kind="mono", seed=43,
               what="configs[0]: single 320x240 frame, 4 flows, 10 EM iters, monocular"),
    "C2": dict(w=W, h=H, N=NFLOWS, iters=EM_ITERS, P=NPOSES, kind="mono", seed=100, what=WORKLOAD),
    "C3": dict(w=1242, h=375, N=6, iters=5, P=8192, kind="stereo", seed=41,
               what="configs[2]: KITTI-shape 1242x375, 6 flows, stereo-prior depth init (5 EM iters = the reference default)"),
    "C5": dict(w=1280, h=960, N=12, iters=50, P=4096, kind="prior", seed=41,
               what="configs[4]: 1280x960 RGB-D-prior, 12 flows, 50 EM iters, 4096 hypotheses/camera (bandwidth-stress)"),
}
FP = C.POINTER(C.c_float)


def bench_config(world):
    """identical in both arms"""
    return {"workload": WORKLOAD,
            "parallelism": f"window-per-GPU x{world}" + (", 1 NCCL all_gather of poses per step" if world > 1 else ""),
            "l2": "256 MB device write between timed steps (flush), per-step CUDA events"}


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)"""

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "50"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for k, n in enumerate(names):
                if len(r) > 5 + k and r[5 + k].lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_case(name, seed_offset=0):
    """synthetic window of a BASELINE configuration: (win, kwargs of the window call, bootstrap or None, flags)"""
    import synth

    c = CASES[name]
    win = synth.make_window(c["w"], c["h"], c["N"], seed=c["seed"] + seed_offset)
    cfg = f"--silent --max_iters {c['iters']} --no_trunc_iters 1000 --n_poses_to_sample {c['P']}"
    kw, boot = {}, None
    if c["kind"] == "mono":
        boot = (win["Rs"][0], win["ts"][0], synth.noisy_depth(win, 0.05, seed=7 + seed_offset))
    elif c["kind"] == "stereo":
        basefocal = float(0.54 * win["fx"])
        rng = np.random.default_rng(3)
        disp = (basefocal / win["depth_gt"] * (1 + rng.normal(0, 0.02, win["depth_gt"].shape))).astype(np.float32)
        kw.update(basefocal=basefocal, disparity=disp)
    else:
        kw.update(depth_priors=synth.noisy_depth(win, 0.01)[None], depth_prior_poses=np.zeros((1, 6), np.float32))
    return win, kw, boot, cfg


def make_inputs(rank):
    """the benchmarked window of rank `rank` (context 0); other contexts use make_case("C2", offset)"""
    win, _, boot, _ = make_case("C2", rank)
    return win, boot


def run_cpu_sample(win, boot, iters=2, poses=NPOSES, **kw):
    """bounded CPU sample: same window, `iters` EM iterations, OpenMP over all host cores"""
    import oracle_host

    cfg = f"--silent --max_iters {iters} --no_trunc_iters 1000 --n_poses_to_sample {poses}"
    t0 = time.time()
    r = oracle_host.run_window("cpu", win["flows"], win["fx"], win["fy"], win["cx"], win["cy"], config=cfg, boot=boot,
                               **kw)
    dt = time.time() - t0
    return r["iters"] / dt, dt, r


def bench_reference(args, rank, world):
    """reference arm: rank 0 only"""
    if rank != 0:
        return
    import ffi
    import oracle_host

    win, boot = make_inputs(0)
    cores = os.cpu_count()
    if args.impl == "cpu-port" or not os.path.exists(ffi.REF):
        times, iters = [], 0
        for i in range(args.warmup + args.steps):
            v, dt, r = run_cpu_sample(win, boot, 1)
            if i >= args.warmup:
                times.append(dt)
                iters += r["iters"]
        total = sum(times)
        value = iters / total
        kind, sample = "port", f"one {W}x{H}x{NFLOWS} window, 1 EM iteration per step, CPU port with OpenMP on {cores} cores"
        ms_per_step = 1e3 * total / max(1, args.steps)
    else:
        import torch

        torch.cuda.set_device(0)
        clocks = ClockSampler(0)
        times, iters = [], 0
        # the reference's own host code when it was compiled here (oracle/_ref/libvoldor_host_ref.so), else its
        # restatement; the pose of its essential-matrix bootstrap is handed in (OpenCV is not in this image), the
        # closed-form depth of the bootstrap is computed by the reference inside the timed region
        own_host = os.path.exists(oracle_host.REF_HOST)
        short_windows = []
        R0 = np.asarray(boot[0], np.float32).reshape(3, 3)
        epipolar = (R0, (R0.T.astype(np.float64) @ np.asarray(boot[1], np.float64)).astype(np.float32))
        for i in range(args.warmup + args.steps):
            if i == args.warmup:
                clocks.start()
            ffi.libc_srand(1000 + i)
            torch.cuda.synchronize()
            t0 = time.time()
            backend = "ours_abi" if args.impl == "abi-dropin" else "ref"
            if own_host:
                # py_voldor_wrapper of the reference: its own host code, compiled unmodified (oracle/_ref)
                r = oracle_host.run_reference_host(backend, win["flows"], win["fx"], win["fy"], win["cx"], win["cy"],
                                                   config=CONFIG, epipolar=epipolar)
                # py_voldor_wrapper does not report the iteration count; with truncation off the loop runs max_iters
                # times as long as a camera is left (voldor.cpp:135).  A window that lost cameras is noted on the line.
                r["iters"] = EM_ITERS if r["n_registered"] > 0 else 0
                if r["n_registered"] != NFLOWS:
                    short_windows.append((i, int(r["n_registered"])))
            else:
                r = oracle_host.run_window(backend, win["flows"], win["fx"], win["fy"], win["cx"], win["cy"],
                                           config=CONFIG, boot=boot)
            torch.cuda.synchronize()
            if i >= args.warmup:
                times.append(time.time() - t0)
                iters += r["iters"]
        total = sum(times)
        value = iters / total
        kind = "reference"
        if args.impl == "abi-dropin":
            kind = "abi-dropin"
        sample = (f"full workload: {args.steps} windows of {W}x{H}x{NFLOWS}, {EM_ITERS} EM iterations each; reference "
                  "CUDA kernels (its own .cu files rebuilt for sm_100a, oracle/_ref) on 1 B200 driven by " +
                  ("the reference's own host code through py_voldor_wrapper (voldor.cpp / geometry.cpp / py_export.cpp "
                   "compiled unmodified against an OpenCV stand-in; essential-matrix pose handed in, closed-form "
                   "bootstrap depth computed by the reference inside the timed region)" if own_host else
                   "the reference host orchestration (voldor.cpp/geometry.cpp restated OpenCV-free)") +
                  " on 1 host thread")
        if args.impl == "abi-dropin":
            sample = sample.replace("reference CUDA kernels (its own .cu files rebuilt for sm_100a, oracle/_ref)",
                                    "voldor_b200's gpu_kernels.h entry points (library-level drop-in, host buffers)")
        ms_per_step = 1e3 * total / max(1, args.steps)
        clk = clocks.stop()
    line = {
        "impl": "reference" if args.impl != "abi-dropin" else "abi-dropin", "metric": "EM-iters/sec", "value": value,
        "unit": "EM-iterations/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(world),
        "cpu_baseline": {"value": value, "unit": "EM-iterations/s", "cores": 1 if kind != "port" else cores,
                         "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "EM-iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "frames_per_sec": value * NFLOWS / EM_ITERS,
    }
    if kind != "port":
        line["clocks"] = clk
        if short_windows:
            line["note"] = f"windows that registered fewer than {NFLOWS} frames (step, frames): {short_windows}"
    print(json.dumps(line))


class WindowRunner:
    """one window configuration bound to one execution context of the library: device-resident, pinned-host and
    pageable copies of its inputs, and the three ways of calling the window through the C ABI"""

    def __init__(self, lib, dev, ctx, win, kw, boot, cfg):
        import torch

        self.lib, self.dev, self.ctx, self.cfg = lib, dev, ctx, cfg.encode()
        self.win, self.kw, self.boot = win, kw, boot
        self.N, self.h, self.w = win["flows"].shape[:3]
        self.f = [float(win[k]) for k in ("fx", "fy", "cx", "cy")]
        self.basefocal = float(kw.get("basefocal", 0.0))
        names = ("flows", "disparity", "depth_priors", "depth_prior_poses")
        src = {"flows": win["flows"], "disparity": kw.get("disparity"), "depth_priors": kw.get("depth_priors"),
               "depth_prior_poses": kw.get("depth_prior_poses")}
        self.np_in = {k: (None if src[k] is None else np.ascontiguousarray(src[k], np.float32)) for k in names}
        self.pin_in = {k: (None if v is None else torch.from_numpy(v).pin_memory()) for k, v in self.np_in.items()}
        # poses of the priors are read by the host side of the library: always a host buffer
        self.dev_in = {k: (None if v is None else (v if k == "depth_prior_poses" else v.to(dev)))
                       for k, v in self.pin_in.items()}
        self.N_dp = 0 if src["depth_priors"] is None else src["depth_priors"].shape[0]
        shapes = (("poses", (self.N, 6)), ("covar", (self.N, 36)), ("depth", (self.h, self.w)), ("conf", (self.h, self.w)))
        self.out_h = {k: torch.zeros(s, dtype=torch.float32).pin_memory() for k, s in shapes}
        self.out_d = {k: torch.zeros_like(v, device=dev) for k, v in self.out_h.items() if k in ("depth", "conf")}
        self.out_np = {k: np.zeros(s, np.float32) for k, s in shapes}
        self.h2d_bytes = int(sum(v.numel() * 4 for v in self.pin_in.values() if v is not None))
        self.d2h_bytes = int(sum(v.numel() * 4 for v in self.out_h.values()))

    def bind(self):
        """select this runner's context on the calling thread and install its bootstrap override"""
        import voldor_b200

        self.lib.vb_context_select(self.ctx)
        if self.boot is not None:
            voldor_b200.set_bootstrap_override(*self.boot)
        else:
            voldor_b200.set_bootstrap_override()

    @staticmethod
    def _p(t):
        if t is None:
            return None
        if isinstance(t, np.ndarray):
            return t.ctypes.data_as(FP)
        return C.cast(t.data_ptr(), FP)

    def run(self, mode="resident"):
        """modes: resident (device pointers in, depth/conf out on the device), pinned (host buffers, e2e),
        pageable (numpy buffers through the reference-facing C++ symbol py_voldor_wrapper)"""
        self.lib.vb_context_select(self.ctx)
        n, it = C.c_int(0), C.c_int(0)
        self.n_registered = None
        stats = np.zeros(4, np.float32)
        p = self._p
        if mode == "pageable":
            i, o = self.np_in, self.out_np
            self.lib._Z17py_voldor_wrapperPKfS0_S0_S0_S0_S0_fffffiiiiPKcRiPfS4_S4_S4_(
                p(i["flows"]), p(i["disparity"]), None, p(i["depth_priors"]), p(i["depth_prior_poses"]), None,
                *map(C.c_float, self.f), C.c_float(self.basefocal), self.N, self.N_dp, self.w, self.h, self.cfg,
                C.byref(n), p(o["poses"]), p(o["covar"]), p(o["depth"]), p(o["conf"]))
            self.n_registered = n.value
            return n.value, int(self.cfg.split(b"--max_iters ")[1].split()[0]), stats
        i = self.dev_in if mode == "resident" else self.pin_in
        depth = self.out_d["depth"] if mode == "resident" else self.out_h["depth"]
        conf = self.out_d["conf"] if mode == "resident" else self.out_h["conf"]
        self.lib.vb_py_voldor_wrapper_ex(p(i["flows"]), p(i["disparity"]), None, p(i["depth_priors"]),
                                         p(i["depth_prior_poses"]), None, *map(C.c_float, self.f),
                                         C.c_float(self.basefocal), self.N, self.N_dp, self.w, self.h, self.cfg,
                                         C.byref(n), p(self.out_h["poses"]), p(self.out_h["covar"]), p(depth), p(conf),
                                         C.byref(it), stats.ctypes.data_as(FP))
        self.n_registered = n.value
        return n.value, it.value, stats

    def outputs(self, mode):
        if mode == "pageable":
            o = self.out_np
            return {k: o[k].copy() for k in o}
        import torch

        torch.cuda.synchronize()
        d = self.out_d if mode == "resident" else self.out_h
        return {"poses": self.out_h["poses"].numpy().copy(), "covar": self.out_h["covar"].numpy().copy(),
                "depth": d["depth"].cpu().numpy().copy(), "conf": d["conf"].cpu().numpy().copy()}


def dump_outputs(path, runners, mode):
    """the outputs of the last window each runner solved in `mode`, as voldor() hands them to its caller"""
    os.makedirs(path, exist_ok=True)
    for r in runners:
        o, n = r.outputs(mode), r.n_registered
        arrays = {"poses": o["poses"][:n], "poses_covar": o["covar"][:n].reshape(n, 6, 6), "depth": o["depth"],
                  "depth_conf": o["conf"]}
        for name, a in arrays.items():
            np.save(os.path.join(path, f"ctx{r.ctx}_{name}.npy"), np.ascontiguousarray(a, np.float32))


class ContextWorkers:
    """one persistent host thread per execution context; thread k selects context k once and then runs the windows
    of runner k on request (ctypes releases the GIL during the library call, so the windows overlap on the GPU)"""

    def __init__(self, runners):
        import queue

        self.runners = runners
        self.jobs = [queue.Queue() for _ in runners]
        self.done = queue.Queue()
        self.threads = [threading.Thread(target=self._loop, args=(k,), daemon=True) for k in range(len(runners))]
        for t in self.threads:
            t.start()
        for _ in runners:
            self.done.get()  # bound

    def _loop(self, k):
        import voldor_b200

        r = self.runners[k]
        r.bind()
        self.done.put((k, None))
        while True:
            mode = self.jobs[k].get()
            if mode is None:
                voldor_b200.set_bootstrap_override()
                self.done.put((k, None))
                return
            t0 = time.time()
            try:
                n, it, _ = r.run(mode)
                self.done.put((k, (n, it, time.time() - t0)))
            except Exception as e:  # noqa: BLE001
                self.done.put((k, e))

    def _collect(self, count):
        out = {}
        for _ in range(count):
            k, res = self.done.get()
            if isinstance(res, Exception):
                raise res
            out[k] = res
        return [out[k] for k in sorted(out)]

    def run_all(self, mode):
        for q in self.jobs:
            q.put(mode)
        return self._collect(len(self.jobs))

    def run_one(self, k, mode):
        self.jobs[k].put(mode)
        return self._collect(1)[0]

    def close(self):
        for q in self.jobs:
            q.put(None)
        self._collect(len(self.jobs))


def search_kernel_roofline(lib, runner, ncu_json=None):
    """per-launch duration of the dominant kernel measured in the library with CUDA events on its own stream"""
    lib.vb_context_select(runner.ctx)
    lib.vb_profile_enable(1)
    runner.run("resident")
    sm, sl = C.c_double(0), C.c_longlong(0)
    lib.vb_profile_get(C.byref(sm), C.byref(sl))
    ms3, n3 = (C.c_double * 3)(), (C.c_longlong * 3)()
    lib.vb_profile_get_more(ms3, n3)
    lib.vb_profile_enable(0)
    N, N_dp, w, h = runner.N, runner.N_dp, runner.w, runner.h
    alg_bytes = w * h * (12 * N + 60 + 12 * N_dp)  # + prior depth / pconf / conf fetches
    avg_ms = sm.value / max(1, sl.value)
    peak, peak_src = _peaks()
    achieved = alg_bytes / (avg_ms * 1e-3) / 1e9
    traffic = issue_pct = None
    if ncu_json:
        try:
            with open(os.path.join(ROOT, "profiles", ncu_json)) as f:
                cap = json.load(f)
            traffic, issue_pct = cap.get("dram_bytes_per_launch"), cap.get("issue_active_pct")
        except (OSError, ValueError):
            pass
    def other(k, name, nbytes, what):
        if n3[k] == 0:
            return None
        t = ms3[k] / n3[k]
        return {"kernel": name, "what": what, "algorithmic_bytes": nbytes, "avg_ms": t, "runs_timed": n3[k],
                "achieved": nbytes / (t * 1e-3) / 1e9, "unit": "GB/s", "frac": nbytes / (t * 1e-3) / 1e9 / peak}

    px = w * h
    others = [other(0, "k_update_rigidness", px * (12 * N + 4 + 16 * N_dp), "E-step: flows 8N + rigidness out 4N + depth 4 per pixel"),
              other(1, "k_fb_rows + k_fb_posterior + k_fb_cols + k_fb_posterior", px * 48 * N,
                    "one forward-backward smoothing of the N rigidness maps: 12 map-sized reads/writes"),
              other(2, "k_local_propagation_group x4", 4 * px * (12 * N + 12 + 12 * N_dp), "the four local-propagation passes of one depth step")]
    return {"bound": "hbm", "kernel": "k_cost_and_random_search_pruned", "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": avg_ms, "launches_timed": sl.value,
            "binding_bound": "instruction issue", "issue_slots_busy_pct_ncu": issue_pct,
            "other_kernels": [o for o in others if o]}


def whole_iteration_roofline(case, iters, ms):
    w, h, N, P = case["w"], case["h"], case["N"], case["P"]
    N_dp = 0 if case["kind"] == "mono" else 1
    b = w * h * (76 * N + 56 + 16 * N_dp) + 128 * N * P  # SURVEY §8(d)
    peak, _ = _peaks()
    ach = b * iters / (ms * 1e-3) / 1e9
    return {"algorithmic_bytes_per_iter": b, "achieved": ach, "frac": ach / peak}


def bench_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    import ffi
    import voldor_b200

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    lib = voldor_b200.load_library()
    voldor_b200.set_device(local_rank)  # the worker threads below inherit the library's device, not torch's
    lib.vb_profile_enable.argtypes = [C.c_int]
    lib.vb_profile_get.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_longlong)]
    lib.vb_profile_get_more.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_longlong)]
    M = max(1, min(args.inflight, lib.vb_context_max()))

    # context k of rank r solves its own window (different scene seeds); context 0 = the window of round 1's bench
    runners = []
    for k in range(M):
        win, kw, boot, cfg = make_case("C2", rank + 1000 * k)
        runners.append(WindowRunner(lib, dev, k, win, kw, boot, cfg))
    workers = ContextWorkers(runners)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    gathered = [torch.zeros(NFLOWS * 6, device=dev) for _ in range(world)] if world > 1 else None

    def run_on_own_thread(mode, count):
        return workers.run_all(mode)

    # ---- parity: first window of context 0 from fresh state vs the reference kernels from fresh state -------------
    parity = None
    first = None
    if rank == 0:
        ffi.libc_srand(4242)
    res = run_on_own_thread("resident", M)  # also the first warm-up step (allocations, RNG seeding)
    if rank == 0:
        first = runners[0].outputs("resident")
        first["n"], first["iters"] = res[0][0], res[0][1]

    def timed(mode, steps, warmup, clocks=None):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        iters = frames = 0
        wall = 0.0
        lat = []
        for i in range(warmup + steps):
            if i == warmup:
                if world > 1:
                    dist.barrier()
                torch.cuda.synchronize()
                if clocks:
                    clocks.start()
            flush.fill_(i & 255)  # evict L2 between steps (outside the timed region)
            torch.cuda.synchronize()
            k = i - warmup
            if k >= 0:
                ev[k][0].record()
            t0 = time.time()
            res = run_on_own_thread(mode, M)
            if world > 1:  # the single collective of the path: all ranks learn all poses
                dist.all_gather(gathered, runners[0].out_h["poses"].to(dev, non_blocking=True).reshape(-1))
            if k >= 0:
                ev[k][1].record()
                torch.cuda.synchronize()
                wall += time.time() - t0
                iters += sum(r[1] for r in res)
                frames += sum(r[0] for r in res)
                lat += [r[2] for r in res]
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        dev_ms = sum(a.elapsed_time(b) for a, b in ev)
        ms = max(dev_ms, 1e3 * wall)  # the calls are synchronous: both clocks see the same region
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        cnt = torch.tensor([iters, frames], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        return float(t.item()), float(cnt[0].item()), float(cnt[1].item()), 1e3 * float(np.mean(lat))

    clocks = ClockSampler(local_rank) if rank == 0 else None
    ms_res, iters_res, frames_res, lat_res = timed("resident", args.steps, args.warmup, clocks)
    clk = clocks.stop() if clocks else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, runners, "resident")
    ms_e2e, iters_e2e, _, lat_e2e = timed("pinned", args.steps, max(1, args.warmup // 2))

    # the collective really carried this rank's poses (C4 identity of the exchange)
    allgather_ok = None
    if world > 1:
        mine = runners[0].out_h["poses"].reshape(-1).to(dev)
        allgather_ok = bool(torch.equal(gathered[rank], mine))
        flag = torch.tensor([1.0 if allgather_ok else 0.0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        allgather_ok = bool(flag.item() == 1.0)

    roof = launches_per_window = single = pageable = extras = None
    if rank == 0:
        # one window in flight: latency and throughput of a lone window (what round 1 measured)
        t_single = []
        for i in range(3 + 5):
            flush.fill_(i)
            torch.cuda.synchronize()
            t0 = time.time()
            workers.run_one(0, "resident")
            torch.cuda.synchronize()
            if i >= 3:
                t_single.append(time.time() - t0)
        single = {"ms_per_window": 1e3 * float(np.mean(t_single)),
                  "value": EM_ITERS / float(np.mean(t_single)), "unit": "EM-iterations/s"}
        # pageable numpy buffers through the reference-facing C++ symbol (what pyvoldor_vo.pyx / slam_py calls)
        r0 = runners[0]
        r0.bind()
        t_page = []
        for i in range(2 + 5):
            t0 = time.time()
            r0.run("pageable")
            if i >= 2:
                t_page.append(time.time() - t0)
        pageable = {"value": EM_ITERS / float(np.mean(t_page)), "unit": "EM-iterations/s",
                    "ms_per_window": 1e3 * float(np.mean(t_page)), "h2d_bytes_per_step": r0.h2d_bytes,
                    "d2h_bytes_per_step": r0.d2h_bytes,
                    "how": "py_voldor_wrapper (C++ symbol bound by pyvoldor_vo.pyx), pageable numpy in/out, 1 window in flight"}

        roof = search_kernel_roofline(lib, r0, "r02_ncu_search_kernel.json")
        roof["whole_iteration"] = whole_iteration_roofline(CASES["C2"], iters_res / world, ms_res)
        roof["note"] = ("instruction-issue-bound kernel (Fisk posteriors: 6 powers + expf + logf + 7 IEEE divisions per "
                        "likelihood term, rounding points pinned by bit-parity; candidates that provably cannot win are "
                        "rejected after their first terms): HBM fraction reported as BASELINE.json asks; see DESIGN.md "
                        "§6 and profiles/r02_summary.md for the issue roofline of the whole path")
        # kernel launches per window (counted once, outside the timed region, with the CUPTI-based profiler)
        try:
            from torch.profiler import ProfilerActivity, profile

            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                r0.run("resident")
                torch.cuda.synchronize()
            launches_per_window = sum(1 for e in prof.events() if e.device_type.name == "CUDA" and
                                      ("k_" in e.name or "vb" in e.name) and "Memcpy" not in e.name)
        except Exception:
            launches_per_window = None

        # parity of the benchmarked configuration itself, against the reference kernels from the same fresh state
        if os.path.exists(ffi.REF) and not args.no_parity:
            import oracle_host

            ffi.libc_srand(4242)
            ref = oracle_host.run_window("ref", r0.win["flows"], *r0.f, config=CONFIG, boot=r0.boot)
            same = (first["n"] == ref["n_registered"] and first["iters"] == ref["iters"] and
                    ffi.bits_equal(first["poses"][:ref["n_registered"]], ref["poses"]) and
                    ffi.bits_equal(first["covar"][:ref["n_registered"]].reshape(-1, 6, 6), ref["poses_covar"]) and
                    ffi.bits_equal(first["depth"], ref["depth"]) and ffi.bits_equal(first["conf"], ref["depth_conf"]))
            parity = bool(same)

        if not args.no_extras and world == 1:
            extras = {}
            for name in ("C1", "C3", "C5"):
                win, kw, boot, cfg = make_case(name)
                r = WindowRunner(lib, dev, 0, win, kw, boot, cfg)
                r.bind()
                ts, its = [], 0
                for i in range(1 + 3):
                    flush.fill_(i)
                    torch.cuda.synchronize()
                    t0 = time.time()
                    n, it, _ = r.run("resident")
                    torch.cuda.synchronize()
                    if i >= 1:
                        ts.append(time.time() - t0)
                        its += it
                tp = []
                for i in range(1 + 2):
                    t0 = time.time()
                    r.run("pinned")
                    torch.cuda.synchronize()
                    if i >= 1:
                        tp.append(time.time() - t0)
                c = CASES[name]
                e = {"workload": c["what"], "value": its / sum(ts), "unit": "EM-iterations/s",
                     "ms_per_window": 1e3 * float(np.mean(ts)), "frames_registered": n,
                     "e2e": {"value": c["iters"] / float(np.mean(tp)), "unit": "EM-iterations/s",
                             "h2d_bytes_per_step": r.h2d_bytes, "d2h_bytes_per_step": r.d2h_bytes},
                     "roofline": search_kernel_roofline(lib, r)}
                e["roofline"]["whole_iteration"] = whole_iteration_roofline(c, its, 1e3 * sum(ts))
                if name == "C1" and not args.no_cpu_baseline:
                    v, dt, rr = run_cpu_sample(win, boot, c["iters"], c["P"])
                    e["cpu_baseline"] = {"value": v, "unit": "EM-iterations/s", "cores": os.cpu_count(), "kind": "port",
                                         "sample": f"the full C1 window ({c['iters']} EM iterations, {dt:.1f} s): CPU "
                                                   "restatement with OpenMP on all host cores under the restated "
                                                   "reference orchestration"}
                extras[name] = e
                del r
            runners[0].bind()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, dt, _ = run_cpu_sample(runners[0].win, runners[0].boot, 2)
        cpu = {"value": v, "unit": "EM-iterations/s", "cores": os.cpu_count(), "kind": "port",
               "sample": f"the same {W}x{H}x{NFLOWS} window, 2 EM iterations ({dt:.1f} s), CPU port with OpenMP on all "
                         "host cores under the restated reference orchestration"}

    workers.close()
    if rank == 0:
        value = iters_res / (ms_res * 1e-3)
        e2e = iters_e2e / (ms_e2e * 1e-3)
        line = {
            "metric": "EM-iters/sec", "value": value, "unit": "EM-iterations/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(world),
            "windows_in_flight_per_gpu": M,
            "frames_per_sec": frames_res / (ms_res * 1e-3),
            "e2e": {"value": e2e, "unit": "EM-iterations/s", "h2d_bytes_per_step": runners[0].h2d_bytes * M,
                    "d2h_bytes_per_step": runners[0].d2h_bytes * M, "ms_per_step": ms_e2e / args.steps},
            "e2e_pageable": pageable,
            "latency": {"ms_per_window_in_flight": lat_res, "ms_per_window_in_flight_e2e": lat_e2e,
                        "single_window": single},
            "gpu_launches": (launches_per_window or 0) * args.steps * M,
            "gpu_launches_per_window": launches_per_window,
            "parity_checked": parity, "allgather_checked": allgather_ok,
            "clocks": clk, "roofline": roof, "cpu_baseline": cpu, "extra": extras,
        }
        print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "cpu-port", "abi-dropin"])
    ap.add_argument("--inflight", type=int, default=int(os.environ.get("VB_BENCH_INFLIGHT", "8")),
                    help="independent windows in flight per GPU (execution contexts)")
    ap.add_argument("--no-cpu-baseline", dest="no_cpu_baseline", action="store_true")
    ap.add_argument("--no-extras", dest="no_extras", action="store_true")
    ap.add_argument("--no-parity", dest="no_parity", action="store_true")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="write the outputs of the last timed step as float32 .npy files into DIR")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl != "ours":
        bench_reference(args, rank, world)
        return
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; voldor_b200 has no CPU fallback")
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        bench_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist

            dist.destroy_process_group()


if __name__ == "__main__":
    main()
