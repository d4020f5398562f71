"""Run on the GPU box: time of lfba_solver_covariance beside one LM round, at cfg3 and cfg4.

Both workloads refine points, so the covariance needs distance constraints to fix the scale: cfg3's preset has three,
cfg4's has none and is timed with n_constraints = 3 set in its scene spec (the output says so). Per workload: one full
solve with opt.profile = 1 gives the mean device time of one LM round (per-stage CUDA events, stream drained every
round); then the covariance at the solution is called `--reps` times after one warm-up call, and the host wall time of
each call (it ends in a stream synchronise) and its CUDA-event times (whole call, selected inversion) are reported as
median / min / max. The GPU's name, power limit and SM clocks are read in the same run.

With --points, each repetition also calls covariance(with_points=True) right after the plain call on the same session,
and reports its wall time, its device time of the per-point stage (points_ms) and, timed on its own with CUDA events
through torch, the device-to-host copy of the 9 P doubles it returns into pageable host memory.

  python scripts/gpu_covariance_time.py [--reps 7] [--points] [--out covariance_time.json] [cfg3 cfg4]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from lifcal_b200 import api, capi  # noqa: E402


def gpu_state():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unavailable"


def d2h_copy_ms(n_doubles, reps):
    """Device time of copying n doubles into pageable host memory (a fresh NumPy array, as the API returns)."""
    import torch
    src = torch.zeros(n_doubles, dtype=torch.float64, device="cuda")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = []
    for i in range(reps + 1):
        dst = torch.from_numpy(np.zeros(n_doubles))
        e0.record()
        dst.copy_(src)
        e1.record()
        torch.cuda.synchronize()
        if i:  # the first copy is a warm-up
            out.append(e0.elapsed_time(e1))
    return out


def spread(v):
    return {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "max": round(max(v), 4), "n": len(v)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workloads", nargs="*", default=["cfg3", "cfg4"])
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--points", action="store_true", help="also time covariance(with_points=True)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if api.device_count() < 1:
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    results = []
    for name in args.workloads:
        preset = int(name[-1])
        spec_kw = {"order": 1}
        note = "preset scene"
        if capi.scene_spec(preset).n_constraints == 0:
            spec_kw["n_constraints"] = 3
            note = "preset scene with n_constraints = 3 set in the scene spec (the preset has none)"
        sc = capi.make_scene(preset, **spec_kw)
        ds = api.DeviceSolver(sc.problem, api.default_options(profile=1))
        ds.set_parameters(sc.camera_init, sc.views_init, sc.points_init)
        s = ds.run()
        rounds = s["kernel_calls"]["lens_pose_tables"]
        round_ms = sum(s["kernel_ms"].values()) / rounds
        ds.covariance()  # warm-up
        if args.points:
            ds.covariance(with_points=True)
        wall, dev, inv = [], [], []
        pwall, pdev, pts = [], [], []
        for _ in range(args.reps):
            t = time.perf_counter()
            c = ds.covariance()
            wall.append(1e3 * (time.perf_counter() - t))
            dev.append(c["info"]["gpu_ms"])
            inv.append(c["info"]["selinv_ms"])
            if args.points:
                t = time.perf_counter()
                cp = ds.covariance(with_points=True)
                pwall.append(1e3 * (time.perf_counter() - t))
                pdev.append(cp["info"]["gpu_ms"])
                pts.append(cp["info"]["points_ms"])
        info = c["info"]
        ds.close()
        r = {"workload": name, "scene": note, "gpu": gpu_state(), "N": s["num_observations"],
             "n_reduced": info["n_reduced"], "gauge_frame": info["gauge_frame"], "lm_rounds": rounds,
             "lm_round_ms_mean": round(round_ms, 4), "covariance_wall_ms": spread(wall),
             "covariance_gpu_ms": spread(dev), "selinv_gpu_ms": spread(inv),
             "covariance_over_lm_round": round(statistics.median(dev) / round_ms, 3),
             "sigma2": info["sigma2"], "std_camera": [float(x) for x in c["std_camera"]]}
        if args.points:
            n_pts = int(sc.problem.n_points)
            r.update({"P": n_pts, "points_copy_mb": round(72 * n_pts / 1e6, 3),
                      "covariance_points_wall_ms": spread(pwall), "covariance_points_gpu_ms": spread(pdev),
                      "points_gpu_ms": spread(pts), "points_d2h_copy_ms": spread(d2h_copy_ms(9 * n_pts, args.reps)),
                      "points_over_lm_round": round(statistics.median(pts) / round_ms, 3),
                      "median_std_points": [float(x) for x in np.median(cp["std_points"][np.any(cp["points"] != 0,
                                                                                                 axis=(1, 2))], axis=0)]})
        print(json.dumps(r))
        sys.stdout.flush()
        results.append(r)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
