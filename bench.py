#!/usr/bin/env python
"""bench.py — LF-BA hot-path benchmark (contract: one JSON line on rank 0).

Metric (BASELINE.json): "LM iters/s & M residual+Jacobian evals/s, 1/2/4/8 B200 vs Ceres CPU".
  metric  = M residual+Jacobian evals/s over complete LM solves (every LM iteration makes exactly one fused
            residual+Jacobian pass over all observations), `lm_iters_per_s` is reported next to it.
  step    = one complete LM solve (lfba_solver_run) of the workload from the same initial guess.
  value   = device-resident: observations already indexed in HBM, timed with CUDA events inside the library on its
            own stream (summary.solve_gpu_ms), max over ranks.
  e2e     = the same metric through the drop-in call lfba_solve() with HOST buffers: H2D of all observation arrays
            (pinned), device indexing, LM solve, D2H of camera/views/points — everything inside the timed region.
Workload: BASELINE.json configs[3] — 1M points x 1000 frames (window 4), ~1.1e8 micro-image observations, 2 radial +
tangential, robust (Cauchy 0.5), poses + points refined, micro-lens-centre adjustment. It fits one B200 (~10 GB), so it
is the N=1 workload too; with N GPUs the same scene is sharded by point/frame range (strong scaling).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg4|cfg3|cfg2|cfg1]
                  [--dump-outputs DIR]
  torchrun --nproc-per-node N bench.py --gpus N ...      (one rank per GPU, NCCL)

--dump-outputs DIR writes what the last timed solve returned to its caller as float64 .npy files: camera.npy (17),
views.npy (F x 6), points.npy (P x 3; with N ranks points_rank<r>.npy, the point range of rank r) and iteration_cost.npy
(the cost of every LM row). The scene comes from a fixed seed, so two builds run with the same arguments can be compared
output for output. cfg4, the largest workload, writes 24 MB.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# per-launch DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) of the dominant kernel from the ncu --set full
# capture of the same build (profiles/README.md); None where no capture exists for that workload
# per-launch DRAM traffic and FP64 instruction counts from `ncu --set full` of this build (profiles/r02_ncu_eval_kernels_cfg4.txt)
NCU_TRAFFIC = {"cfg4": 3.788e9}             # k_eval_rows: 2.658 GB read + 1.129 GB written (profiles/r02_ncu_eval_kernels_cfg4_final.txt)
NCU_TRAFFIC_EVAL_ONLY = {"cfg4": 3.7229e10}  # k_eval_only, live camera columns: 3.195 GB read + 34.034 GB written
FP64_INST_PER_OBS = 227.3  # (dfma + dmul + dadd thread instructions of k_eval_rows<9,2,1,3>) / observations = 2.5492e10 / 112137616
REC_STRIDE_NC9 = 36        # doubles per track record at NC = 9 (lfba_device.cuh rec_stride)
METRIC = "lm_residual_jacobian_evals_per_s"
UNIT = "M evals/s"
WORKLOADS = {"cfg1": 1, "cfg2": 2, "cfg3": 3, "cfg4": 4}
WORKLOAD_DESC = {
    "cfg1": "calib_marker 500 pts x 10 frames, 3 distance constraints",
    "cfg2": "recalib 5k pts x 20 frames (fL,B fixed, bounds)",
    "cfg3": "full calibration 50k pts x 100 frames, window 20",
    "cfg4": "scaled scene 1M pts x 1000 frames, window 4, ~1.1e8 observations",
}


# ---------------------------------------------------------------------------------------------------
# helpers shared with tests/test_sharding_gloo.py
# ---------------------------------------------------------------------------------------------------
def shard_range(n_points: int, rank: int, world: int):
    """Contiguous point range of a rank. Points are generated sorted by the start of their visibility window, so a
    point range is a frame range; every observation of a point stays on the point's rank."""
    lo = (n_points * rank) // world
    hi = (n_points * (rank + 1)) // world
    return lo, hi


def broadcast_unique_id(uid: bytes | None, device="cuda") -> bytes:
    """Rank 0 creates the 128-byte ncclUniqueId (lfba_comm_unique_id); torch.distributed is only the plumbing."""
    import torch
    import torch.distributed as dist
    t = torch.zeros(128, dtype=torch.uint8, device=device)
    if dist.get_rank() == 0:
        t.copy_(torch.tensor(list(uid), dtype=torch.uint8))
    dist.broadcast(t, src=0)
    return bytes(t.cpu().tolist())


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                smax.append(float(r[2]))
                pw.append(float(r[3]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def pinned_problem(pa):
    """Copies of the problem arrays in pinned host memory (torch is plumbing: it only owns the page-locked pages)."""
    import torch
    from lifcal_b200 import capi
    keep = []

    def pin(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        keep.append(t)
        return t.numpy()
    out = capi.ProblemArrays.__new__(capi.ProblemArrays)
    out.__dict__.update(pa.__dict__)
    for k in ("obs_x", "obs_y", "ml_x", "ml_y", "point_idx", "frame_idx"):
        setattr(out, k, pin(getattr(pa, k)))
    out._keep = keep
    return out


# ---------------------------------------------------------------------------------------------------
# CPU baseline: the Ceres-2.1.0-equivalent oracle on the SAME scene (same seed, every observation)
# ---------------------------------------------------------------------------------------------------
def _mem_available_gb() -> float:
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable"):
                return int(line.split()[1]) / 1e6
    except OSError:
        pass
    return 0.0


def host_threads() -> int:
    """All host cores this process may use — torchrun exports OMP_NUM_THREADS=1, which would silently make the CPU arm
    single-threaded at N > 1 (the reference uses hardware_concurrency(), src/CameraCalibration.cpp:961)."""
    from oracle import binding as ob
    try:
        ncores = len(os.sched_getaffinity(0))
    except AttributeError:
        ncores = os.cpu_count() or 1
    return max(ob.max_threads(), ncores)


def dump_outputs(out_dir: str, **arrays):
    """--dump-outputs: every array as out_dir/<name>.npy in float64."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, np.float64))


def solve_outputs(camera, views, points, summary, lo=0, hi=None) -> dict:
    """What a solve returns to its caller, in the shapes --dump-outputs writes; points lo:hi only (a rank's range)."""
    return {"camera": camera, "views": np.reshape(views, (-1, 6)), "points": np.reshape(points, (-1, 3))[lo:hi],
            "iteration_cost": [r["cost"] for r in summary["iterations"]]}


def run_cpu_baseline(workload: str, lm_iterations: int | None, scene=None, repeats: int = 1, warmup: int = 0):
    """Times the oracle on the benchmarked scene itself. cfg1-cfg3: the complete solve. cfg4 (1.12e8 observations, about
    35 s per Jacobian pass on 16 cores): a solve TRUNCATED after `lm_iterations` LM iterations — every Ceres iteration
    costs the same (one Jacobian evaluation, one Schur elimination + dense LLT, one cost evaluation), so the
    evaluations-per-second rate of the truncated solve is the rate of the complete one. Jacobian stored in Ceres' block
    layout (416 B per observation: 47 GB at cfg4) when the host has the memory, else the block-recompute mode."""
    from lifcal_b200 import capi
    from oracle import binding as ob
    if scene is None:
        scene = capi.Scene(capi.scene_spec(WORKLOADS[workload], order=1))
    pa = scene.problem
    n = pa.n_obs
    threads = host_threads()
    need_gb = 416.0 * n / 1e9 + 16.0 * n / 1e9 + 8.0 * threads * (17 + 6 * pa.n_frames) ** 2 / 1e9
    streaming = _mem_available_gb() < 1.3 * need_gb + 8.0
    opts = ob.default_options() if lm_iterations is None else ob.default_options(max_num_iterations=int(lm_iterations))
    dt, evals, rows = 0.0, 0, 0
    for k in range(warmup + repeats):
        t0 = time.perf_counter()
        cam, vw, pt, s = ob.solve(pa, scene.camera_init, scene.views_init, scene.points_init, options=opts, threads=threads,
                                  streaming=streaming)
        if k >= warmup:
            dt += time.perf_counter() - t0
            evals += s["num_jacobian_evals"]
            rows += s["num_iterations"]
    what = "complete solve" if lm_iterations is None else f"solve truncated after {lm_iterations} LM iteration(s) (rate extrapolates: every iteration costs the same)"
    return {"value": n * evals / dt / 1e6, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"the benchmarked scene itself ({workload}, same seed, all {n} observations): {what}; "
                      f"{repeats} solve(s) timed after {warmup} warm-up: {rows} LM rows, {evals} Jacobian evaluations in {dt:.1f} s; oracle = Ceres-2.1.0-equivalent "
                      f"restatement (Jet<26> autodiff, DENSE_SCHUR, dense LLT), functor pinned bit-exact to the reference "
                      f"headers; Jacobian {'recomputed per point block (block_passes=%d)' % s['block_passes'] if streaming else 'stored in Ceres block layout'}",
            "lm_iters_per_s": max(0, rows - repeats) / dt, "seconds": dt, "n_obs": n, "lm_rows": rows, "repeats": repeats,
            "warmup": warmup,
            "jacobian_evals": evals, "same_scene": True, "oracle_mode": "streaming" if streaming else "stored",
            "final_cost": s["final_cost"], "outputs": solve_outputs(cam, vw, pt, s)}


# ---------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("LFBA_BENCH_WORKLOAD", "cfg4"), choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-iterations", type=int, default=3,
                    help="cfg4 only: LM iterations of the CPU solve that --impl reference times (the scene is the full one)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed solve returned as DIR/<name>.npy (float64; see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")

    # The contract is ONE JSON line on stdout. Libraries write banners there (NCCL prints its version at communicator
    # creation): everything but the final line goes to stderr.
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    config = {"workload": f"{args.workload}: {WORKLOAD_DESC[args.workload]}", "flags": "nRadial=2,tangential,robust(Cauchy 0.5),"
              "refinePoses,refinePoints,mlAdj", "l2": "inputs larger than L2 (no flush needed)"}

    # ------------------------------------------------------------------ reference arm: CPU oracle on the same scene
    if args.impl == "reference":
        if rank != 0:
            return 0
        # cfg4: a CPU step takes minutes (1.12e8 observations); choose a small --steps there
        iters = None if args.workload != "cfg4" else args.cpu_iterations
        cb = run_cpu_baseline(args.workload, iters, repeats=args.steps, warmup=args.warmup)
        line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup,
                "steps_note": "a step is one LM solve of the FULL benchmarked scene on the host cores (cfg4: truncated after "
                              "--cpu-iterations LM iterations; the rate extrapolates)",
                "ms_per_step": 1e3 * cb["seconds"] / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic", "config": config, "lm_iters_per_s": cb["lm_iters_per_s"],
                "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "same_scene", "oracle_mode")},
                "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "final_cost": cb["final_cost"], "gpu_launches": 0}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, **cb["outputs"])
        emit(line)
        return 0

    # ------------------------------------------------------------------ our arm
    import torch
    from lifcal_b200 import api, capi
    if api.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device (the LF-BA path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))

    # ---- synthetic scene: every rank generates its own shard (counter-based RNG) ----
    preset = WORKLOADS[args.workload]
    spec = capi.scene_spec(preset, order=1)
    P = spec.n_points
    if world > 1 and spec.n_constraints > 0:
        spec.n_constraints = 0  # constraint-coupled points would all go to rank 0; the scaling workload has none
    lo, hi = shard_range(P, rank, world)
    if world > 1:
        spec.point_begin, spec.point_end = lo, hi
    t_gen = time.perf_counter()
    sc = capi.Scene(spec)
    t_gen = time.perf_counter() - t_gen
    pa = sc.problem
    n_local = pa.n_obs
    opt = api.default_options(device=local_rank)

    comm = None
    if world > 1:
        uid = broadcast_unique_id(api.comm_unique_id() if rank == 0 else None)
        comm = api.Communicator(rank, world, uid)  # one NCCL communicator per rank for the whole run
    t_setup = time.perf_counter()
    ds = api.DeviceSolver(pa, opt, communicator=comm)
    ds.set_parameters(sc.camera_init, sc.views_init, sc.points_init)
    t_setup = time.perf_counter() - t_setup

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up ----
    s = None
    for _ in range(max(3, args.warmup)):
        s = ds.run()
    n_global = s["num_observations"]
    # ---- timed: exactly K solves ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    t0 = time.perf_counter()
    gpu_ms, evals, iters, launches = 0.0, 0, 0, 0
    for _ in range(args.steps):
        s = ds.run()
        gpu_ms += s["solve_gpu_ms"]
        evals += s["num_jacobian_evals"]
        iters += s["num_iterations"]
        launches += s["gpu_launches"]
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    # read back before time_eval below evaluates on the same session
    outputs = solve_outputs(*ds.get_parameters(), s, lo, hi) if args.dump_outputs else None
    if dist is not None:
        t = torch.tensor([gpu_ms, wall], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        gpu_ms, wall = float(t[0].item()), float(t[1].item())
    value = n_global * evals / (gpu_ms * 1e-3) / 1e6

    # ---- dominant kernel: fused eval, timed live with CUDA events on the library's stream ----
    # Algorithmic HBM bytes of one launch (DESIGN.md section 4): 20 B per observation (double2 + int32 of the packed
    # stream) + the per-track record written, (9 + 3 NC) * 8 B = 288 B per (point, frame) track.
    eval_ms = ds.time_eval(reps=10, materialize=False)
    rec_stride = REC_STRIDE_NC9
    alg_bytes = 20.0 * n_local + 8.0 * rec_stride * s["num_tracks"]
    peak, peak_src = measured_peaks()
    # FP64 peak: MEASURED_PEAKS.json has no FP64 figure, so the DFMA rate is measured here, on this device, in this run
    # (dependent-chain-free DFMA kernel, lfba_measure_fp64_peak); nominal 148 SMs x 64 lanes x 2 x 1.965 GHz = 37.2 TFLOP/s
    fp64_peak = api.measure_fp64_peak(local_rank)
    ach_tf = FP64_INST_PER_OBS * n_local / (eval_ms * 1e-3) * 2.0 / 1e12  # every FP64 instruction counted as one FMA (2 flop)
    roofline = {"bound": "fp64", "kernel": "k_eval_rows (fused residual + analytic Jacobian + Cauchy weighting + per-track Gram "
                "-> normal-equation blocks; Jacobian never leaves registers)",
                "achieved": ach_tf, "peak": fp64_peak, "unit": "TFLOP/s", "frac": ach_tf / fp64_peak,
                "traffic": NCU_TRAFFIC.get(args.workload),
                "peak_source": "DFMA rate measured in this run on this device (MEASURED_PEAKS.json has no FP64 entry)",
                "ms_per_launch": eval_ms, "fp64_inst_per_observation": FP64_INST_PER_OBS,
                "fp64_inst_source": "ncu smsp__sass_thread_inst_executed_op_fp64 of the same build / observations (profiles/README.md)",
                "fused_eval_m_evals_per_s": n_local / (eval_ms * 1e-3) / 1e6,
                "hbm": {"bound": "hbm", "achieved": alg_bytes / (eval_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": alg_bytes / (eval_ms * 1e-3) / 1e9 / peak, "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": alg_bytes,
                        "note": "secondary: 20 B per observation streamed + one track record written per (point, frame); the "
                                "kernel is FP64-pipe bound (DESIGN.md section 4)"}}
    extra = {}
    if rank == 0 and world == 1:
        try:
            # eval-only kernel, Jacobian materialised: SURVEY.md 8(d) algorithmic bytes = 56 + 16 (NC + 6 + 3) = 344 B per
            # observation at NC = 9 (reads 40 B, writes r 16 B and the 2 x (NC + 6 + 3) LIVE Jacobian columns)
            mat_ms = ds.time_eval(reps=3, materialize=2)  # camera block as its live 2 x NC columns
            mat_bytes = 344.0 * n_local
            extra["roofline_eval_only"] = {"bound": "hbm", "kernel": "k_eval_only (residual + Jacobian materialised per observation)",
                                           "achieved": mat_bytes / (mat_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                           "frac": mat_bytes / (mat_ms * 1e-3) / 1e9 / peak, "ms_per_launch": mat_ms,
                                           "algorithmic_bytes_per_launch": mat_bytes, "bytes_per_observation": 344,
                                           "traffic": NCU_TRAFFIC_EVAL_ONLY.get(args.workload),
                                           "m_evals_per_s": n_local / (mat_ms * 1e-3) / 1e6}
        except Exception as e:  # noqa: BLE001
            extra["roofline_eval_only"] = {"error": str(e)}
    ds.close()

    # ---- e2e: the drop-in call with host (pinned) buffers, H2D + indexing + solve + D2H inside the timed region ----
    e2e = None
    if not args.no_e2e:
        ppa = pinned_problem(pa)
        o2 = api.default_options(device=local_rank)
        ts, ev2, h2d = [], 0, []
        if world == 1:
            # the caller's own parameter arrays (updated in place, like the reference's), page-locked like the observations;
            # they are reset to the initial values OUTSIDE the timed region
            pin_par = [torch.empty(n_, dtype=torch.float64).pin_memory()
                       for n_ in (17, sc.views_init.size, sc.points_init.size)]
            par = [t_.numpy() for t_ in pin_par]
            for k in range(1 + args.steps):
                for dst, src in zip(par, (sc.camera_init, sc.views_init, sc.points_init)):
                    dst[:] = np.asarray(src, np.float64).ravel()
                barrier()
                t1 = time.perf_counter()
                cam, vw, pt, s2 = api.solve(ppa, par[0], par[1], par[2], o2, inplace=True)
                torch.cuda.synchronize()
                dt = time.perf_counter() - t1
                if k > 0:
                    ts.append(dt)
                    ev2 += s2["num_jacobian_evals"]
                    h2d.append(s2.get("h2d_gbs"))
        else:
            for k in range(1 + args.steps):
                barrier()
                t1 = time.perf_counter()
                d2 = api.DeviceSolver(ppa, o2, communicator=comm)
                d2.set_parameters(sc.camera_init, sc.views_init, sc.points_init)
                s2 = d2.run()
                d2.get_parameters()
                torch.cuda.synchronize()
                dt = time.perf_counter() - t1
                d2.close()
                tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                if k > 0:
                    ts.append(float(tt.item()))
                    ev2 += s2["num_jacobian_evals"]
                    h2d.append(s2.get("h2d_gbs"))
        tot = sum(ts)
        F = pa.n_frames
        e2e = {"value": n_global * ev2 / tot / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(40 * n_local + 8 * (17 + 6 * F + 3 * P)),
               "d2h_bytes_per_step": int(8 * (17 + 6 * F + 3 * P)), "s_per_solve": tot / len(ts),
               "h2d_gbs_achieved": [round(v, 1) for v in h2d if v], "s_per_solve_each": [round(v, 4) for v in ts],
               "api": "lfba_solve (C ABI, pinned host buffers)" if world == 1 else "lfba_solver_create+run per rank"}

    if comm is not None:
        comm.close()
    if outputs is not None:
        if world > 1:  # every rank writes the points of its own range; camera, views and rows are the same on all ranks
            mine = {f"points_rank{rank}": outputs.pop("points")}
            outputs = dict(outputs, **mine) if rank == 0 else mine
        dump_outputs(args.dump_outputs, **outputs)
    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return 0
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": gpu_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": config, "lm_iters_per_s": iters / (gpu_ms * 1e-3),
            "lm_iterations_per_solve": iters / args.steps, "observations": n_global, "tracks_rank0": s["num_tracks"],
            "lenses_rank0": s["num_lenses"], "reduced_system_size": s["reduced_system_size"],
            "wall_s_per_step": wall / args.steps, "final_cost": s["final_cost"], "scene_gen_s": t_gen, "setup_s": t_setup,
            "clocks": clocks, "gpu_launches": launches, "roofline": roofline, "e2e": e2e}
    line.update(extra)
    if world == 1 and not args.no_cpu_baseline:
        # same scene object the GPU just solved; cfg4: one LM iteration (two Jacobian passes) keeps the default run short
        small = args.workload in ("cfg1", "cfg2")
        cb = run_cpu_baseline(args.workload, 1 if args.workload == "cfg4" else None, scene=sc, repeats=2 if small else 1,
                              warmup=1 if small else 0)
        line["cpu_baseline"] = {k: v for k, v in cb.items()
                                if k in ("value", "unit", "cores", "kind", "sample", "lm_iters_per_s", "same_scene", "oracle_mode")}
    emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
