"""Run on the GPU box: device time per launch of the Schur-assembly and back-substitution kernels, from torch.profiler
(CUPTI kernel records) around one solve of a workload, in a run of its own.

  python scripts/gpu_kernel_times.py [--tree DIR] [--out times.json] [cfg4 ...]

--tree picks the source tree whose built library is loaded (default: this one), so two builds can be compared in one
call. One warm-up solve, then one profiled solve. Prints one JSON line per workload: per kernel, launches and mean /
total device microseconds, plus the GPU's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

KERNELS = ("k_points", "k_frame_all", "k_frame_finish", "k_pairs", "k_coupled", "k_point_step", "k_eval_rows")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workloads", nargs="*", default=["cfg4"])
    ap.add_argument("--tree", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    sys.path.insert(0, os.path.abspath(a.tree))
    import torch
    from torch.profiler import ProfilerActivity, profile

    from lifcal_b200 import api, capi
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()[0]
    lines = []
    for name in a.workloads:
        sc = capi.make_scene(int(name[-1]), order=1)
        ds = api.DeviceSolver(sc.problem)
        ds.set_parameters(sc.camera_init, sc.views_init, sc.points_init)
        ds.run()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            s = ds.run()
            torch.cuda.synchronize()
        ds.close()
        per, other = {}, set()
        for ev in prof.events():
            k = next((k for k in KERNELS if k + "<" in ev.name or k + "(" in ev.name), None)
            if k is None:
                other.add(ev.name)
                continue
            e = per.setdefault(k, {"launches": 0, "total_us": 0.0})
            e["launches"] += 1
            e["total_us"] += ev.time_range.elapsed_us()  # a kernel record: its device start / end
        for e in per.values():
            e["mean_us"] = e["total_us"] / e["launches"]
        line = {"workload": name, "tree": os.path.abspath(a.tree), "gpu": gpu, "rows": s["num_iterations"],
                "kernels": per, "unmatched": sorted(other)[:40] if not per else []}
        print(json.dumps(line), flush=True)
        lines.append(line)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
