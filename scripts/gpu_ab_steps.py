"""Run on the GPU box: A/B of the benchmark's step time between two source trees (each already built in place).

  python scripts/gpu_ab_steps.py OLD_TREE NEW_TREE [--rounds 3] [--steps 20] [--workload cfg4] [--out ab.json]

Runs `python <tree>/bench.py --workload W --steps K --no-cpu-baseline --no-e2e` alternately in the two trees, `--rounds`
times each (old first in even rounds, new first in odd ones), and keeps every run's ms_per_step, value and clocks. Then,
once per tree, the device memory a solver session holds at the workload: free memory (cudaMemGetInfo through torch)
before the session is created and after its parameters are set. The GPU's name and power limit are read in the same
run. Prints one JSON document (and writes it to --out): the runs, per-tree median / min / max, and whether every new
run was faster than every old one.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

MEM_PROBE = r"""
import json, sys, torch
sys.path.insert(0, sys.argv[1])
from lifcal_b200 import api, capi
sc = capi.make_scene(int(sys.argv[2][-1]), order=1)
torch.cuda.init()
free0 = torch.cuda.mem_get_info()[0]
ds = api.DeviceSolver(sc.problem)
ds.set_parameters(sc.camera_init, sc.views_init, sc.points_init)
torch.cuda.synchronize()
free1 = torch.cuda.mem_get_info()[0]
ds.close()
print(json.dumps({"session_bytes": free0 - free1}))
"""


def _last_json(text):
    for line in reversed(text.splitlines()):
        line = line.strip()
        if line.startswith("{"):
            return json.loads(line)
    raise RuntimeError("no JSON line in:\n" + text[-2000:])


def _run(cmd, cwd):
    r = subprocess.run(cmd, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"{' '.join(cmd)} (in {cwd}) exited {r.returncode}:\n{r.stdout[-4000:]}")
    return r.stdout


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--workload", default="cfg4")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    trees = {"old": os.path.abspath(a.old), "new": os.path.abspath(a.new)}
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()[0]
    runs = []
    for r in range(a.rounds):
        for label in (("old", "new") if r % 2 == 0 else ("new", "old")):
            out = _run([sys.executable, os.path.join(trees[label], "bench.py"), "--workload", a.workload,
                        "--steps", str(a.steps), "--no-cpu-baseline", "--no-e2e"], trees[label])
            j = _last_json(out)
            runs.append({"tree": label, "round": r, "ms_per_step": j["ms_per_step"], "value": j["value"],
                         "final_cost": j.get("final_cost"), "clocks": j.get("clocks")})
            print(json.dumps(runs[-1]), flush=True)
    summary = {}
    for label in trees:
        ms = [x["ms_per_step"] for x in runs if x["tree"] == label]
        summary[label] = {"median_ms_per_step": statistics.median(ms), "min": min(ms), "max": max(ms), "n": len(ms)}
        mem = _run([sys.executable, "-c", MEM_PROBE, trees[label], a.workload], trees[label])
        summary[label]["session_bytes"] = _last_json(mem)["session_bytes"]
    res = {"gpu": gpu, "workload": a.workload, "steps": a.steps, "trees": trees, "runs": runs, "summary": summary,
           "median_change": summary["new"]["median_ms_per_step"] / summary["old"]["median_ms_per_step"] - 1.0,
           "every_new_faster_than_every_old": summary["new"]["max"] < summary["old"]["min"],
           "session_bytes_saved": summary["old"]["session_bytes"] - summary["new"]["session_bytes"]}
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
