"""Cost of the AOV pass (DESIGN.md "AOV buffers"): ms_total of a run_view with AOVs off and on, alternated on one GPU.

    python tools/aov_cost.py [--workloads c1 c3] [--runs 2] [--out results/aov_cost.json]

For each workload (bench.py's C1 / C3 camera and settings, builder ploc8 unless CRT_BUILDER says otherwise) one scene and two
render handles are built, one warm-up frame is rendered on each, then `runs` frames alternate off, on, off, on ... The colour of
the two handles must be bit-identical. Prints one JSON object with the GPU's name and power limit (read in the same process) and,
per workload, the ms_total of every run, the kernel launches and the AOV pass's share of the frame (mean on / mean off - 1)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else "unavailable: " + q.stderr.strip()


def measure(crt, name, runs):
    import numpy as np
    from bench import Workload
    wl = Workload(name)
    scene, _ = wl.build_scene(crt, 0)
    M = crt.inverse_view_matrix(wl.eye, wl.lookat, wl.up)
    renders = {}
    for aov in (False, True):
        R = crt.Render(scene, wl.width, wl.height, wl.spp, wl.P_RR, wl.light_sample_n)
        R.set_aov(aov)
        R.run_view(wl.eye, M, wl.fovy_rad)                       # warm-up: module load, pool and AOV buffer allocation
        renders[aov] = R
    ms = {False: [], True: []}
    launches = {}
    for _ in range(runs):
        for aov in (False, True):
            renders[aov].run_view(wl.eye, M, wl.fovy_rad)
            st = renders[aov].stats()
            ms[aov].append(st["ms_total"])
            launches[aov] = st["kernel_launches"]
    same = bool(np.array_equal(renders[False].get_accum_i64(), renders[True].get_accum_i64()))
    cov = renders[True].get_aov()["coverage"]
    off, on = sum(ms[False]) / runs, sum(ms[True]) / runs
    return {"workload": wl.desc, "width": wl.width, "height": wl.height, "spp": wl.spp, "ms_total_off": ms[False], "ms_total_on": ms[True],
            "kernel_launches_off": launches[False], "kernel_launches_on": launches[True], "aov_share_of_frame": on / off - 1.0,
            "colour_identical": same, "mean_coverage": float(cov.mean())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["c1", "c3"])
    ap.add_argument("--runs", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import cudaraytracing_b200 as crt
    if crt.device_count() < 1:
        raise SystemExit("aov_cost: no CUDA device")
    res = {"gpu": gpu_info(), "builder": os.environ.get("CRT_BUILDER", "ploc8")}
    for name in args.workloads:
        res[name] = measure(crt, name, args.runs)
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
