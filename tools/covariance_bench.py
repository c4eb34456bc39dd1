"""Cost of the parameter covariance (tscm_solver_covariance, csrc/tscm_covariance.cuh) next to one
LM iteration (tscm_solver_time_stage(4)) on the same solver, in the same run.

Workloads: config 3 (8 cameras x 5,000 frames, dense) and the config-4 ring (16 cameras) at its full
100,000 frames.  Per workload: solve, warm up the covariance twice, then `--repeats` timed calls —
the kernels' device time (CUDA events, `kernel_ms`) and the host wall clock of the whole call (it
ends in a device synchronise: plain-residual evaluation, undamped assembly, kernels, copies) —
then one LM iteration timed over `--iters` graph replays.  Writes JSON (with the device name and
power limit) to --out and prints it."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

from tscm_calib_b200 import capi, synth  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(",")]
        return name, power
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})", "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="3,4")
    ap.add_argument("--cfg4-frames", type=int, default=100000)
    ap.add_argument("--repeats", type=int, default=10)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = gpu_info()
    out = {"device": name, "power_limit": power, "workloads": []}
    for cfg in [int(c) for c in a.configs.split(",")]:
        sp = synth.config_batched(4, a.cfg4_frames, processes=8) if cfg == 4 else synth.config(cfg)
        p = sp.problem
        s = capi.Solver(p, capi.default_options())
        s.set_parameters(sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
        res = s.run()
        sol = s.get_parameters()
        for _ in range(2):
            s.covariance()
        kms, wall = [], []
        for _ in range(a.repeats):
            t0 = time.perf_counter()
            cov = s.covariance()
            wall.append((time.perf_counter() - t0) * 1e3)
            kms.append(cov.kernel_ms)
        ok = bool(np.all(np.isfinite(cov.camera)) and np.all(np.isfinite(cov.board)))
        # one LM iteration from the solution, fixed-iteration mode
        s.set_options(capi.default_options(disable_tolerances=1, max_num_iterations=a.iters + 5))
        s.set_parameters(*sol)
        it_ms = s.time_stage(4, a.iters)
        s.close()
        w = {"config": cfg, "cameras": p.num_cameras, "frames": p.num_frames, "views": p.num_views,
             "observations": p.num_observations, "live_camera_parameters": cov.camera.shape[0],
             "solve_iterations": res.num_iterations, "covariance_kernel_ms_median": float(np.median(kms)),
             "covariance_kernel_ms_min": float(np.min(kms)), "covariance_call_ms_median": float(np.median(wall)),
             "lm_iteration_ms": it_ms, "residual_variance": cov.residual_variance, "finite": ok}
        out["workloads"].append(w)
        print(json.dumps(w), flush=True)
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
