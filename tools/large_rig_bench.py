"""Timing of the large-rig path (tscm_options.allow_large_rigs, DESIGN.md 5f) on one GPU.

Stage 2 (the reduced solve alone) for the single CTA and the cluster form at NL 98 and 202, and for
the cluster form at NL 208 to 416; stage 4 (one whole LM iteration from the captured graph) for a
32-camera dense array and a 32-camera ring; one covariance call at NL 410.  Times are CUDA events
around `repeats` launches after a warm-up of the same shape.  The device name and power limit are
read in the same run.

    python tools/large_rig_bench.py --out profiles/r04_large_rig_bench.json
"""
import argparse
import dataclasses
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tscm_calib_b200 import capi, synth  # noqa: E402


def device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = (v.strip() for v in q.stdout.splitlines()[0].split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def rig(num_cameras, num_frames, fixed_camera=0, kind="array"):
    if kind == "array":
        sp = synth.generate(num_cameras=num_cameras, num_frames=num_frames, rig="array", dense=True,
                            seed=40 + num_cameras)
    else:
        sp = synth.generate(num_cameras=num_cameras, num_frames=num_frames, rig="ring", seed=70 + num_cameras)
    if fixed_camera != 0:
        p = sp.problem
        q = capi.ProblemArrays(p.board_xy, p.view_camera, p.view_frame, p.obs_xy, p.num_cameras, p.num_frames,
                               fixed_camera=fixed_camera)
        sp = dataclasses.replace(sp, problem=q)
    return sp


def opts(**kw):
    return capi.default_options(allow_large_rigs=1, disable_tolerances=1, max_num_iterations=1 << 20, **kw)


def stage(sp, st, repeats, form="auto"):
    s = capi.Solver(sp.problem, opts())
    try:
        s.set_reduced_solve(form)
        s.set_parameters(sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
        s.time_stage(st, max(3, repeats // 10))                 # warm-up of this shape
        s.set_parameters(sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
        return s.time_stage(st, repeats), s.reduced_size()
    finally:
        s.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--repeats", type=int, default=200)
    a = ap.parse_args()
    res = {"device": device_info(), "stage2": [], "stage4": [], "covariance": None}
    for C, fixed in ((8, 0), (16, 0)):
        sp = rig(C, 60, fixed)
        for form in ("single", "cluster"):
            ms, nl = stage(sp, 2, a.repeats, form)
            res["stage2"].append({"NL": nl, "cameras": C, "form": form, "ms": ms})
            print("stage 2", nl, form, f"{ms * 1e3:.1f} us", flush=True)
    for C, fixed in ((16, -1), (20, 0), (24, 11), (32, 31), (32, -1)):
        ms, nl = stage(rig(C, 30, fixed), 2, a.repeats, "auto")
        res["stage2"].append({"NL": nl, "cameras": C, "form": "cluster", "ms": ms})
        print("stage 2", nl, "cluster", f"{ms * 1e3:.1f} us", flush=True)
    for kind, F in (("array", 2000), ("ring", 20000)):
        sp = rig(32, F, 0, kind)
        ms, nl = stage(sp, 4, 50)
        res["stage4"].append({"rig": kind, "cameras": 32, "frames": F, "views": int(sp.problem.num_views), "NL": nl,
                              "ms_per_iteration": ms})
        print("stage 4", kind, F, f"{ms:.3f} ms", flush=True)
    sp = rig(32, 30, 31)
    s = capi.Solver(sp.problem, opts())
    s.set_parameters(sp.gt_intrinsics, sp.gt_cam_rt, sp.gt_board_rt)
    s.covariance()                                               # warm-up (allocations)
    t = time.perf_counter()
    cov = s.covariance()
    call_ms = (time.perf_counter() - t) * 1e3
    s.close()
    res["covariance"] = {"NL": int(cov.camera.shape[0]), "kernel_ms": cov.kernel_ms, "call_ms": call_ms,
                         "finite": bool(np.isfinite(cov.camera).all())}
    print("covariance", res["covariance"], flush=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
