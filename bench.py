#!/usr/bin/env python
"""bench.py — LM iterations/s and residual+Jacobian Gobs/s of the calibration solve.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

A "step" is ONE Levenberg-Marquardt iteration (Schur elimination, reduced solve,
back-substitution, residual+Jacobian+normal-equation pass at the candidate point,
accept/reject) over BASELINE.json config 3: 8 cameras x 5,000 frames x 88 corners =
3.52 M observations, synthetic, generated through the TS model.

Scaling is STRONG, as BASELINE.json names it ("5,000 frames ... sharded across 8 B200"): the
5,000 frames of the ONE config-3 problem are dealt to the N ranks (one process per GPU), the
reduced camera system and the evaluation record are exchanged by this library's own kernels
over NVLink peer memory each iteration.  `value` = 3.52 M observations x LM iterations / s.
The weak-scaling figure of round 1 (5,000 frames per GPU) is reported beside it as `weak`.

The JSON line also carries:
  lm_iterations_per_sec   the other half of BASELINE.json's metric
  parity_check            N > 1: the sharded solve (default Ceres options, run to convergence)
                          against the 1-GPU solve of the same problem — iteration counts,
                          per-iteration cost, final parameters; N = 1: the GPU solve of the
                          cpu_baseline sample against the oracle's
  roofline                the dominant kernel (k_eval5) against measured HBM peak, plus
                          roofline_fp64 against the measured DFMA peak (the kernel is
                          FP64-pipe bound, SURVEY.md §8d)
  cpu_baseline            the CPU oracle (Ceres-semantics port) timed on this box
  e2e                     the same metric through ONE tscm_solve() call — the call the
                          reference adapters make in place of ceres::Solve — with HOST buffers;
                          at N > 1 rank 0 alone makes the call with options.num_gpus = N
  masked (N = 1)          config 3 with per-frame all-or-nothing visibility masks
  stress_cfg4_sample      (N = 1) a 20,000-frame sample of BASELINE config 4's generator
                          (16-camera ring, sparse visibility: the per-camera-pair Schur form)

`--impl reference` times the CPU restatement of the reference's Ceres path (the
reference itself cannot be built: Ceres/Eigen/OpenCV are absent) on the host cores.

`--dump-outputs DIR` writes the parameters the timed LM iterations end at, as a caller of the
solve receives them, to DIR/intrinsics.npy (C x 9), DIR/cam_rt.npy (C x 6) and DIR/board_rt.npy
(F x 6), float64.  The workload is synthesised from fixed seeds, so two builds run with the same
arguments can be compared file for file.
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

sys.dont_write_bytecode = True      # the tree may be read-only; the benchmark leaves nothing in it
ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOAD = "config3: 8 cameras x 5000 frames x 88 corners (3.52M observations), dense visibility"
METRIC = "LM residual+Jacobian throughput at 3.52M corner observations"
UNIT = "Gobs/s"
ALG_BYTES_PER_OBS_EVAL = 24.0   # SURVEY.md §8(d): J-pass with per-view blocks materialised
ALG_FLOPS_PER_OBS_EVAL = 1060.0  # SURVEY.md §8(d): forward 130 + Jacobian 250 + outer products 680
STEP = ("one LM iteration (Schur + reduced solve + back-substitution + residual/Jacobian/"
        "normal-equation pass + accept/reject)")
L2_NOTE = ("per-step working set at N = 1 (observations 56 MB, moment buffer 60 MB, per-view records "
           "2 x 34 MB, Schur rows 48 MB) exceeds the 126 MB L2; no explicit flush")


def config_block(world: int, **extra):
    """The `config` object: the SAME keys on both arms (the driver compares them)."""
    c = {"workload": WORKLOAD, "observations_total": 3520000, "observations_per_gpu": 3520000 // max(1, world),
         "step": STEP, "l2": L2_NOTE,
         "parallelism": (f"strong: the 5000 frames are sharded over {world} GPU(s), one process per GPU; "
                         "[S | rhs] and the evaluation record are exchanged by this library's kernels over "
                         "NVLink peer memory (CUDA IPC)") if world > 1 else "single GPU",
         "sample": None}
    c.update(extra)
    return c


def captured_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture
    (profiles/r*_traffic.json, written by tools/make_profile_summary.py); None if absent."""
    import glob
    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json"))):
        try:
            with open(path) as f:
                d = json.load(f)
            if kernel in d:
                best = d[kernel]["dram_bytes"]
        except Exception:
            pass
    return best


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "100", "-i", str(self.device)], stdout=subprocess.PIPE,
                stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 8:
                for name, val in zip(names, r[4:8]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def write_outputs(directory, intrinsics, cam_rt, board_rt):
    """--dump-outputs: the solved parameters as DIR/<name>.npy, float64."""
    os.makedirs(directory, exist_ok=True)
    for name, a in (("intrinsics", intrinsics), ("cam_rt", cam_rt), ("board_rt", board_rt)):
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def fixed_iteration_options(n, **kw):
    from tscm_calib_b200 import capi
    return capi.default_options(max_num_iterations=int(n), disable_tolerances=1, **kw)


def time_oracle(problem, intr, cam_rt, board_rt, iterations, threads):
    from oracle import oracle
    opt = fixed_iteration_options(iterations)
    t0 = time.perf_counter()
    a, b, c, s = oracle.solve(problem, intr, cam_rt, board_rt, opt, num_threads=threads)
    dt = time.perf_counter() - t0
    assert s.num_iterations == iterations + 1, s
    return dt, (a, b, c, s)


REFERENCE_NOTE = ("the reference's own ceres::Solve cannot be built here (Ceres, Eigen, OpenCV absent); this is the "
                  "oracle port: Ceres semantics, SCALAR dual-number Jets (real Ceres vectorises Jets with Eigen and "
                  "may be a small integer factor faster per thread), frames over std::thread; the reference itself "
                  "never sets num_threads, i.e. runs ONE thread")


def run_reference(args):
    """The reference arm: CPU restatement of the reference's Ceres path on the host cores."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from tscm_calib_b200 import synth
    threads = os.cpu_count() or 1
    frames = args.reference_frames
    sp = synth.config(3, num_frames=frames)
    if args.warmup > 0:
        time_oracle(sp.problem, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt, min(args.warmup, 1), threads)
    dt, (a, b, c, _) = time_oracle(sp.problem, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt, args.steps,
                                   threads)
    if args.dump_outputs:
        write_outputs(args.dump_outputs, a, b, c)
    gobs = sp.num_observations * args.steps / dt / 1e9
    sample = (f"{frames} of 5000 frames of config 3 ({sp.num_observations} observations), "
              f"{args.steps} LM iterations incl. iteration-0 evaluation, {threads} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": gobs, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": config_block(max(world, args.gpus), sample=sample),
        "lm_iterations_per_sec_at_sample": args.steps / dt,
        "lm_iterations_per_sec_at_3.52M": gobs * 1e9 / 3.52e6,
        "cpu_baseline": {"value": gobs, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "note": REFERENCE_NOTE},
        "e2e": {"value": gobs, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def oracle_solve(problem, intr, cam_rt, board_rt, opt, threads):
    from oracle import oracle
    return oracle.solve(problem, intr, cam_rt, board_rt, opt, num_threads=threads)


def rel(a, b, floor=1e-9):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / (np.abs(b) + floor))) if a.size else 0.0


def compare_solves(res, ref, params, ref_params):
    n = min(len(res.cost), len(ref.cost))
    out = {
        "iterations": [int(res.num_iterations), int(ref.num_iterations)],
        "termination": [res.termination, ref.termination],
        "cost_rel": float(np.max(np.abs(res.cost[:n] - ref.cost[:n]) / ref.cost[:n])) if n else None,
        "param_rel": max(rel(x, y) for x, y in zip(params, ref_params)),
    }
    out["ok"] = bool(out["iterations"][0] == out["iterations"][1] and out["termination"][0] == out["termination"][1]
                     and out["cost_rel"] is not None and out["cost_rel"] <= 1e-9 and out["param_rel"] <= 1e-7)
    return out


def run_b200(args):
    import torch
    import torch.distributed as dist
    from tscm_calib_b200 import capi, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the calibration solve has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"        # the version banner would land on stdout next to the JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        cpu_group = dist.new_group(backend="gloo")   # host-side waits that keep the other GPUs idle
    capi.load_library()
    if args.debug_flags:
        capi.set_debug(args.debug_flags)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- the workload: ONE config-3 problem, its frames dealt to the ranks --------------------
    sp = synth.config(3, num_frames=args.frames)
    total_obs = sp.num_observations
    if world > 1:
        problem, fr = synth.shard_frames(sp, rank, world)
    else:
        problem, fr = sp.problem, np.arange(sp.problem.num_frames)
    intr, cam_rt, board_rt = sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt[fr]
    total_iters = args.warmup + args.steps
    opt = fixed_iteration_options(total_iters + 8)
    solver = capi.Solver(problem, opt, device=local_rank)
    if world > 1:
        capi.attach_ranks(solver, rank, world)
    solver.set_parameters(intr, cam_rt, board_rt)

    # ---- warm-up, then EXACTLY `steps` LM iterations, device-timed ------------------
    if args.warmup > 0:
        solver.time_stage(4, args.warmup)
        solver.set_parameters(intr, cam_rt, board_rt)     # restart from the same initial point
    barrier()
    launches0 = solver.launch_count()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_iter = solver.time_stage(4, args.steps)      # CUDA events on the solver's stream
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = solver.launch_count() - launches0
    if args.dump_outputs:
        # the point the last timed iteration left on the device; at N > 1 every rank holds the
        # board poses of its own frames, gathered on rank 0 into the order of the whole problem
        intr_out, cam_out, board_out = solver.get_parameters()
        if world > 1:
            parts = [None] * world
            dist.all_gather_object(parts, (fr, board_out), group=cpu_group)
            board_out = np.zeros((sp.problem.num_frames, 6))
            for frames, part in parts:
                board_out[frames] = part
        if rank == 0:
            write_outputs(args.dump_outputs, intr_out, cam_out, board_out)
    ms_iter = max_over_ranks(ms_iter)
    it_per_s = 1e3 / ms_iter
    value = total_obs * it_per_s / 1e9

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_iter, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_block(world, observations_per_gpu=int(problem.num_observations)),
        "lm_iterations_per_sec": it_per_s,
        "gpu_launches": int(launches),
        "clocks": clocks,
    }

    # ---- roofline of the dominant kernel, timed alone with CUDA events ----------------------
    # The J-pass (residual + analytic Jacobian + normal-equation blocks) is two kernels:
    # k_eval5 (persistent, per-view moments; the dominant kernel of the iteration) and
    # k_view_blocks (per-view blocks from the moments).  Every rank runs the same stage sequence
    # (the set-up in front of a timed stage contains exchanges); rank 0 reports its shard.
    solver.time_stage(0, 3)
    ms_pass = solver.time_stage(0, 20)
    ms_main = solver.time_stage(6, 20)
    ms_blocks = solver.time_stage(7, 20)
    stages = {}
    for sid, name in ((5, "evaluation_pass"), (1, "schur"), (2, "reduced_solve"), (3, "backsub")):
        solver.time_stage(sid, 2)
        stages[name] = solver.time_stage(sid, 10)
    if rank == 0:
        n_obs = problem.num_observations
        hbm_peak, how = measured_peaks()
        achieved = n_obs * ALG_BYTES_PER_OBS_EVAL / (ms_main * 1e-3) / 1e9
        line["roofline"] = {
            "kernel": "k_eval5", "bound": "hbm", "achieved": achieved, "peak": hbm_peak,
            "unit": "GB/s", "frac": achieved / hbm_peak,
            "traffic": captured_traffic("k_eval5") if world == 1 else None,
            "peak_source": how, "ms_per_launch": ms_main, "observations_per_launch": int(n_obs),
            "algorithmic_bytes_per_observation": ALG_BYTES_PER_OBS_EVAL,
            "note": "k_eval5 is FP64-pipe bound (arithmetic intensity ~44 flop/B vs machine "
                    "balance ~5.3 flop/B); see roofline_fp64.  traffic = DRAM bytes of one launch "
                    "from the committed ncu capture (profiles/)",
        }
        peak_sampler = ClockSampler(local_rank)
        peak_sampler.start()
        fp64_peak = max(capi.device_fp64_peak(local_rank) for _ in range(3))
        peak_clocks = peak_sampler.stop()
        tf = n_obs * ALG_FLOPS_PER_OBS_EVAL / (ms_pass * 1e-3) / 1e12
        line["roofline_fp64"] = {
            "kernel": "k_eval5+k_view_blocks", "bound": "fp64",
            "achieved": tf, "peak": fp64_peak, "unit": "TFLOP/s", "frac": tf / fp64_peak,
            "peak_source": "measured in this run (DFMA microbenchmark, tscm_device_fp64_peak; nominal 148 SM x 64 "
                           "FMA/clk x 2 x 1.965 GHz = 37.2)",
            "peak_clocks": peak_clocks,
            "algorithmic_flops_per_observation": ALG_FLOPS_PER_OBS_EVAL,
            "ms_per_pass": ms_pass, "ms_main_kernel": ms_main, "ms_view_blocks": ms_blocks,
            "whole_iteration_frac": total_obs / world * 1300.0 / (ms_iter * 1e-3) / 1e12 / fp64_peak,
            "note": "SURVEY 8(d)'s 1,060 flop/observation J-pass (projection, Jacobian, normal-equation "
                    "blocks) over the time of the whole pass (both kernels); whole_iteration_frac = 1.3 kflop "
                    "per observation and iteration over ms_per_step",
        }
        line["stage_ms"] = stages
    solver.close()

    # ---- config 3 as BASELINE words it, "with per-frame visibility masks" (N = 1 side figure) -------
    # The headline keeps dense visibility (exactly 3.52 M observations); here every (camera, frame)
    # pair is detected or not as a whole (main.cpp:33-37), which leaves ragged frames for the Schur
    # kernels.
    if world == 1 and not args.no_masked:
        masked = {}
        for rig in ("array", "ring"):       # forward-looking array (almost every board seen), outward ring (a third)
            spm = synth.config(3, num_frames=args.frames, dense=False, rig=rig)
            sm = capi.Solver(spm.problem, fixed_iteration_options(args.warmup + 20 + 8), device=local_rank)
            init_m = (spm.init_intrinsics, spm.init_cam_rt, spm.init_board_rt)
            sm.set_parameters(*init_m)
            sm.time_stage(4, max(args.warmup, 1))
            sm.set_parameters(*init_m)
            ms_m = sm.time_stage(4, 20)
            sm.close()
            masked[rig] = {"value": spm.num_observations / (ms_m * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": ms_m,
                           "observations_total": int(spm.num_observations),
                           "visible_fraction": float(spm.visible.mean())}
            del spm
        line["masked"] = dict(masked["array"], ring=masked["ring"],
                              what="config 3 with all-or-nothing visibility masks per (camera, frame), 20 timed "
                                   "iterations: the forward-looking array rig of the headline, and (`ring`) the same "
                                   "8 cameras looking outward, where a frame is seen by a third of them")

    # ---- BASELINE config 4 (stress: 16-camera ring, visibility masks) on a bounded sample, N = 1 ------
    # The full 100,000 frames take minutes to synthesise on the host (tools/stress_cfg4.py runs them:
    # profiles/r0*_stress_cfg4*.json); a 20,000-frame sample of the same generator exercises the
    # sparse-visibility Schur form (per-camera-pair kernels) inside the driver's run.
    if world == 1 and args.stress_frames > 0:
        sps = synth.config_batched(4, args.stress_frames, batch=10000, processes=min(4, os.cpu_count() or 1))
        ss = capi.Solver(sps.problem, fixed_iteration_options(args.warmup + 10 + 8), device=local_rank)
        init_s = (sps.init_intrinsics, sps.init_cam_rt, sps.init_board_rt)
        ss.set_parameters(*init_s)
        ss.time_stage(4, max(args.warmup, 1))
        ss.set_parameters(*init_s)
        ms_s = ss.time_stage(4, 10)
        ss.close()
        line["stress_cfg4_sample"] = {
            "value": sps.num_observations / (ms_s * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": ms_s,
            "observations_total": int(sps.num_observations), "frames": int(args.stress_frames),
            "visible_fraction": float(sps.visible.mean()),
            "what": f"config 4 generator (16-camera ring, masks) at {args.stress_frames} of its 100,000 frames, "
                    "10 timed LM iterations; the full size on 1/2/4/8 GPUs: profiles/r0*_stress_cfg4*.json"}
        del sps

    # ---- weak scaling beside it (N > 1): 5,000 frames per GPU, one common rig ------------------------
    if world > 1 and not args.no_weak:
        spw = synth.config(3, num_frames=args.frames, frame_seed=rank)
        sw = capi.Solver(spw.problem, fixed_iteration_options(args.warmup + 20 + 8), device=local_rank)
        capi.attach_ranks(sw, rank, world)
        sw.set_parameters(spw.init_intrinsics, spw.init_cam_rt, spw.init_board_rt)
        sw.time_stage(4, args.warmup)
        sw.set_parameters(spw.init_intrinsics, spw.init_cam_rt, spw.init_board_rt)
        barrier()
        ms_w = max_over_ranks(sw.time_stage(4, 20))
        barrier()
        sw.close()
        line["weak"] = {"value": spw.num_observations * world / (ms_w * 1e-3) / 1e9, "unit": UNIT,
                        "ms_per_step": ms_w, "observations_total": int(spw.num_observations * world),
                        "what": "5,000 frames per GPU (3.52 M observations each), 20 timed iterations"}
        del spw

    # ---- parity inside the run ---------------------------------------------------------------------
    # N > 1: the sharded solve with the reference's options (Ceres defaults, 50 iterations, run to
    # convergence) against the 1-GPU solve of the same 5,000-frame problem on rank 0.
    popt = capi.default_options()
    if world > 1:
        ps_ = capi.Solver(problem, popt, device=local_rank)
        capi.attach_ranks(ps_, rank, world)
        ps_.set_parameters(intr, cam_rt, board_rt)
        res = ps_.run()
        pa, pb, pc = ps_.get_parameters()
        per_cam, overall, rms = ps_.reprojection_error()
        ps_.close()
        barrier()
        if rank == 0:
            a1, b1, c1, ref = capi.solve(sp.problem, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt, popt,
                                         device=local_rank)
            s1 = capi.Solver(sp.problem, popt, device=local_rank)
            s1.set_parameters(a1, b1, c1)
            _, overall1, rms1 = s1.reprojection_error()
            s1.close()
            chk = compare_solves(res, ref, (pa, pb, pc), (a1, b1, c1[fr]))
            chk["rms_px"] = [rms, rms1]
            chk["rms_abs_diff"] = abs(rms - rms1)
            chk["ok"] = bool(chk["ok"] and chk["rms_abs_diff"] <= 1e-9)
            chk["what"] = (f"config 3 sharded over {world} ranks vs the same problem on 1 GPU: default options, "
                           "to convergence; bars: iterations and termination equal, cost per iteration 1e-9 "
                           "relative, parameters 1e-7 relative, RMS reprojection error 1e-9 px")
            line["parity_check"] = chk
        barrier()

    # ---- end to end through ONE tscm_solve() call with HOST buffers ---------------------------------
    # The call a reference adapter makes instead of ceres::Solve (multi_calib.cpp:216): problem
    # description, observations (page-locked host memory from tscm_host_alloc) and the initial
    # parameters in, parameters and summary out.  The first call builds the solver for this problem
    # structure, the timed call finds it in the library's cache (a re-calibration).  At N > 1 rank 0
    # alone calls, with options.num_gpus = N: the single-process path MultiCalib::calibrate() takes.
    e2e_iters = args.steps
    barrier()
    if rank == 0:
        obs = capi.pinned_array(sp.problem.obs_xy.shape)
        obs[...] = sp.problem.obs_xy
        hp = capi.ProblemArrays(sp.problem.board_xy, sp.problem.view_camera, sp.problem.view_frame, obs,
                                sp.problem.num_cameras, sp.problem.num_frames, sp.problem.fixed_camera)
        e_opt = fixed_iteration_options(e2e_iters, num_gpus=world)
        init = (sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
        t0 = time.perf_counter()
        capi.solve(hp, *init, e_opt, device=0 if world > 1 else local_rank)
        dt_cold = time.perf_counter() - t0
        times = []
        for _ in range(3):
            t0 = time.perf_counter()
            a, b, c, r = capi.solve(hp, *init, e_opt, device=0 if world > 1 else local_rank)
            times.append(time.perf_counter() - t0)
        dt = float(np.median(times))
        assert r.num_iterations == e2e_iters + 1
        h2d = hp.obs_xy.nbytes + sum(x.nbytes for x in init)
        d2h = a.nbytes + b.nbytes + c.nbytes + 5 * 8 * (e2e_iters + 1)
        line["e2e"] = {
            "value": total_obs * e2e_iters / dt / 1e9, "unit": UNIT,
            "h2d_bytes_per_step": h2d / e2e_iters, "d2h_bytes_per_step": d2h / e2e_iters,
            "lm_iterations_per_sec": e2e_iters / dt, "seconds_per_call": dt,
            "first_call": {"seconds_per_call": dt_cold, "lm_iterations_per_sec": e2e_iters / dt_cold,
                           "what": "the call that also builds the solver (index tables, one arena allocation, "
                                   "graph capture, module load on the first use of a device)"},
            "what": f"one tscm_solve() call = {e2e_iters} LM iterations on host buffers: H2D of the observations "
                    "(page-locked, 56 MB) and initial parameters, on-device transposition, iteration zero, the "
                    "iterations, D2H of parameters and trace; median of 3 calls that reuse the solver the first "
                    "call left in the library's cache; bytes are per call / steps"
                    + (f"; options.num_gpus = {world}, one host thread drives all devices" if world > 1 else ""),
        }
        capi.cache_release()
        del obs, hp
    if world > 1:
        dist.barrier(group=cpu_group)       # the other ranks wait on the HOST: an NCCL barrier would spin on their GPUs

    # ---- CPU baseline beside it (rank 0, N = 1 only) ------------------------------------
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        frames = args.cpu_frames
        spc = sp if frames == args.frames else synth.config(3, num_frames=frames)
        iters = args.cpu_iterations      # ~10-20 s of CPU work on 16 host threads
        dt, _ = time_oracle(spc.problem, spc.init_intrinsics, spc.init_cam_rt, spc.init_board_rt, iters, threads)
        line["cpu_baseline"] = {
            "value": spc.num_observations * iters / dt / 1e9, "unit": UNIT, "cores": threads,
            "kind": "port",
            "sample": f"{frames} of 5000 frames of config 3 ({spc.num_observations} observations), "
                      f"{iters} LM iterations incl. iteration-0 evaluation, Ceres-semantics oracle "
                      f"(dual-number autodiff, dense Schur), {threads} threads, {dt:.1f} s",
            "lm_iterations_per_sec_at_3.52M": spc.num_observations * iters / dt / 3.52e6,
            "note": REFERENCE_NOTE,
        }
        # parity inside the run: a bounded sample solved to convergence with the reference's options
        # (Ceres defaults) by the oracle and by the GPU
        spp = synth.config(3, num_frames=args.parity_frames)
        initp = (spp.init_intrinsics, spp.init_cam_rt, spp.init_board_rt)
        a0, b0, c0, s0 = oracle_solve(spp.problem, *initp, popt, threads)
        a, b, c, s = capi.solve(spp.problem, *initp, popt, device=local_rank)
        chk = compare_solves(s, s0, (a, b, c), (a0, b0, c0))
        chk["what"] = (f"GPU vs the CPU oracle on {args.parity_frames} frames of config 3 ({spp.num_observations} "
                       "observations), default options, to convergence; bars: iterations and termination equal, "
                       "cost per iteration 1e-9 relative, parameters 1e-7 relative")
        line["parity_check"] = chk
        capi.cache_release()
        # the reference never sets Solver::Options::num_threads (Ceres default 1): the same
        # port on ONE thread is the faithful picture of what a reference user runs today
        sp1 = synth.config(3, num_frames=max(1, frames // 10))
        it1 = max(2, iters // 10)
        dt1, _ = time_oracle(sp1.problem, sp1.init_intrinsics, sp1.init_cam_rt, sp1.init_board_rt, it1, 1)
        line["cpu_baseline_single_thread"] = {
            "value": sp1.num_observations * it1 / dt1 / 1e9, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"{sp1.problem.num_frames} of 5000 frames of config 3 ({sp1.num_observations} "
                      f"observations), {it1} LM iterations, 1 thread (Ceres' default num_threads, which the "
                      f"reference leaves in force), {dt1:.1f} s",
            "lm_iterations_per_sec_at_3.52M": sp1.num_observations * it1 / dt1 / 3.52e6,
        }
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=5000, help="frames of config 3 (the whole problem)")
    ap.add_argument("--cpu-iterations", type=int, default=30, help="cpu_baseline LM iterations")
    ap.add_argument("--cpu-frames", type=int, default=5000, help="cpu_baseline sample size (frames)")
    ap.add_argument("--reference-frames", type=int, default=5000, help="--impl reference sample size (frames)")
    ap.add_argument("--parity-frames", type=int, default=1000, help="N = 1 parity_check sample size (frames)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-weak", action="store_true", help="skip the weak-scaling side figure at N > 1")
    ap.add_argument("--no-masked", action="store_true", help="skip the masked-visibility side figure at N = 1")
    ap.add_argument("--stress-frames", type=int, default=20000,
                    help="frames of the config-4 sample timed beside the headline at N = 1 (0 = skip)")
    ap.add_argument("--debug-flags", type=int, default=0, help="tscm_set_debug() flags (4 = no programmatic dependent launch)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the parameters the timed iterations end at to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3
        run_b200(args)


if __name__ == "__main__":
    main()
