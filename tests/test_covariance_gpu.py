"""GPU suite of the parameter covariance (tscm_solver_covariance / tscm_compute_covariance,
csrc/tscm_covariance.cuh) against the dense CPU restatement (tests/covariance_reference.py), across Schur forms, GPUs
and processes, and against its meaning (Monte-Carlo).

Agreement bars: the synthetic rigs' J^T J has an equilibrated condition number kappa of 1e10-1e11
(the triple-sphere xi, lambda, alpha and the focal lengths are strongly correlated), so two correct
inversions that sum in different orders agree to ~kappa * eps only.  Parity is therefore checked to
max(1e-9, 4 kappa eps) on the correlation-normalised blocks and on their diagonals, kappa of the
equilibrated H of the dense restatement; sigma^2 to 1e-12 relative."""
import os
import subprocess
import sys

import numpy as np
import pytest

import covariance_reference as ref
from conftest import ROOT
from tscm_calib_b200 import capi, synth

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps


def device_count():
    import torch
    return torch.cuda.device_count()


def normalised(S):
    d = np.sqrt(np.abs(np.diagonal(S, axis1=-2, axis2=-1)))
    return S / (d[..., :, None] * d[..., None, :])


def agreement_tol(H, floor=1e-9):
    return max(floor, 4.0 * ref.conditioning(H) * EPS)


def config2_tol(oracle, floor):
    sp = synth.config(2)
    return agreement_tol(ref.jtj(oracle, sp.problem, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)[0], floor)


def assert_cov_close(cov, cam, brd, s2, tol, s2_rtol=1e-12):
    np.testing.assert_allclose(normalised(cov.camera), normalised(cam), rtol=0, atol=tol)
    np.testing.assert_allclose(np.diag(cov.camera), np.diag(cam), rtol=tol)
    np.testing.assert_allclose(normalised(cov.board), normalised(brd), rtol=0, atol=tol)
    np.testing.assert_allclose(np.diagonal(cov.board, axis1=1, axis2=2), np.diagonal(brd, axis1=1, axis2=2),
                               rtol=tol)
    assert cov.residual_variance == pytest.approx(s2, rel=s2_rtol)


CASES = {
    "cfg1": lambda: (synth.config(1), capi.default_options()),
    "cfg2": lambda: (synth.config(2), capi.default_options()),
    "cfg5-huber": lambda: (synth.config(5), capi.default_options(loss_type="huber", loss_scale=1.0)),
    "cfg5-cauchy": lambda: (synth.config(5), capi.default_options(loss_type="cauchy", loss_scale=1.0)),
    "ragged": lambda: (synth.generate(num_cameras=4, num_frames=60, board=(7, 5), rig="calib", seed=71),
                       capi.default_options()),
    "ring16": lambda: (synth.config(4, num_frames=300), capi.default_options(max_num_iterations=15)),
}


@pytest.mark.parametrize("point", ["initial", "solved"])
@pytest.mark.parametrize("case", list(CASES))
def test_covariance_matches_oracle(oracle, case, point):
    sp, opt = CASES[case]()
    x = (sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    s = capi.Solver(sp.problem, opt)
    s.set_parameters(*x)
    if point == "solved":
        s.run()
        x = s.get_parameters()
    cov = s.covariance()
    s.close()
    assert cov.camera.shape == (len(capi.live_columns(sp.problem)),) * 2 and cov.kernel_ms > 0
    rc, cam, brd, s2, H = ref.covariance(oracle, sp.problem, *x, options=opt)
    assert rc == 0
    assert_cov_close(cov, cam, brd, s2, agreement_tol(H))


def test_schur_forms_agree(oracle):
    sp = synth.config(2)
    out = {}
    for form in ("rows", "fused", "pairs"):
        s = capi.Solver(sp.problem, capi.default_options(), schur_form=form)
        s.set_parameters(sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
        out[form] = s.covariance()
        s.close()
    base = out["rows"]
    tol = config2_tol(oracle, 1e-12)
    for form in ("fused", "pairs"):
        assert_cov_close(out[form], base.camera, base.board, base.residual_variance, tol=tol)


def test_rank_deficient_gauge_is_reported_and_solver_still_runs():
    sp = synth.config(2)
    p = sp.problem
    q = capi.ProblemArrays(p.board_xy, p.view_camera, p.view_frame, p.obs_xy, p.num_cameras, p.num_frames,
                           fixed_camera=-1)
    s = capi.Solver(q, capi.default_options(max_num_iterations=5))
    s.set_parameters(sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    with pytest.raises(capi.TscmError) as e:
        s.covariance()
    assert e.value.code == capi.ERR_RANK_DEFICIENT and "rank deficient" in str(e.value)
    res = s.run()
    assert res.num_iterations > 1 and np.isfinite(res.final_cost)
    s.close()


def test_no_side_effects_on_a_later_run():
    sp = synth.config(2)
    opt = capi.default_options(loss_type="huber", loss_scale=1.0)
    x = (sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    traces = []
    for with_cov in (False, True):
        s = capi.Solver(sp.problem, opt)
        s.set_parameters(*x)
        s.run()
        if with_cov:
            s.covariance()
        traces.append((s.run(), s.get_parameters()))
        s.close()
    (a, pa), (b, pb) = traces
    for k in ("cost", "radius", "gradient_max_norm", "step_norm", "step_flags"):
        np.testing.assert_array_equal(getattr(a, k), getattr(b, k))
    for u, v in zip(pa, pb):
        np.testing.assert_array_equal(u, v)


def test_one_shot_after_solve_equals_resident():
    sp = synth.config(2)
    opt = capi.default_options()
    capi.cache_release()
    a, b, c, _ = capi.solve(sp.problem, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt, opt, device=0)
    one = capi.covariance(sp.problem, a, b, c, opt, device=0)
    s = capi.Solver(sp.problem, opt, device=0)
    s.set_parameters(a, b, c)
    res = s.covariance()
    s.close()
    np.testing.assert_array_equal(one.camera, res.camera)
    np.testing.assert_array_equal(one.board, res.board)
    assert one.residual_variance == res.residual_variance
    capi.cache_release()


def test_monte_carlo_meaning():
    """Start at ground truth, solve 300 noise draws (sigma = 0.1 px) through the cached solver with
    the default options: the empirical variance of the well-determined live camera parameters (every
    free rt, cx, cy) matches sigma^2 diag(Sigma), and the residual variance matches sigma^2.
    fx, fy, xi, lambda and alpha are left out: this rig determines them only weakly (predicted
    sigma of 50-85 px for fx, fy and of twice lambda itself), far outside the range in which any
    linearisation describes the estimator, and Ceres' default tolerances stop the solves short
    along that valley."""
    sp = synth.config(2, perturb=0)
    p = sp.problem
    opt = capi.default_options()
    gt = (sp.gt_intrinsics, sp.gt_cam_rt, sp.gt_board_rt)
    uv = synth.generate(num_cameras=4, num_frames=200, board=(11, 8), rig="calib", seed=2, noise_px=0.0).problem.obs_xy
    s = capi.Solver(p, opt)
    s.set_parameters(*gt)
    cov = s.covariance(boards=False)
    rng = np.random.default_rng(20261020)
    cols = capi.live_columns(p)
    keep = np.array([k < 6 or k in (8, 9) for _, k in cols])
    xs, s2s = [], []
    for _ in range(300):
        s.set_observations(uv + 0.1 * rng.standard_normal(uv.shape))
        s.set_parameters(*gt)
        s.run()
        intr, cam_rt, _ = s.get_parameters()
        xs.append([cam_rt[m, k] if k < 6 else intr[m, k - 6] for m, k in cols])
        s2s.append(s.covariance(boards=False).residual_variance)
    s.close()
    emp = np.var(np.array(xs), axis=0, ddof=1)[keep]
    pred = 0.01 * np.diag(cov.camera)[keep]
    ratio = emp / pred
    assert keep.sum() == 3 * 6 + 4 * 2
    assert np.all((ratio > 0.6) & (ratio < 1.6)), ratio
    assert 0.85 < ratio.mean() < 1.15, ratio.mean()
    assert abs(np.mean(s2s) / 0.01 - 1) < 0.05


@pytest.mark.parametrize("n", [2, 4])
def test_num_gpus_equals_one_gpu(oracle, n):
    if device_count() < n:
        pytest.skip(f"needs {n} GPUs")
    sp = synth.config(2)
    x = (sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    one = capi.Solver(sp.problem, capi.default_options(), device=0)
    one.set_parameters(*x)
    r1 = one.covariance()
    one.close()
    s = capi.Solver(sp.problem, capi.default_options(num_gpus=n), device=0)
    s.set_parameters(*x)
    rn = s.covariance()
    s.close()
    assert_cov_close(rn, r1.camera, r1.board, r1.residual_variance, config2_tol(oracle, 1e-10))


@pytest.mark.parametrize("world", [2])
def test_multi_process_ranks_match_one_gpu(world):
    if device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", str(29611 + world),
           os.path.join(ROOT, "tools", "dist_covariance.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0 and "DIST COVARIANCE PASS" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


def test_full_size_config3():
    sp = synth.config(3)
    s = capi.Solver(sp.problem, capi.default_options())
    s.set_parameters(sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    s.run()
    cov = s.covariance()
    s.close()
    assert cov.kernel_ms > 0
    # the camera block is positive definite to within its conditioning (its smallest eigenvalues
    # sit ~1e-17 below its largest): positive semi-definite after normalisation, up to roundoff;
    # the 6 x 6 board blocks are well conditioned and strictly positive definite
    for M in [cov.camera] + list(cov.board):
        assert np.all(np.isfinite(M))
        np.testing.assert_allclose(M, M.T, rtol=0, atol=1e-12 * np.max(np.abs(M)))
    assert np.linalg.eigvalsh(normalised(cov.camera)).min() > -1e-9
    assert np.all(np.diag(cov.camera) > 0)
    assert np.linalg.eigvalsh(cov.board).min() > 0
    assert cov.residual_variance == pytest.approx(0.01, rel=0.05)


def build_adapter_wrapper(out_dir):
    """tests/hostmath/multicalib_covariance.cpp + the C++ adapter, linked against the library,
    built into `out_dir` (a temporary directory: the tree may be read-only)."""
    import ctypes as C
    from tscm_calib_b200 import build as tbuild
    lib = tbuild.build_cuda()
    host = os.path.join(ROOT, "tscm_calib_b200", "host")
    srcs = [os.path.join(ROOT, "tests", "hostmath", "multicalib_covariance.cpp"),
            os.path.join(host, "ts_camera.cpp"), os.path.join(host, "multi_calib_b200.cpp")]
    out = os.path.join(str(out_dir), "libmulticalib_covariance.so")
    env = dict(os.environ)
    env.pop("CXX", None)
    libdir = os.path.dirname(lib)
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", out] + srcs +
                   ["-L" + libdir, "-ltscm_b200", "-Wl,-rpath," + libdir], check=True, env=env)
    return C.CDLL(out)


def test_adapter_compute_covariance_matches_capi(tmp_path):
    """MultiCalib::compute_covariance (host/multi_calib_b200.cpp) through a C wrapper."""
    from tscm_calib_b200.capi import _dp, _ip
    wrapper = build_adapter_wrapper(tmp_path)
    sp = synth.config(2)
    p = sp.problem
    Cn, F = p.num_cameras, p.num_frames
    intr = np.ascontiguousarray(sp.init_intrinsics, dtype=np.float64).copy()
    cam_rt = np.ascontiguousarray(sp.init_cam_rt, dtype=np.float64).copy()
    board_rt = np.ascontiguousarray(sp.init_board_rt, dtype=np.float64).copy()
    cam_sd, board_sd = np.zeros((Cn, 15)), np.zeros((F, 6))
    rc = wrapper.multicalib_covariance(
        Cn, F, p.corners_per_board, p.num_views, _dp(p.board_xy), _ip(p.view_camera), _ip(p.view_frame),
        _dp(p.obs_xy), _dp(intr), _dp(cam_rt), _dp(board_rt), _dp(cam_sd), _dp(board_sd))
    assert rc == 1
    # the same solve and covariance through the C-ABI
    a, b, c, _ = capi.solve(p, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt, capi.default_options())
    np.testing.assert_allclose(intr, a, rtol=1e-12)
    cov = capi.covariance(p, a, b, c, capi.default_options())
    np.testing.assert_allclose(cam_sd, capi.camera_std_dev(p, cov), rtol=1e-9, atol=0)
    bsd = np.sqrt(cov.residual_variance * np.diagonal(cov.board, axis1=1, axis2=2))
    np.testing.assert_allclose(board_sd, bsd, rtol=1e-9, atol=0)
