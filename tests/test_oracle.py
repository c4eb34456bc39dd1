"""CPU suite: the oracle against the committed golden vectors (independent numpy /
mpmath restatement), against the kernels' host-compiled arithmetic, and against
domain properties.  Tolerances: per-iteration cost 1e-9 rel, parameters 1e-7 rel,
Jacobian 1e-10 (BASELINE.json north_star)."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_options, load_golden, rel_err
from tscm_calib_b200 import capi, synth
from tscm_calib_b200.capi import _dp

GOLDEN_SOLVES = ["mono_cfg1", "rig3_small", "rig4_huber", "rig4_cauchy"]


def hostmath_eval(hostmath, p, intr, cam_rt, board_rt, loss_type=0, loss_scale=1.0):
    N = p.num_observations
    a = np.ascontiguousarray(intr, dtype=np.float64)
    b = np.ascontiguousarray(cam_rt, dtype=np.float64)
    c = np.ascontiguousarray(board_rt, dtype=np.float64)
    r, J, cost = np.zeros((N, 2)), np.zeros((N, 2, 21)), C.c_double()
    rc = hostmath.hostmath_eval_jacobian(C.byref(p.c), _dp(a), _dp(b), _dp(c), loss_type,
                                         C.c_double(loss_scale), _dp(r), _dp(J), C.byref(cost))
    assert rc == 0
    return r, J, cost.value


@pytest.mark.parametrize("name", GOLDEN_SOLVES)
def test_oracle_solve_matches_golden(oracle, name):
    p, z = load_golden(name)
    opt = golden_options(z)
    a, b, c, s = oracle.solve(p, z["init_intrinsics"], z["init_cam_rt"], z["init_board_rt"], opt)
    assert s.termination == str(z["termination"])
    assert s.num_iterations == len(z["cost"])
    np.testing.assert_allclose(s.cost, z["cost"], rtol=1e-9)
    # the radius depends on rho = cost_change / model_cost_change, which is
    # ill-conditioned (relative error ~ eps * cost / cost_change) once the decrease per
    # step is tiny; it is not one of the north-star parity quantities.
    np.testing.assert_allclose(s.radius, z["radius"], rtol=1e-6)
    np.testing.assert_array_equal(s.step_flags, z["flags"])
    np.testing.assert_allclose(s.step_norm, z["step_norm"], rtol=1e-6, atol=1e-12)
    assert rel_err(a, z["final_intrinsics"], 1e-9) < 1e-7
    assert rel_err(b, z["final_cam_rt"], 1e-9) < 1e-7
    assert rel_err(c, z["final_board_rt"], 1e-9) < 1e-7


@pytest.mark.parametrize("name", GOLDEN_SOLVES[:2])
def test_oracle_jets_match_golden_autodiff(oracle, name):
    p, z = load_golden(name)
    r, J, _ = oracle.eval_jacobian(p, z["init_intrinsics"], z["init_cam_rt"], z["init_board_rt"])
    np.testing.assert_allclose(r, z["initial_residuals"], rtol=0, atol=1e-10)
    stride = int(z["jacobian_sample_stride"])
    np.testing.assert_allclose(J[::stride], z["initial_jacobian_sample"], rtol=1e-10, atol=1e-10)


@pytest.mark.parametrize("golden", ["jacobian_mpmath", "jacobian_sympy"])
def test_jets_and_analytic_jacobian_match_mpmath(oracle, hostmath, golden):
    """50-digit central differences (mpmath) and sympy's SYMBOLIC derivative of the functor
    multi_calib.h:146-195 (make_golden_sympy.py: nothing hand-derived) pin both the Jet autodiff
    and the hand-derived Jacobian, including the theta^2 <= eps Taylor branch of
    AngleAxisRotatePoint."""
    z = np.load(os.path.join(GOLDEN, golden + ".npz"))
    n = len(z["r"])
    taylor = 0
    for k in range(n):
        p = capi.ProblemArrays(z["board"][k][None, :], [0], [0], z["obs"][k][None, None, :], 1, 1,
                               fixed_camera=-1)
        intr, crt, brt = z["intr"][k][None], z["cam_rt"][k][None], z["board_rt"][k][None]
        taylor += int(np.all(brt[0, :3] == 0))
        for r, J, _ in (oracle.eval_jacobian(p, intr, crt, brt),
                        hostmath_eval(hostmath, p, intr, crt, brt)):
            np.testing.assert_allclose(r[0], z["r"][k], rtol=0, atol=1e-10)
            scale = np.maximum(np.abs(z["J"][k]), 1.0)
            assert np.max(np.abs(J[0] - z["J"][k]) / scale) < 1e-10
    assert taylor >= 3


@pytest.mark.parametrize("cfg", [1, 2])
def test_analytic_jacobian_matches_jets(oracle, hostmath, cfg):
    sp = synth.config(cfg)
    args = (sp.problem, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    r0, J0, c0 = oracle.eval_jacobian(*args)
    r, J, c = hostmath_eval(hostmath, *args)
    np.testing.assert_allclose(r, r0, rtol=0, atol=1e-10)
    assert np.max(np.abs(J - J0) / np.maximum(np.abs(J0), 1.0)) < 1e-10
    assert abs(c - c0) <= 1e-12 * c0
    # the constant block has no Jacobian columns (multi_calib.cpp:186)
    fixed = np.repeat(sp.problem.view_camera == 0, sp.problem.corners_per_board)
    assert np.all(J[fixed][:, :, :6] == 0) and np.all(J0[fixed][:, :, :6] == 0)
    # skew columns b, c are structurally zero (TS.h:122-125)
    assert np.all(J0[:, :, 19:] == 0)


def test_mono_functor_equals_rig_functor_with_identity_camera(oracle):
    """TS.h:100-131 == multi_calib.h:146-195 with camera_rt = 0, bit for bit."""
    sp = synth.config(1)
    p = sp.problem
    r_rig, J_rig, c_rig = oracle.eval_jacobian(p, sp.init_intrinsics, np.zeros((1, 6)),
                                               sp.init_board_rt)
    r_mono, J_mono, c_mono = oracle.eval_jacobian_mono(p, sp.init_intrinsics, sp.init_board_rt)
    np.testing.assert_array_equal(r_rig, r_mono)
    assert abs(c_rig - c_mono) <= 4e-16 * c_rig * 8   # same terms, different summation order
    np.testing.assert_array_equal(J_rig[:, :, 12:21], J_mono[:, :, 0:9])   # intrinsic block
    np.testing.assert_array_equal(J_rig[:, :, 6:12], J_mono[:, :, 9:15])   # board pose block


def test_zero_noise_recovers_ground_truth(oracle):
    sp = synth.generate(num_cameras=3, num_frames=40, board=(11, 8), rig="calib", seed=31,
                        noise_px=0.0)
    opt = capi.default_options(max_num_iterations=100, function_tolerance=1e-14,
                               parameter_tolerance=1e-14)
    a, b, c, s = oracle.solve(sp.problem, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt, opt)
    assert s.final_cost < 1e-12 * s.initial_cost
    _, _, rms = oracle.reprojection_error(sp.problem, a, b, c)
    assert rms < 1e-6
    assert rel_err(b[1:], sp.gt_cam_rt[1:], 1e-3) < 1e-4


def test_reprojection_error_readout(oracle):
    """multi_calib.cpp:235-283: mean Euclidean error; RMS = sqrt(2 cost / N) without loss."""
    sp = synth.config(2)
    p = sp.problem
    per, overall, rms = oracle.reprojection_error(p, sp.gt_intrinsics, sp.gt_cam_rt, sp.gt_board_rt)
    r, _, cost = oracle.eval_jacobian(p, sp.gt_intrinsics, sp.gt_cam_rt, sp.gt_board_rt)
    e = np.sqrt((r * r).sum(axis=1))
    assert abs(overall - e.mean()) < 1e-9
    assert abs(rms - np.sqrt(2 * cost / len(e))) < 1e-9
    cam = np.repeat(p.view_camera, p.corners_per_board)
    for m in range(p.num_cameras):
        assert abs(per[m] - e[cam == m].mean()) < 1e-9
    assert 0.10 < overall < 0.15            # 0.1 px noise per axis


def test_project_matches_synth_projection(oracle):
    """TS.cpp:332-344 restated twice (C++ oracle, numpy generator)."""
    rng = np.random.default_rng(3)
    pts = rng.normal(0, 300, (200, 3)) + np.array([0, 0, 500.0])
    intr = synth.CALIB_INTRINSICS[1].copy()
    intr[7:] = [0.3, -0.2]                   # skew terms are part of project()
    uv, _ = synth.ts_project(intr, pts)
    np.testing.assert_allclose(oracle.project(intr, pts), uv, rtol=1e-13, atol=1e-10)


def test_loss_correction_against_numpy(oracle, hostmath):
    from oracle import numpy_ref as nr
    sp = synth.generate(num_cameras=2, num_frames=8, board=(6, 5), rig="calib", seed=41,
                        outlier_fraction=0.2)
    p = sp.problem
    P = nr.Problem.from_arrays(p)
    r, J = nr.evaluate(P, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    for kind in (1, 2):
        cost, rc, Jc = nr.apply_loss(kind, 1.5, r, J)
        r1, J1, c1 = hostmath_eval(hostmath, p, sp.init_intrinsics, sp.init_cam_rt,
                                   sp.init_board_rt, kind, 1.5)
        np.testing.assert_allclose(r1, rc, rtol=1e-12, atol=1e-10)
        assert np.max(np.abs(J1[:, :, :19] - Jc[:, :, :19]) / np.maximum(np.abs(Jc[:, :, :19]), 1.0)) < 1e-10
        assert abs(c1 - cost) < 1e-12 * cost


def test_reduced_system_is_schur_complement_of_dense_normal_equations(oracle):
    """SchurEliminator output == dense J^T J + D^2 Schur complement (numpy)."""
    from oracle import numpy_ref as nr
    sp = synth.generate(num_cameras=3, num_frames=12, board=(6, 5), rig="calib", seed=51)
    p = sp.problem
    radius = 1e4
    lhs, rhs = oracle.reduced_system(p, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt, radius)
    P = nr.Problem.from_arrays(p)
    L = nr.Layout(P)
    r, J = nr.evaluate(P, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    col = L.column_index()
    Jd = np.zeros((2 * len(col), L.n))
    for a in range(2):
        for k in range(21):
            ok = col[:, k] >= 0
            Jd[2 * np.nonzero(ok)[0] + a, col[ok, k]] = J[ok, a, k]
    scale = 1.0 / (1.0 + np.sqrt((Jd * Jd).sum(axis=0)))
    Js = Jd * scale
    H = Js.T @ Js
    D2 = np.clip(np.diag(H), 1e-6, 1e32) / radius
    A = H + np.diag(D2)
    g = Js.T @ r.reshape(-1)
    ne = L.n_e
    Aee, Aef, Aff = A[:ne, :ne], A[:ne, ne:], A[ne:, ne:]
    S = Aff - Aef.T @ np.linalg.solve(Aee, Aef)
    b = g[ne:] - Aef.T @ np.linalg.solve(Aee, g[:ne])
    sc = np.sqrt(np.abs(np.diag(S)))
    assert np.max(np.abs(lhs - S) / np.outer(sc, sc)) < 1e-9
    assert np.max(np.abs(rhs - b)) / np.max(np.abs(b)) < 1e-9


def test_oracle_multithreaded_equals_single_thread(oracle):
    sp = synth.generate(num_cameras=4, num_frames=60, board=(11, 8), rig="calib", seed=61)
    opt = capi.default_options()
    a1, b1, c1, s1 = oracle.solve(sp.problem, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt, opt, 1)
    a4, b4, c4, s4 = oracle.solve(sp.problem, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt, opt, 4)
    assert s1.num_iterations == s4.num_iterations
    np.testing.assert_allclose(s4.cost, s1.cost, rtol=1e-9)   # summation order differs
    assert rel_err(a4, a1, 1e-9) < 1e-8


def test_iteration_cap_and_trace_bookkeeping(oracle):
    """max_num_iterations = k records iterations 0..k (k+1 summaries), NO_CONVERGENCE."""
    sp = synth.config(2)
    opt = capi.default_options(max_num_iterations=3)
    _, _, _, s = oracle.solve(sp.problem, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt, opt)
    assert s.termination == "NO_CONVERGENCE" and s.num_iterations == 4
    assert s.num_successful_steps + s.num_unsuccessful_steps == 4
    assert s.step_flags[0] == 3 and s.cost[0] == s.initial_cost
    assert s.final_cost == s.cost.min()


def test_analytic_jacobian_matches_jets_on_extreme_geometry(oracle, hostmath):
    """The hand-derived Jacobian against Jet autodiff away from the comfortable configs:
    the 16-camera ring (incidence up to 110 degrees, boards near the image border), intrinsics
    pushed to the edge of the model's range, near-zero and near-pi rotations, and a board almost
    on the optical axis (r -> 0, where d(u, v)/dP loses its usual scale)."""
    rng = np.random.default_rng(314)
    sp = synth.config(4, num_frames=120)
    p = sp.problem
    worst = 0.0
    for trial in range(4):
        intr = sp.init_intrinsics.copy()
        cam_rt = sp.init_cam_rt.copy()
        board_rt = sp.init_board_rt.copy()
        if trial == 1:      # strong mirror terms
            intr[:, 4] = rng.uniform(-0.45, 0.3, len(intr))
            intr[:, 5] = rng.uniform(-0.25, 0.25, len(intr))
            intr[:, 6] = rng.uniform(0.35, 0.75, len(intr))
        if trial == 2:      # rotations at the Taylor branch and close to pi
            board_rt[::3, :3] = rng.normal(0, 1e-9, (len(board_rt[::3]), 3))
            ax = rng.normal(0, 1, (len(board_rt[1::3]), 3))
            board_rt[1::3, :3] = ax / np.linalg.norm(ax, axis=1, keepdims=True) * (np.pi - 1e-4)
        if trial == 3:      # far and very near boards
            board_rt[::2, 3:] *= 6.0
            board_rt[1::2, 3:] *= 0.3
        r0, J0, c0 = oracle.eval_jacobian(p, intr, cam_rt, board_rt)
        r, J, c = hostmath_eval(hostmath, p, intr, cam_rt, board_rt)
        ok = np.isfinite(J0).all(axis=(1, 2)) & np.isfinite(r0).all(axis=1)
        assert ok.mean() > 0.9                                  # (points behind the mirror give NaN in both)
        np.testing.assert_array_equal(np.isfinite(J).all(axis=(1, 2)), ok)
        scale = np.maximum(np.abs(J0[ok]).max(axis=2, keepdims=True), 1.0)   # per residual row
        err = float(np.max(np.abs(J[ok] - J0[ok]) / scale))
        worst = max(worst, err)
        assert err < 1e-10, (trial, err)
        np.testing.assert_allclose(r[ok], r0[ok], rtol=1e-12, atol=1e-9)
    # a board centred on the optical axis of camera 0, 400 mm away, facing it
    K = p.corners_per_board
    one = capi.ProblemArrays(p.board_xy - p.board_xy.mean(axis=0), np.zeros(1, np.int32), np.zeros(1, np.int32),
                             np.full((K, 2), 600.0), 1, 1, 0)
    intr1 = sp.gt_intrinsics[:1].copy()
    pose = np.array([[1e-3, -2e-3, 0.3, 0.0, 0.0, 400.0]])
    r0, J0, _ = oracle.eval_jacobian(one, intr1, np.zeros((1, 6)), pose)
    r, J, _ = hostmath_eval(hostmath, one, intr1, np.zeros((1, 6)), pose)
    scale = np.maximum(np.abs(J0).max(axis=2, keepdims=True), 1.0)
    assert np.max(np.abs(J - J0) / scale) < 1e-10


@pytest.mark.parametrize("case", ["cfg2", "ring", "cfg5-huber"])
def test_moment_formulation_equals_direct_gram(hostmath, case):
    """The per-view normal-equation blocks rebuilt from the 36 + 108 moment sums (what k_eval5 +
    k_view_blocks do, DESIGN.md §5) against the direct Gram of the Jacobian rows [J | r] of the
    same view: BB, BC, BI, CC, CI, II — 210 entries per view."""
    loss, scale = 0, 1.0
    if case == "cfg2":
        sp = synth.config(2, num_frames=40)
    elif case == "ring":
        sp = synth.config(4, num_frames=60)
    else:
        sp, loss = synth.config(5, num_frames=40), capi.LOSS["huber"]
    p = sp.problem
    a = np.ascontiguousarray(sp.init_intrinsics)
    b = np.ascontiguousarray(sp.init_cam_rt)
    c = np.ascontiguousarray(sp.init_board_rt)
    mom, direct = np.zeros((p.num_views, 210)), np.zeros((p.num_views, 210))
    rc = hostmath.hostmath_view_blocks(C.byref(p.c), _dp(a), _dp(b), _dp(c), loss, C.c_double(scale),
                                       _dp(mom), _dp(direct))
    assert rc == 0
    # entries of one block live on very different scales (rotation vs translation vs focal
    # columns): compare against the geometric mean of the two diagonal entries involved
    assert np.isfinite(direct).all() and np.isfinite(mom).all()
    blocks = [(0, 21), (21, 57), (57, 105), (105, 126), (126, 174), (174, 210)]   # BB BC BI CC CI II
    for lo, hi in blocks:
        ref = direct[:, lo:hi]
        scale_b = np.abs(ref).max(axis=1, keepdims=True) + 1e-300
        assert np.max(np.abs(mom[:, lo:hi] - ref) / scale_b) < 1e-11, (case, lo)
