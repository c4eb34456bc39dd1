"""GPU parity tests (run on the B200 box): every call goes through the C-ABI of
libtscm_b200.so and is compared with the CPU oracle / the committed golden vectors.
North-star tolerances: Jacobian 1e-10, per-iteration cost 1e-9 relative, final
parameters 1e-7 relative, RMS reprojection error 1e-9 px."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_options, load_golden, rel_err
from tscm_calib_b200 import capi, synth

pytestmark = pytest.mark.gpu

COST_RTOL, PARAM_RTOL, RMS_ATOL, JAC_TOL = 1e-9, 1e-7, 1e-9, 1e-10


def assert_same_solve(res, ref, params, ref_params, cost_rtol=COST_RTOL):
    assert res.termination == ref.termination
    assert res.num_iterations == ref.num_iterations
    assert res.num_successful_steps == ref.num_successful_steps
    np.testing.assert_allclose(res.cost, ref.cost, rtol=cost_rtol)
    np.testing.assert_array_equal(res.step_flags, ref.step_flags)
    np.testing.assert_allclose(res.radius, ref.radius, rtol=1e-6)
    for x, x0 in zip(params, ref_params):
        assert rel_err(x, x0, 1e-9) < PARAM_RTOL


@pytest.mark.parametrize("cfg", [1, 2])
def test_residuals_and_jacobian_match_oracle(oracle, cfg):
    sp = synth.config(cfg)
    s = capi.Solver(sp.problem)
    s.set_parameters(sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    r, J, cost = s.eval_jacobian()
    r0, J0, c0 = oracle.eval_jacobian(sp.problem, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    np.testing.assert_allclose(r, r0, rtol=0, atol=JAC_TOL)
    assert np.max(np.abs(J - J0) / np.maximum(np.abs(J0), 1.0)) < JAC_TOL
    assert abs(cost - c0) < 1e-12 * c0
    s.close()


@pytest.mark.parametrize("golden", ["jacobian_mpmath", "jacobian_sympy"])
def test_jacobian_matches_mpmath_golden(golden):
    """k_eval_rows against 50-digit central differences and against sympy's symbolic derivative
    of the reference functor (tests/golden/make_golden_sympy.py)."""
    z = np.load(os.path.join(GOLDEN, golden + ".npz"))
    for k in range(len(z["r"])):
        p = capi.ProblemArrays(z["board"][k][None, :], [0], [0], z["obs"][k][None, None, :], 1, 1,
                               fixed_camera=-1)
        s = capi.Solver(p)
        s.set_parameters(z["intr"][k][None], z["cam_rt"][k][None], z["board_rt"][k][None])
        r, J, _ = s.eval_jacobian()
        np.testing.assert_allclose(r[0], z["r"][k], rtol=0, atol=JAC_TOL)
        assert np.max(np.abs(J[0] - z["J"][k]) / np.maximum(np.abs(z["J"][k]), 1.0)) < JAC_TOL
        s.close()


@pytest.mark.parametrize("cfg", [1, 2])
def test_reduced_camera_system_matches_oracle(oracle, cfg):
    sp = synth.config(cfg)
    s = capi.Solver(sp.problem)
    s.set_parameters(sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    for radius in (1e4, 3.0):
        lhs, rhs = s.reduced_system(radius)
        lhs0, rhs0 = oracle.reduced_system(sp.problem, sp.init_intrinsics, sp.init_cam_rt,
                                           sp.init_board_rt, radius)
        idx = oracle.live_reduced_index(sp.problem)
        dead = np.setdiff1d(np.arange(lhs0.shape[0]), idx)
        # dropped b, c rows couple to nothing: the oracle's rows hold only the LM diagonal
        off = lhs0[np.ix_(dead, idx)]
        assert np.all(off == 0) and np.all(rhs0[dead] == 0)
        lhs0, rhs0 = lhs0[np.ix_(idx, idx)], rhs0[idx]
        sc = np.sqrt(np.abs(np.diag(lhs0)))
        assert np.max(np.abs(lhs - lhs0) / np.outer(sc, sc)) < 1e-10
        assert np.max(np.abs(rhs - rhs0)) / np.max(np.abs(rhs0)) < 1e-10
        np.testing.assert_array_equal(lhs, lhs.T)
    s.close()


@pytest.mark.parametrize("name", ["mono_cfg1", "rig3_small", "rig4_huber", "rig4_cauchy"])
def test_solve_matches_golden_vectors(name):
    p, z = load_golden(name)
    opt = golden_options(z)
    a, b, c, s = capi.solve(p, z["init_intrinsics"], z["init_cam_rt"], z["init_board_rt"], opt)
    assert s.termination == str(z["termination"])
    assert s.num_iterations == len(z["cost"])
    np.testing.assert_allclose(s.cost, z["cost"], rtol=COST_RTOL)
    np.testing.assert_array_equal(s.step_flags, z["flags"])
    assert rel_err(a, z["final_intrinsics"], 1e-9) < PARAM_RTOL
    assert rel_err(b, z["final_cam_rt"], 1e-9) < PARAM_RTOL
    assert rel_err(c, z["final_board_rt"], 1e-9) < PARAM_RTOL


@pytest.mark.parametrize("cfg,iters", [(1, 100), (2, 50)])
def test_solve_matches_oracle(oracle, cfg, iters):
    sp = synth.config(cfg)
    opt = capi.default_options(max_num_iterations=iters)
    init = (sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    a, b, c, s = capi.solve(sp.problem, *init, opt)
    a0, b0, c0, s0 = oracle.solve(sp.problem, *init, opt)
    assert_same_solve(s, s0, (a, b, c), (a0, b0, c0))
    _, e, rms = oracle.reprojection_error(sp.problem, a, b, c)
    _, e0, rms0 = oracle.reprojection_error(sp.problem, a0, b0, c0)
    assert abs(rms - rms0) < RMS_ATOL and abs(e - e0) < RMS_ATOL
    # camera 0's extrinsic is the constant block: untouched, bit for bit
    np.testing.assert_array_equal(b[0], sp.init_cam_rt[0])
    # b, c intrinsics are carried through unchanged
    np.testing.assert_array_equal(a[:, 7:], sp.init_intrinsics[:, 7:])


@pytest.mark.parametrize("loss", ["huber", "cauchy"])
def test_robust_loss_config5_matches_oracle(oracle, loss):
    sp = synth.config(5)
    opt = capi.default_options(loss_type=loss, loss_scale=1.0)
    init = (sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    a, b, c, s = capi.solve(sp.problem, *init, opt)
    a0, b0, c0, s0 = oracle.solve(sp.problem, *init, opt)
    assert_same_solve(s, s0, (a, b, c), (a0, b0, c0))


def test_fixed_iteration_mode_and_iteration_cap(oracle):
    sp = synth.config(2)
    init = (sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    for opt in (capi.default_options(max_num_iterations=3),
                capi.default_options(max_num_iterations=12, disable_tolerances=1)):
        a, b, c, s = capi.solve(sp.problem, *init, opt)
        a0, b0, c0, s0 = oracle.solve(sp.problem, *init, opt)
        assert s.termination == "NO_CONVERGENCE" and s.num_iterations == opt.max_num_iterations + 1
        assert_same_solve(s, s0, (a, b, c), (a0, b0, c0))


def test_resident_solver_reruns_and_readout(oracle):
    sp = synth.config(2)
    s = capi.Solver(sp.problem, capi.default_options())
    init = (sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    s.set_parameters(*init)
    r1 = s.run()
    p1 = s.get_parameters()
    per, overall, rms = s.reprojection_error()
    per0, overall0, rms0 = oracle.reprojection_error(sp.problem, *p1)
    np.testing.assert_allclose(per, per0, rtol=0, atol=1e-9)
    assert abs(overall - overall0) < 1e-9 and abs(rms - rms0) < 1e-9
    # same initial point again -> identical trajectory (deterministic reductions)
    s.set_parameters(*init)
    r2 = s.run()
    np.testing.assert_array_equal(r1.cost, r2.cost)
    for x, y in zip(p1, s.get_parameters()):
        np.testing.assert_array_equal(x, y)
    # warm start from the solution: converges immediately
    r3 = s.run()
    assert r3.termination == "CONVERGENCE" and r3.num_iterations <= 2
    assert s.launch_count() > 0
    s.close()


def test_ragged_visibility_single_view_frames_and_tiny_board(oracle):
    """Frames seen by one camera only, cameras with few views, K = 35 (not a multiple of
    32), a 42-iteration trajectory.  (A 5x3 board makes lambda so weakly determined that two
    independent CPU restatements already differ by 5e-7 in it; 7x5 is well-posed.)"""
    sp = synth.generate(num_cameras=4, num_frames=60, board=(7, 5), rig="calib", seed=71)
    assert sp.visible.sum(axis=0).min() == 1
    opt = capi.default_options()
    init = (sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    a, b, c, s = capi.solve(sp.problem, *init, opt)
    a0, b0, c0, s0 = oracle.solve(sp.problem, *init, opt)
    assert_same_solve(s, s0, (a, b, c), (a0, b0, c0))


def test_taylor_branch_zero_rotation_board(oracle):
    """A board pose with an exactly-zero angle-axis (theta^2 <= eps branch) that is free."""
    sp = synth.generate(num_cameras=2, num_frames=10, board=(6, 5), rig="calib", seed=72)
    init_b = sp.init_board_rt.copy()
    s = capi.Solver(sp.problem)
    init_b[3, :3] = 0.0
    s.set_parameters(sp.init_intrinsics, sp.init_cam_rt, init_b)
    r, J, _ = s.eval_jacobian()
    r0, J0, _ = oracle.eval_jacobian(sp.problem, sp.init_intrinsics, sp.init_cam_rt, init_b)
    np.testing.assert_allclose(r, r0, rtol=0, atol=1e-9)
    assert np.max(np.abs(J - J0) / np.maximum(np.abs(J0), 1.0)) < JAC_TOL
    s.close()


def test_zero_noise_recovers_ground_truth():
    sp = synth.generate(num_cameras=3, num_frames=40, board=(11, 8), rig="calib", seed=31,
                        noise_px=0.0)
    opt = capi.default_options(max_num_iterations=100, function_tolerance=1e-14,
                               parameter_tolerance=1e-14)
    s = capi.Solver(sp.problem, opt)
    s.set_parameters(sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    res = s.run()
    assert res.final_cost < 1e-12 * res.initial_cost
    assert s.reprojection_error()[2] < 1e-6
    _, cam_rt, _ = s.get_parameters()
    assert rel_err(cam_rt[1:], sp.gt_cam_rt[1:], 1e-3) < 1e-4
    s.close()


def test_full_size_config3_properties():
    """BASELINE config 3 (8 cameras x 5000 frames x 88 corners = 3.52 M observations):
    size-independent properties — cost decreases monotonically over accepted steps,
    the optimum has RMS ~ sigma*sqrt(2), identical reruns are bit-identical."""
    sp = synth.config(3)
    assert sp.num_observations == 3_520_000
    s = capi.Solver(sp.problem, capi.default_options())
    init = (sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    s.set_parameters(*init)
    r1 = s.run()
    assert r1.termination == "CONVERGENCE"
    ok = r1.step_flags == 3
    assert np.all(np.diff(r1.cost[ok]) < 0)
    per, overall, rms = s.reprojection_error()
    assert abs(rms - 0.1 * np.sqrt(2)) < 2e-3
    assert abs(rms - np.sqrt(2 * r1.final_cost / sp.num_observations)) < 1e-9
    s.set_parameters(*init)
    r2 = s.run()
    np.testing.assert_array_equal(r1.cost, r2.cost)
    s.close()


def test_config3_sample_of_frames_matches_oracle(oracle):
    """The oracle finishes 8 cameras x 300 frames in seconds: same dense geometry as config 3."""
    sp = synth.config(3, num_frames=300)
    opt = capi.default_options()
    init = (sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    a, b, c, s = capi.solve(sp.problem, *init, opt)
    a0, b0, c0, s0 = oracle.solve(sp.problem, *init, opt, num_threads=4)
    assert_same_solve(s, s0, (a, b, c), (a0, b0, c0))


def test_sixteen_camera_ring_uses_wide_schur_path(oracle):
    """Config 4 geometry at reduced frame count: 16 cameras (202 live reduced parameters,
    the 1024-thread Schur instantiation), partial visibility."""
    sp = synth.config(4, num_frames=400)
    opt = capi.default_options(max_num_iterations=15)
    init = (sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    a, b, c, s = capi.solve(sp.problem, *init, opt)
    a0, b0, c0, s0 = oracle.solve(sp.problem, *init, opt, num_threads=4)
    assert_same_solve(s, s0, (a, b, c), (a0, b0, c0))


@pytest.mark.parametrize("case", ["cfg2", "ragged", "ring16"])
def test_pair_schur_reduced_system_matches_oracle(oracle, case):
    """S and rhs from k_pair_frames / k_pair_blocks (per-view blocks) -> k_schur_pairs2 ->
    k_reduce_pairs (csrc/tscm_schur_pairs.cuh), forced on problems that would otherwise take the
    dense-row kernels (tscm_solver_set_schur_form)."""
    sp = {"cfg2": lambda: synth.config(2),
          "ragged": lambda: synth.generate(num_cameras=4, num_frames=60, board=(7, 5), rig="calib", seed=71),
          "ring16": lambda: synth.config(4, num_frames=700)}[case]()   # > 128 common frames per pair: several items
    s = capi.Solver(sp.problem, schur_form="pairs")
    s.set_parameters(sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    for radius in (1e4, 3.0):
        lhs, rhs = s.reduced_system(radius)
        lhs0, rhs0 = oracle.reduced_system(sp.problem, sp.init_intrinsics, sp.init_cam_rt,
                                           sp.init_board_rt, radius)
        idx = oracle.live_reduced_index(sp.problem)
        lhs0, rhs0 = lhs0[np.ix_(idx, idx)], rhs0[idx]
        sc = np.sqrt(np.abs(np.diag(lhs0)))
        assert np.max(np.abs(lhs - lhs0) / np.outer(sc, sc)) < 1e-10
        assert np.max(np.abs(rhs - rhs0)) / np.max(np.abs(rhs0)) < 1e-10
        np.testing.assert_array_equal(lhs, lhs.T)
    s.close()


@pytest.mark.parametrize("form", ["pairs", "fused", "rows"])
@pytest.mark.parametrize("case", ["cfg2", "cfg5-huber", "ragged"])
def test_every_schur_form_solves_like_the_oracle(oracle, case, form):
    if case == "cfg2":
        sp, opt = synth.config(2), capi.default_options()
    elif case == "cfg5-huber":
        sp, opt = synth.config(5), capi.default_options(loss_type=capi.LOSS["huber"], loss_scale=1.0)
    else:
        sp = synth.generate(num_cameras=4, num_frames=60, board=(7, 5), rig="calib", seed=71)
        opt = capi.default_options()
    init = (sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    a, b, c, s = capi.solve_resident(sp.problem, *init, opt, schur_form=form)
    a0, b0, c0, s0 = oracle.solve(sp.problem, *init, opt)
    assert_same_solve(s, s0, (a, b, c), (a0, b0, c0))


def test_pair_schur_is_deterministic_and_agrees_with_dense_rows():
    """Same problem through the dense-row kernels and through the pair kernels: iteration
    counts equal, costs to round-off; the pair path twice: bit-identical."""
    sp = synth.config(3, num_frames=400)
    opt = capi.default_options(max_num_iterations=12)
    init = (sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    a0, b0, c0, s0 = capi.solve_resident(sp.problem, *init, opt, schur_form="rows")
    a1, b1, c1, s1 = capi.solve_resident(sp.problem, *init, opt, schur_form="pairs")
    a2, b2, c2, s2 = capi.solve_resident(sp.problem, *init, opt, schur_form="pairs")
    np.testing.assert_array_equal(s1.cost, s2.cost)
    for x, y in ((a1, a2), (b1, b2), (c1, c2)):
        np.testing.assert_array_equal(x, y)
    assert s0.num_iterations == s1.num_iterations
    np.testing.assert_allclose(s1.cost, s0.cost, rtol=1e-10)
    for x, y in ((a1, a0), (b1, b0), (c1, c0)):
        np.testing.assert_allclose(x, y, rtol=1e-7, atol=1e-9)


def test_errors_are_reported_not_swallowed():
    sp = synth.config(1)
    s = capi.Solver(sp.problem)
    bad = capi.default_options(loss_type=7)
    with pytest.raises(capi.TscmError):
        s.set_options(bad)
    with pytest.raises(capi.TscmError):
        s.reduced_system(-1.0)
    s.close()
