"""Rigs of 17 to 32 cameras (tscm_options.allow_large_rigs): the reduced system factored by a
thread-block cluster (k_solve_cluster), its covariance, and the limits of the opt-in.

- The cluster form against the single-CTA k_solve where both run (NL <= 202), through the test
  hook tscm_solver_set_reduced_solve.
- Reduced systems of 208 to 416 live parameters against the CPU oracle: dense forward arrays
  (frames with up to 32 views: k_post_eval's 32-lane form) and a sparse ring (pair Schur form).
- Convergence, determinism, covariance against the dense reference, and every refusal.

Every creation asserts its paths through the "[tscm create] paths: ..." line of debug flag 1."""
import dataclasses
import re

import numpy as np
import pytest

import covariance_reference as ref
from test_covariance_gpu import agreement_tol, assert_cov_close
from test_gpu_parity import assert_same_solve
from tscm_calib_b200 import capi, synth

pytestmark = pytest.mark.gpu

ERR_INVALID = 1              # TSCM_ERR_INVALID_ARGUMENT
ERR_UNSUPPORTED = 5          # TSCM_ERR_UNSUPPORTED
DEFAULT_NL = 202             # include/tscm.h: the default limit
LARGE_NL = 416               # ... and the limit with allow_large_rigs = 1
PATHS = re.compile(r"\[tscm create\] paths: (.*)")


@pytest.fixture(autouse=True)
def debug_paths():
    capi.set_debug(1)
    yield
    capi.set_debug(0)


def created_paths(capfd):
    """The paths line of the one solver created since the last call."""
    err = capfd.readouterr().err
    found = PATHS.findall(err)
    assert len(found) == 1, err
    return {k: v if k == "form" else int(v) for k, v in (kv.split("=") for kv in found[0].split())}


def assert_paths(got, **want):
    for k, v in want.items():
        assert got[k] == v, (k, got)


def opts(**kw):
    return capi.default_options(allow_large_rigs=1, **kw)


def with_fixed(sp, fixed_camera):
    if fixed_camera == 0:
        return sp
    p = sp.problem
    q = capi.ProblemArrays(p.board_xy, p.view_camera, p.view_frame, p.obs_xy, p.num_cameras, p.num_frames,
                           fixed_camera=fixed_camera)
    return dataclasses.replace(sp, problem=q)


def dense(num_cameras, num_frames, fixed_camera=0, **kw):
    sp = synth.generate(num_cameras=num_cameras, num_frames=num_frames, rig="array", dense=True,
                        seed=40 + num_cameras, **kw)
    assert sp.visible.all()
    return with_fixed(sp, fixed_camera)


def ring(num_cameras, num_frames, fixed_camera=0):
    return with_fixed(synth.generate(num_cameras=num_cameras, num_frames=num_frames, rig="ring",
                                     seed=70 + num_cameras), fixed_camera)


def lanes(problem):
    """k_post_eval's lanes per frame for this problem's most-viewed frame."""
    m = np.bincount(problem.view_frame).max()
    return 8 if m <= 8 else (16 if m <= 16 else 32)


def init_point(sp):
    return sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt


def run_solver(sp, form, iters):
    s = capi.Solver(sp.problem, opts(max_num_iterations=iters))
    try:
        s.set_reduced_solve(form)
        s.set_parameters(*init_point(sp))
        res = s.run()
        return s.get_parameters(), res
    finally:
        s.close()


# ---- 1. the cluster form against the single CTA --------------------------------------------------
AB = {
    "c8": (lambda: dense(8, 60), dict(NL=98, cluster=0, lpf=8)),
    "c10-fixed4": (lambda: dense(10, 60, fixed_camera=4), dict(NL=124, cluster=0, lpf=16)),
    "c16": (lambda: dense(16, 40), dict(NL=DEFAULT_NL, form="pairs", cluster=0, lpf=16)),
}


@pytest.mark.parametrize("case", list(AB))
def test_cluster_matches_single_cta(capfd, case):
    make, want = AB[case]
    sp = make()
    identical = []
    for iters in (1, 10):
        p1, r1 = run_solver(sp, "single", iters)
        assert_paths(created_paths(capfd), **want)
        p2, r2 = run_solver(sp, "cluster", iters)
        assert_paths(created_paths(capfd), **want)
        assert r1.num_iterations == r2.num_iterations and r1.termination == r2.termination
        np.testing.assert_array_equal(r1.step_flags, r2.step_flags)
        np.testing.assert_allclose(r2.cost, r1.cost, rtol=1e-12, atol=0)
        for a, b in zip(p1, p2):
            np.testing.assert_allclose(b, a, rtol=1e-9, atol=0)
        identical.append(all(np.array_equal(a, b) for a, b in zip(p1, p2)) and np.array_equal(r1.cost, r2.cost))
    print(case, "bit-identical (1 step, 10 iterations):", identical)


# ---- 2. reduced systems of 208 to 416 live parameters against the oracle -------------------------
def check_large(oracle, capfd, sp, want, iters=6):
    x = init_point(sp)
    want = dict(want, lpf=lanes(sp.problem))
    s = capi.Solver(sp.problem, opts())
    try:
        paths = created_paths(capfd)
        assert_paths(paths, **want)
        s.set_parameters(*x)
        idx = oracle.live_reduced_index(sp.problem)
        for radius in (1e4, 3.0):
            lhs, rhs = s.reduced_system(radius)
            lhs0, rhs0 = oracle.reduced_system(sp.problem, *x, radius)
            lhs0, rhs0 = lhs0[np.ix_(idx, idx)], rhs0[idx]
            sc = np.sqrt(np.abs(np.diag(lhs0)))
            assert np.max(np.abs(lhs - lhs0) / np.outer(sc, sc)) < 1e-10
            assert np.max(np.abs(rhs - rhs0)) / np.max(np.abs(rhs0)) < 1e-10
        per, overall, rms = s.reprojection_error()
        per0, overall0, rms0 = oracle.reprojection_error(sp.problem, *x)
        np.testing.assert_allclose(per, per0, rtol=0, atol=1e-9)
        assert abs(overall - overall0) < 1e-9 and abs(rms - rms0) < 1e-9
    finally:
        s.close()
    o = opts(max_num_iterations=iters)
    a, b, c, res = capi.solve_resident(sp.problem, *x, o)
    assert_paths(created_paths(capfd), **want)
    a0, b0, c0, res0 = oracle.solve(sp.problem, *x, capi.default_options(max_num_iterations=iters), num_threads=4)
    assert_same_solve(res, res0, (a, b, c), (a0, b0, c0))
    np.testing.assert_allclose(res.gradient_max_norm[0], res0.gradient_max_norm[0], rtol=1e-10)
    np.testing.assert_allclose(res.gradient_max_norm[1:], res0.gradient_max_norm[1:], rtol=1e-7)
    np.testing.assert_allclose(res.step_norm, res0.step_norm, rtol=1e-6, atol=1e-12)
    return paths


LARGE = {
    # the first system the default limit refuses
    "c16-free": (lambda: dense(16, 30, fixed_camera=-1), dict(NL=208, form="pairs", cluster=2)),
    "c17-fixed0": (lambda: dense(17, 30), dict(NL=215, form="pairs", cluster=2)),
    "c24-fixed11": (lambda: dense(24, 30, fixed_camera=11), dict(NL=306, form="pairs", cluster=3)),
    "c32-fixed31": (lambda: dense(32, 30, fixed_camera=31), dict(NL=410, form="pairs", cluster=4)),
    "c32-free": (lambda: dense(32, 30, fixed_camera=-1), dict(NL=LARGE_NL, form="pairs", cluster=4)),
    # sparse: ragged views per frame
    "ring24": (lambda: ring(24, 60), dict(NL=306, form="pairs", cluster=3)),
}


@pytest.mark.parametrize("case", list(LARGE))
def test_large_reduced_systems_match_the_oracle(oracle, capfd, case):
    make, want = LARGE[case]
    paths = check_large(oracle, capfd, make(), want)
    assert paths["solve_smem"] <= paths["smem_optin"]
    print(case, paths)


# ---- 3. convergence and determinism ---------------------------------------------------------------
def test_zero_noise_32_cameras_converge_and_repeat_bit_identically(capfd):
    sp = dense(32, 30, noise_px=0.0, perturb=0.1)
    x = init_point(sp)
    o = opts(max_num_iterations=200)
    a, b, c, res = capi.solve_resident(sp.problem, *x, o)
    assert_paths(created_paths(capfd), NL=410, cluster=4, lpf=32)
    assert res.final_cost < 1e-9 * res.initial_cost, res
    np.testing.assert_allclose(a[:, :7], sp.gt_intrinsics[:, :7], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(b, sp.gt_cam_rt, rtol=0, atol=1e-5)
    np.testing.assert_allclose(c, sp.gt_board_rt, rtol=0, atol=1e-5)
    a2, b2, c2, res2 = capi.solve_resident(sp.problem, *x, o)
    created_paths(capfd)
    for u, v in ((a, a2), (b, b2), (c, c2), (res.cost, res2.cost), (res.step_norm, res2.step_norm)):
        np.testing.assert_array_equal(u, v)
    print(res.termination, "iterations", res.num_iterations, "cost", res.initial_cost, "->", res.final_cost)


# ---- 4. covariance --------------------------------------------------------------------------------
@pytest.mark.parametrize("num_cameras,fixed,nl", [(17, 0, 215), (32, 31, 410)])
def test_large_covariance_matches_the_reference(oracle, capfd, num_cameras, fixed, nl):
    sp = dense(num_cameras, 30, fixed_camera=fixed)
    x = (sp.gt_intrinsics, sp.gt_cam_rt, sp.gt_board_rt)
    s = capi.Solver(sp.problem, opts())
    assert_paths(created_paths(capfd), NL=nl)
    s.set_parameters(*x)
    cov = s.covariance()
    s.close()
    rc, cam, brd, s2, H = ref.covariance(oracle, sp.problem, *x)
    assert rc == 0 and cov.camera.shape == (nl, nl)
    assert_cov_close(cov, cam, brd, s2, agreement_tol(H))
    print(nl, "kernel ms", cov.kernel_ms, "tol", agreement_tol(H))


def test_large_covariance_without_fixed_camera_is_rank_deficient(capfd):
    sp = dense(20, 20, fixed_camera=-1)
    x = (sp.gt_intrinsics, sp.gt_cam_rt, sp.gt_board_rt)
    s = capi.Solver(sp.problem, opts())
    assert_paths(created_paths(capfd), NL=260, cluster=2)
    s.set_parameters(*x)
    with pytest.raises(capi.TscmError) as e:
        s.covariance()
    s.close()
    assert e.value.code == capi.ERR_RANK_DEFICIENT, str(e.value)


# ---- 5. refusals ----------------------------------------------------------------------------------
def tiny_problem(num_cameras, fixed_camera):
    """One frame seen by every camera, 4 corners: enough for every check made before the device."""
    board = np.array([[0.0, 0.0], [1.0, 0.0], [0.0, 1.0], [1.0, 1.0]])
    cams = np.arange(num_cameras, dtype=np.int32)
    return capi.ProblemArrays(board, cams, np.zeros(num_cameras, np.int32), np.zeros((num_cameras, 4, 2)),
                              num_cameras, 1, fixed_camera=fixed_camera)


def test_33_cameras_are_refused_everywhere(capfd):
    p = tiny_problem(33, -1)
    x = (np.zeros((33, 9)), np.zeros((33, 6)), np.zeros((1, 6)))
    calls = {"Solver": lambda: capi.Solver(p, opts()),
             "solve": lambda: capi.solve(p, *x, opts()),
             "covariance": lambda: capi.covariance(p, *x, opts())}
    for name, call in calls.items():
        with pytest.raises(capi.TscmError) as e:
            call()
        msg = str(e.value)
        assert e.value.code == ERR_UNSUPPORTED and f"limit of {LARGE_NL}" in msg and "429 live" in msg, (name, msg)
    assert PATHS.search(capfd.readouterr().err) is None


def test_sharded_large_rig_is_refused_before_devices_matter(capfd):
    p = tiny_problem(16, -1)
    for call in (lambda: capi.Solver(p, opts(num_gpus=2)),
                 lambda: capi.solve(p, np.zeros((16, 9)), np.zeros((16, 6)), np.zeros((1, 6)), opts(num_gpus=2))):
        with pytest.raises(capi.TscmError) as e:
            call()
        assert e.value.code == ERR_UNSUPPORTED and "num_gpus" in str(e.value), str(e.value)
    assert PATHS.search(capfd.readouterr().err) is None


def test_forced_forms_that_cannot_hold_the_system_are_refused(capfd):
    sp = dense(24, 20)
    s = capi.Solver(sp.problem, opts())
    assert_paths(created_paths(capfd), NL=306, form="pairs", cluster=3)
    with pytest.raises(capi.TscmError) as e:
        s.set_reduced_solve("single")
    assert e.value.code == ERR_UNSUPPORTED and "single-CTA" in str(e.value)
    for form in ("rows", "fused"):
        with pytest.raises(capi.TscmError) as e:
            s.set_schur_form(form)
        assert e.value.code == ERR_UNSUPPORTED, str(e.value)
    with pytest.raises(capi.TscmError) as e:
        s.set_options(capi.default_options())
    assert e.value.code == ERR_INVALID and "allow_large_rigs" in str(e.value)
    # still usable on its own paths
    s.set_reduced_solve("auto")
    s.set_options(opts(max_num_iterations=3))
    s.set_parameters(*init_point(sp))
    res = s.run()
    assert res.num_iterations >= 1 and np.isfinite(res.final_cost)
    s.close()


def test_solver_cache_keys_on_the_opt_in(capfd):
    """tscm_solve at one structure with and without the opt-in: never the other's cached solver."""
    sp = dense(16, 20, fixed_camera=-1)                # NL 208
    x = init_point(sp)
    capi.solve(sp.problem, *x, opts(max_num_iterations=2))
    assert_paths(created_paths(capfd), NL=208, cluster=2)
    with pytest.raises(capi.TscmError) as e:
        capi.solve(sp.problem, *x, capi.default_options(max_num_iterations=2))
    assert e.value.code == ERR_UNSUPPORTED and f"limit of {DEFAULT_NL}" in str(e.value)
    sp8 = dense(8, 20)                                 # NL 98: both accepted, two solvers
    r_large = capi.solve(sp8.problem, *init_point(sp8), opts(max_num_iterations=3))
    assert_paths(created_paths(capfd), NL=98, cluster=0)
    r_default = capi.solve(sp8.problem, *init_point(sp8), capi.default_options(max_num_iterations=3))
    assert_paths(created_paths(capfd), NL=98, cluster=0)
    r_again = capi.solve(sp8.problem, *init_point(sp8), capi.default_options(max_num_iterations=3))
    assert PATHS.search(capfd.readouterr().err) is None          # cache hit
    for u, v, w in zip(r_large[:3], r_default[:3], r_again[:3]):
        np.testing.assert_array_equal(u, v)
        np.testing.assert_array_equal(v, w)
