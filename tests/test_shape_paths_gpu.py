"""The kernel paths that create_shard picks from the shape of the problem, each against the CPU
oracle: the dense-row Schur update with one and two 4x4 tiles per thread, both k_solve
instantiations, k_post_eval with 16 lanes per frame, the tail split of k_eval5 (2 and 4 parts,
partial last corner group, fewer than four groups), a fixed camera other than 0, no fixed camera,
and the largest and the first rejected reduced system.

Every case asserts the paths it claims through the line that create_shard prints with debug flag 1
("[tscm create] paths: ..."), so a misrouted case fails instead of passing on another branch.
Shapes that depend on the device are built from its SM count and opt-in shared memory."""
import dataclasses
import re

import numpy as np
import pytest

import covariance_reference as ref
from conftest import rel_err
from test_covariance_gpu import agreement_tol, assert_cov_close
from test_gpu_parity import assert_same_solve
from tscm_calib_b200 import capi, synth

pytestmark = pytest.mark.gpu

ERR_UNSUPPORTED = 5          # TSCM_ERR_UNSUPPORTED
MAX_NL = 202                 # include/tscm.h: the largest reduced system a solver accepts
PATHS = re.compile(r"\[tscm create\] paths: (.*)")


@pytest.fixture(scope="module")
def device():
    import torch
    p = torch.cuda.get_device_properties(0)
    return {"sms": p.multi_processor_count, "smem_optin": p.shared_memory_per_block_optin}


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


def dense(num_cameras, num_frames, board=(11, 8), fixed_camera=0, **kw):
    sp = synth.generate(num_cameras=num_cameras, num_frames=num_frames, board=board, rig="array", dense=True,
                        seed=40 + num_cameras, **kw)
    assert sp.visible.all()
    if fixed_camera != 0:
        p = sp.problem
        q = capi.ProblemArrays(p.board_xy, p.view_camera, p.view_frame, p.obs_xy, p.num_cameras, p.num_frames,
                               fixed_camera=fixed_camera)
        sp = dataclasses.replace(sp, problem=q)
    return sp


def init_point(sp):
    return sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt


def assert_point_matches(oracle, s, sp, x):
    """Reduced camera system (k_eval5 -> k_view_blocks -> k_post_eval -> Schur) at two radii and
    the reprojection error (k_eval5's error read-out) at x."""
    idx = oracle.live_reduced_index(sp.problem)
    for radius in (1e4, 3.0):
        lhs, rhs = s.reduced_system(radius)
        lhs0, rhs0 = oracle.reduced_system(sp.problem, *x, radius)
        lhs0, rhs0 = lhs0[np.ix_(idx, idx)], rhs0[idx]
        sc = np.sqrt(np.abs(np.diag(lhs0)))
        assert np.max(np.abs(lhs - lhs0) / np.outer(sc, sc)) < 1e-10
        assert np.max(np.abs(rhs - rhs0)) / np.max(np.abs(rhs0)) < 1e-10
        np.testing.assert_array_equal(lhs, lhs.T)
    per, overall, rms = s.reprojection_error()
    per0, overall0, rms0 = oracle.reprojection_error(sp.problem, *x)
    np.testing.assert_allclose(per, per0, rtol=0, atol=1e-9)
    assert abs(overall - overall0) < 1e-9 and abs(rms - rms0) < 1e-9


def assert_trace_matches(s, s0, params, params0):
    """assert_same_solve, plus the two trace quantities behind gradient_tolerance and
    parameter_tolerance: the gradient max-norm (frame part from k_post_eval) and the step norm
    (from k_backsub's partials)."""
    assert_same_solve(s, s0, params, params0)
    np.testing.assert_allclose(s.gradient_max_norm[0], s0.gradient_max_norm[0], rtol=1e-10)
    np.testing.assert_allclose(s.gradient_max_norm[1:], s0.gradient_max_norm[1:], rtol=1e-7)
    np.testing.assert_allclose(s.step_norm, s0.step_norm, rtol=1e-6, atol=1e-12)


def check_case(oracle, capfd, sp, want, iters=10):
    """Point comparison through a resident solver, then a short solve; both creations must take
    the paths `want`."""
    x = init_point(sp)
    s = capi.Solver(sp.problem)
    try:
        paths = created_paths(capfd)
        assert_paths(paths, **want)
        s.set_parameters(*x)
        assert_point_matches(oracle, s, sp, x)
    finally:
        s.close()
    opt = capi.default_options(max_num_iterations=iters)
    a, b, c, res = capi.solve_resident(sp.problem, *x, opt)
    assert_paths(created_paths(capfd), **want)
    a0, b0, c0, res0 = oracle.solve(sp.problem, *x, opt, num_threads=4)
    assert_trace_matches(res, res0, (a, b, c), (a0, b0, c0))
    return paths


# ---- reduced systems of 111 to 202 live parameters -------------------------------------------
WIDE = {
    # 9 cameras: dense rows, one tile per thread, k_solve<1,4>, 16 lanes per frame
    "c9": (lambda: dense(9, 100), dict(NL=111, form="rows", ept=1, solveT=1, lpf=16)),
    # a 7-column camera in the middle of the live table, k_solve<4,7>
    "c10-fixed4": (lambda: dense(10, 100, fixed_camera=4), dict(NL=124, form="rows", ept=1, solveT=4, lpf=16)),
    # the two shapes of k_schur_update<2>: the fixed camera last, and no fixed camera (NL 143,
    # about 10 KB under the shared memory of the dense-row form)
    "c11-fixed10": (lambda: dense(11, 100, fixed_camera=10), dict(NL=137, form="rows", ept=2, solveT=4, lpf=16)),
    "c11-free": (lambda: dense(11, 100, fixed_camera=-1), dict(NL=143, form="rows", ept=2, solveT=4, lpf=16)),
    # the first width past the dense-row form
    "c12": (lambda: dense(12, 100), dict(NL=150, form="pairs", solveT=4, lpf=16)),
    # the largest accepted system; exactly 16 views per frame
    "c16": (lambda: dense(16, 60), dict(NL=MAX_NL, form="pairs", solveT=4, lpf=16)),
}


@pytest.mark.parametrize("case", list(WIDE))
def test_wide_reduced_systems_match_the_oracle(oracle, capfd, device, case):
    make, want = WIDE[case]
    sp = make()
    paths = check_case(oracle, capfd, sp, want)
    assert paths["smem_optin"] == device["smem_optin"] and paths["solve_smem"] <= paths["smem_optin"]
    print(case, paths)


def test_dense_rows_are_refused_past_their_shared_memory(capfd):
    """12 cameras: the dense-row form does not fit; forcing it reports, and the solver stays usable."""
    sp = dense(12, 40)
    s = capi.Solver(sp.problem)
    assert_paths(created_paths(capfd), form="pairs")
    with pytest.raises(capi.TscmError) as e:
        s.set_schur_form("rows")
    assert e.value.code == ERR_UNSUPPORTED and "dense-row" in str(e.value)
    s.set_parameters(*init_point(sp))
    res = s.run()
    assert res.num_iterations > 1 and np.isfinite(res.final_cost)
    s.close()


def test_largest_system_covariance_matches_the_reference(oracle, capfd):
    """Covariance at NL = 202, the largest system k_cov_factor / k_cov_inverse / k_cov_frames
    accept, at the ground truth (the perturbed start is conditioned 1e14)."""
    sp = dense(16, 30)
    x = (sp.gt_intrinsics, sp.gt_cam_rt, sp.gt_board_rt)
    s = capi.Solver(sp.problem)
    paths = created_paths(capfd)
    assert_paths(paths, NL=MAX_NL, form="pairs", solveT=4, lpf=16)
    s.set_parameters(*x)
    cov = s.covariance()
    s.close()
    rc, cam, brd, s2, H = ref.covariance(oracle, sp.problem, *x)
    assert rc == 0 and cov.camera.shape == (MAX_NL, MAX_NL)
    assert_cov_close(cov, cam, brd, s2, agreement_tol(H))
    print(paths, "tol", agreement_tol(H))


def test_first_rejected_system_is_refused_everywhere(capfd, device):
    """16 cameras with no fixed camera (NL 208): TSCM_ERR_UNSUPPORTED from the resident solver, the
    one-shot solve and the one-shot covariance, naming the limit; nothing runs."""
    sp = dense(16, 20, fixed_camera=-1)
    x = init_point(sp)
    calls = {"Solver": lambda: capi.Solver(sp.problem),
             "solve": lambda: capi.solve(sp.problem, *x),
             "covariance": lambda: capi.covariance(sp.problem, *x)}
    msgs = []
    for name, call in calls.items():
        with pytest.raises(capi.TscmError) as e:
            call()
        msg = str(e.value)
        assert e.value.code == ERR_UNSUPPORTED, (name, msg)
        assert f"limit of {MAX_NL}" in msg and "208 live parameters" in msg, (name, msg)
        need = int(re.search(r"needs (\d+) bytes", msg).group(1))
        assert need > device["smem_optin"] and f"allows {device['smem_optin']}" in msg, (name, msg)
        msgs.append(f"{name}: {msg}")
    assert PATHS.search(capfd.readouterr().err) is None
    print("\n".join(msgs))


# ---- the tail split of k_eval5 -----------------------------------------------------------------
def split_cases(sms):
    """(problem, expected paths) per regime; tiles = ceil(V / 32), V = cameras x frames."""
    S = sms
    # 9 cameras: V not a multiple of 32, ceil(9 F / 32) = S + 2
    F9 = 32 * (S + 2) // 9
    if 9 * F9 % 32 == 0:
        F9 -= 1
    assert (9 * F9 + 31) // 32 == S + 2 and 9 * F9 % 32
    return {
        "split4": (lambda: dense(8, 4 * (S + 2)), dict(e5tiles=S + 2, e5whole=S, e5split=4)),
        "split2": (lambda: dense(8, 4 * (S + 50)), dict(e5tiles=S + 50, e5whole=S, e5split=2)),
        "split1-tail": (lambda: dense(8, 4 * (S + 130)), dict(e5tiles=S + 130, e5whole=S, e5split=1)),
        "two-rounds-tail": (lambda: dense(8, 4 * (2 * S + 20)), dict(e5tiles=2 * S + 20, e5whole=2 * S, e5split=4)),
        "c9-partial-tile": (lambda: dense(9, F9), dict(e5tiles=S + 2, e5whole=S, e5split=4, lpf=16)),
        # 35 corners: five groups of 8 (the last one partial) in parts of 1/1/1/2 groups
        "k35": (lambda: dense(8, 4 * (S + 2), board=(7, 5)), dict(e5tiles=S + 2, e5whole=S, e5split=4)),
        # 24 corners: three groups, so the split stops at 2
        "k24": (lambda: dense(8, 4 * (S + 2), board=(6, 4)), dict(e5tiles=S + 2, e5whole=S, e5split=2)),
    }


SPLITS = ["split4", "split2", "split1-tail", "two-rounds-tail", "c9-partial-tile", "k35", "k24"]


@pytest.mark.parametrize("case", SPLITS)
def test_eval5_tail_split_matches_the_oracle(oracle, capfd, device, case):
    make, want = split_cases(device["sms"])[case]
    paths = check_case(oracle, capfd, make(), dict(e5grid=device["sms"], **want), iters=6)
    assert paths["e5tiles"] > paths["e5whole"]
    print(case, paths)


# ---- the frame part of the gradient max-norm ---------------------------------------------------
def gradient_blocks(oracle, problem, x):
    """Plain gradient J^T r per frame (F x 6) and per camera (C x 15, rt | intrinsics; the fixed
    camera's rt is constant and left out) from the oracle's Jacobian."""
    V, K = problem.num_views, problem.corners_per_board
    r, J, _ = oracle.eval_jacobian(problem, *x)
    gv = np.einsum("vkj,vk->vj", J.reshape(V, 2 * K, 21), r.reshape(V, 2 * K))
    g_frame = np.zeros((problem.num_frames, 6))
    np.add.at(g_frame, problem.view_frame, gv[:, 6:12])
    g_cam = np.zeros((problem.num_cameras, 15))
    np.add.at(g_cam, problem.view_camera, np.concatenate([gv[:, :6], gv[:, 12:]], axis=1))
    if problem.fixed_camera >= 0:
        g_cam[problem.fixed_camera, :6] = 0.0
    return g_frame, g_cam


@pytest.mark.parametrize("slot", ["cta-first", "cta-last", "last-frame"])
def test_frame_gradient_max_norm_matches_the_oracle(oracle, capfd, slot):
    """Zero-noise 9-camera rig at its ground truth (gradient ~1e-8 everywhere) with ONE board pose
    turned by 1e-3 rad: that frame's gradient block sets the max-norm, so gradient_max_norm[0] is
    k_post_eval's 16-lane sum over that frame's views.  The frame sits in the first or the last
    slot of a k_post_eval block (512 / 16 = 32 frames each) or is the last frame of the problem."""
    fpc, F = 512 // 16, 101
    f = {"cta-first": fpc, "cta-last": 2 * fpc - 1, "last-frame": F - 1}[slot]
    sp = dense(9, F, noise_px=0.0, perturb=0.0)
    board_rt = sp.gt_board_rt.copy()
    board_rt[f, :3] += 1e-3
    x = (sp.gt_intrinsics, sp.gt_cam_rt, board_rt)
    g_frame, g_cam = gradient_blocks(oracle, sp.problem, x)
    top = np.abs(g_frame[f]).max()
    rest = max(np.abs(np.delete(g_frame, f, axis=0)).max(), np.abs(g_cam).max())
    assert top > 1.5 * rest, (top, rest)         # otherwise the case would not test k_post_eval
    opt = capi.default_options(max_num_iterations=1)
    a, b, c, res = capi.solve_resident(sp.problem, *x, opt)
    paths = created_paths(capfd)
    assert_paths(paths, lpf=16)
    a0, b0, c0, res0 = oracle.solve(sp.problem, *x, opt)
    assert rel_err(res0.gradient_max_norm[0], top) < 1e-9
    np.testing.assert_allclose(res.gradient_max_norm[0], res0.gradient_max_norm[0], rtol=1e-10)
    print(slot, f, paths, "frame block", top, "rest", rest)
