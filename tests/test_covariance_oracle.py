"""CPU suite of the covariance definition (include/tscm.h, tscm_solver_covariance): the dense
restatement of tests/covariance_reference.py, built on the oracle's autodiff Jacobian, against an
independent numpy inversion and against the inverse of the oracle's undamped reduced system.

Agreement bars: the synthetic rigs' J^T J has an equilibrated condition number kappa of 1e10-1e11
(the triple-sphere xi, lambda, alpha and the focal lengths are strongly correlated), so two correct
inversions agree to ~kappa * eps only, whatever the algorithm: max(1e-10, 4 kappa eps) on the
correlation-normalised blocks and on their diagonals."""
import numpy as np
import pytest

import covariance_reference as ref
from tscm_calib_b200 import capi, synth

EPS = np.finfo(np.float64).eps


def normalised(S):
    d = np.sqrt(np.abs(np.diagonal(S, axis1=-2, axis2=-1)))
    return S / (d[..., :, None] * d[..., None, :])


def tol_of(H):
    return max(1e-10, 4.0 * ref.conditioning(H) * EPS)


@pytest.mark.parametrize("idx", [1, 2])
def test_dense_covariance_is_inverse_of_jtj(oracle, idx):
    sp = synth.config(idx)
    p = sp.problem
    args = (p, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    rc, cam, brd, s2, H = ref.covariance(oracle, *args)
    assert rc == 0
    NL = cam.shape[0]
    # equilibrated LU inverse (numpy), independent of the Cholesky route
    d = 1.0 / np.sqrt(np.diag(H))
    Sigma = d[:, None] * np.linalg.inv(d[:, None] * H * d[None, :]) * d[None, :]
    tol = tol_of(H)
    np.testing.assert_allclose(normalised(cam), normalised(Sigma[:NL, :NL]), rtol=0, atol=tol)
    np.testing.assert_allclose(np.diag(cam), np.diag(Sigma)[:NL], rtol=tol)
    for f in range(p.num_frames):
        blk = Sigma[NL + 6 * f:NL + 6 * f + 6, NL + 6 * f:NL + 6 * f + 6]
        np.testing.assert_allclose(normalised(brd[f]), normalised(blk), rtol=0, atol=tol)
        np.testing.assert_allclose(np.diag(brd[f]), np.diag(blk), rtol=tol)
    r, _, _ = oracle.eval_jacobian(*args)
    assert s2 == pytest.approx(np.sum(r * r) / (2 * p.num_observations - H.shape[0]), rel=1e-12)


@pytest.mark.parametrize("loss", ["none", "huber", "cauchy"])
def test_camera_block_is_inverse_of_undamped_reduced_system(oracle, loss):
    """Sigma_cc = D_c S~^-1 D_c with S~ the oracle's Jacobi-scaled reduced system at radius -> inf
    (its loss-corrected Jacobian: this also pins the corrector restatement)."""
    sp = synth.config(2 if loss == "none" else 5)
    p = sp.problem
    opt = capi.default_options(loss_type=loss, loss_scale=1.0)
    args = (p, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)
    rc, cam, _, _, H = ref.covariance(oracle, *args, options=opt)
    assert rc == 0
    live = oracle.live_reduced_index(p)
    S = oracle.reduced_system(*args, radius=1e300, options=opt)[0][np.ix_(live, live)]
    opt0 = capi.default_options(loss_type=loss, loss_scale=1.0, jacobi_scaling=0)
    S0 = oracle.reduced_system(*args, radius=1e300, options=opt0)[0][np.ix_(live, live)]
    D = np.sqrt(np.diag(S) / np.diag(S0))      # S~ = D_c S D_c
    Sigma = D[:, None] * np.linalg.inv(S) * D[None, :]
    tol = tol_of(H)
    np.testing.assert_allclose(normalised(cam), normalised(Sigma), rtol=0, atol=tol)
    np.testing.assert_allclose(np.diag(cam), np.diag(Sigma), rtol=tol)


def test_gauge_freedom_is_rank_deficient(oracle):
    sp = synth.config(2)
    p = sp.problem
    q = capi.ProblemArrays(p.board_xy, p.view_camera, p.view_frame, p.obs_xy, p.num_cameras,
                           p.num_frames, fixed_camera=-1)
    rc = ref.covariance(oracle, q, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt)[0]
    assert rc == capi.ERR_RANK_DEFICIENT
    # the GPU tests S~ (not H): its LDL^T pivots along the gauge stay far below the threshold
    live = oracle.live_reduced_index(q)
    S = oracle.reduced_system(q, sp.init_intrinsics, sp.init_cam_rt, sp.init_board_rt, radius=1e300)[0]
    A = S[np.ix_(live, live)].copy()
    piv = []
    for j in range(A.shape[0]):
        piv.append(A[j, j])
        A[j + 1:, j + 1:] -= np.outer(A[j + 1:, j], A[j + 1:, j]) / A[j, j]
    rel = np.sort(np.array(piv) / np.max(np.diag(S)))
    assert np.all(rel[:6] <= 1e-14) and rel[6] > 1e-12


def test_camera_std_dev_layout():
    sp = synth.config(2)
    p = sp.problem
    n = len(capi.live_columns(p))
    assert capi.live_columns(p) == ref.live_columns(p)
    cov = np.diag(np.arange(1, n + 1, dtype=np.float64))
    sd = capi.camera_std_dev(p, cov, 4.0)
    assert sd.shape == (4, 15)
    assert np.all(sd[0, :6] == 0) and np.all(sd[:, 13:] == 0)
    np.testing.assert_allclose(sd[0, 6:13], 2 * np.sqrt(np.arange(1, 8)))
    np.testing.assert_allclose(sd[1, :13], 2 * np.sqrt(np.arange(8, 21)))
