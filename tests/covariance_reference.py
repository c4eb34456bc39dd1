"""Dense CPU restatement of the covariance definition of include/tscm.h (tscm_solver_covariance),
built on the oracle's autodiff Jacobian: H = J^T J over the live parameters [cameras: rt(6) unless
fixed, 7 intrinsics | 6 per frame], with the robust loss applied through Ceres' corrector, dense
Cholesky with the rank test of ceres::Covariance, and the plain-residual variance."""
import numpy as np

RANK_DEFICIENT = 7          # TSCM_ERR_RANK_DEFICIENT


def live_columns(problem):
    cols = []
    for m in range(problem.num_cameras):
        ks = range(6, 13) if m == problem.fixed_camera else range(13)
        cols += [(m, k) for k in ks]
    return cols


def live_jacobian(problem, J):
    """(2N x n) Jacobian over the live parameters from the oracle's N x 2 x 21 Jacobian
    (camera_rt 6, chessboard_rt 6, intrinsic 9)."""
    cols = live_columns(problem)
    NL = len(cols)
    K = problem.corners_per_board
    Jl = np.zeros((problem.num_observations * 2, NL + 6 * problem.num_frames))
    Jv = J.reshape(problem.num_views, K * 2, 21)
    for v in range(problem.num_views):
        m, f = problem.view_camera[v], problem.view_frame[v]
        rows = slice(v * K * 2, (v + 1) * K * 2)
        for i, (mm, k) in enumerate(cols):
            if mm == m:
                Jl[rows, i] = Jv[v, :, k if k < 6 else 12 + (k - 6)]
        Jl[rows, NL + 6 * f:NL + 6 * f + 6] = Jv[v, :, 6:12]
    return Jl, NL


def corrector_scale(r, loss_type, a):
    """sqrt(rho'(s)) per corner, s = |r|^2.  Huber and Cauchy have rho'' <= 0, for which Ceres'
    Corrector scales the Jacobian by sqrt(rho') alone (alpha = 0)."""
    s = np.sum(r * r, axis=-1)
    if loss_type == 0:
        return np.ones_like(s)
    if loss_type == 1:
        rho1 = np.where(s > a * a, a / np.sqrt(np.maximum(s, 1e-300)), 1.0)
    else:
        rho1 = 1.0 / (1.0 + s / (a * a))
    return np.sqrt(rho1)


def jtj(oracle, problem, intrinsics, cam_rt, board_rt, loss_type=0, loss_scale=1.0):
    r, J, _ = oracle.eval_jacobian(problem, intrinsics, cam_rt, board_rt)
    J = J * corrector_scale(r, loss_type, loss_scale)[:, None, None]
    Jl, NL = live_jacobian(problem, J)
    return Jl.T @ Jl, NL, r


def covariance(oracle, problem, intrinsics, cam_rt, board_rt, options=None):
    """(rc, camera NL x NL, board F x 6 x 6, residual variance, H)."""
    lt = int(options.loss_type) if options is not None else 0
    a = float(options.loss_scale) if options is not None else 1.0
    H, NL, r = jtj(oracle, problem, intrinsics, cam_rt, board_rt, lt, a)
    n = H.shape[0]
    # pivots of the LDL^T: squares of the Cholesky diagonal
    try:
        L = np.linalg.cholesky(H)
    except np.linalg.LinAlgError:
        return RANK_DEFICIENT, None, None, None, H
    if np.min(np.diag(L) ** 2) <= 1e-14 * np.max(np.diag(H)):
        return RANK_DEFICIENT, None, None, None, H
    X = np.linalg.inv(L)                      # Sigma = X^T X
    cam = X[:, :NL].T @ X[:, :NL]
    F = problem.num_frames
    brd = np.zeros((F, 6, 6))
    for f in range(F):
        Xf = X[:, NL + 6 * f:NL + 6 * f + 6]
        brd[f] = Xf.T @ Xf
    s2 = np.sum(r * r) / (2 * problem.num_observations - n)
    return 0, cam, brd, s2, H


def conditioning(H):
    """Condition number of the equilibrated H."""
    d = 1.0 / np.sqrt(np.diag(H))
    ev = np.linalg.eigvalsh(d[:, None] * H * d[None, :])
    return ev[-1] / max(ev[0], 1e-300)
