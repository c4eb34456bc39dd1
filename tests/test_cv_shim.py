"""tscm_calib_b200/host/cv_compat.h (the OpenCV subset the C++ adapters use when OpenCV C++ is
absent) against the REAL OpenCV: golden vectors from the cv2 wheel, tests/golden/make_golden_cvshim.py."""
import ctypes as C
import os

import numpy as np

from conftest import ROOT

G = np.load(os.path.join(ROOT, "tests", "golden", "cv_shim.npz"))
dp = C.POINTER(C.c_double)


def _d(a):
    return a.ctypes.data_as(dp)


def test_rodrigues_matches_opencv_both_ways(hostinit):
    for v, R0, back0 in zip(G["rodrigues_vec"], G["rodrigues_mat"], G["rodrigues_back"]):
        R = np.zeros((3, 3))
        hostinit.hostinit_rodrigues(_d(np.ascontiguousarray(v)), 0, _d(R))
        np.testing.assert_allclose(R, R0, atol=1e-14)
        r = np.zeros(3)
        hostinit.hostinit_rodrigues(_d(np.ascontiguousarray(R0)), 1, _d(r))
        # near pi the axis sign is a convention; compare the rotations the vectors stand for
        R2 = np.zeros((3, 3))
        hostinit.hostinit_rodrigues(_d(r), 0, _d(R2))
        np.testing.assert_allclose(R2, R0, atol=1e-12)
        if np.linalg.norm(back0) < 3.0:
            # (OpenCV flushes rotations below ~1e-8 rad to exactly zero; the shim keeps them)
            np.testing.assert_allclose(r, back0, atol=1e-10 if np.linalg.norm(v) > 1e-6 else 1e-8)


def test_planar_pnp_matches_opencv_solvepnpransac(hostinit):
    """Same minimiser as cv2.solvePnPRansac (defaults) on noisy planar boards: never a higher
    reprojection cost, and the same pose to OpenCV's LM stopping tolerance."""
    obj = np.ascontiguousarray(G["pnp_obj"])
    worse = 0
    for img, rv0, tv0, c0 in zip(G["pnp_img"], G["pnp_rvec"], G["pnp_tvec"], G["pnp_cost"]):
        img = np.ascontiguousarray(img)
        r, t = np.zeros(3), np.zeros(3)
        assert hostinit.hostinit_solve_pnp(_d(obj), _d(img), len(obj), _d(r), _d(t)) == 0
        R = np.zeros((3, 3))
        hostinit.hostinit_rodrigues(_d(r), 0, _d(R))
        P = obj @ R.T + t
        cost = float((((P[:, :2] / P[:, 2:3]) - img) ** 2).sum())
        assert cost <= c0 * (1 + 1e-6) + 1e-18, (cost, c0)
        R0 = np.zeros((3, 3))
        hostinit.hostinit_rodrigues(_d(np.ascontiguousarray(rv0)), 0, _d(R0))
        np.testing.assert_allclose(R, R0, atol=5e-6)
        np.testing.assert_allclose(t, tv0, rtol=5e-6, atol=5e-4)
        worse += cost > c0
    assert worse == 0


def test_rodrigues_of_non_orthonormal_matrices_matches_opencv(hostinit):
    """The reference hands cv::Rodrigues matrices that are not rotations (r3 = r1 x r2 from
    float-truncated columns, chained pose-graph products: multi_calib.h:42-57, multi_calib.cpp:6-153).
    OpenCV projects them onto SO(3) (SVD, U V^T) first; so does the shim (ADVICE r01).  Checked
    against cv2.Rodrigues of the same matrices (golden vectors, make_golden_cvshim.py)."""
    z = np.load(os.path.join(ROOT, "tests", "golden", "cv_rodrigues_nonortho.npz"))
    assert len(z["mat"]) == 40
    for M, r0 in zip(z["mat"], z["back"]):
        r = np.zeros(3)
        hostinit.hostinit_rodrigues(_d(np.ascontiguousarray(M)), 1, _d(r))
        np.testing.assert_allclose(r, r0, atol=1e-12)
