"""Generates tests/golden/cv_shim.npz: outputs of the REAL OpenCV (cv2 wheel of this image) for
the three OpenCV calls the host adapters make through tscm_calib_b200/host/cv_compat.h when
OpenCV C++ is not available:

  cv::Rodrigues       both directions   (TS.cpp:70,94; multi_calib.h:16,43; main.cpp YAML)
  cv::solvePnPRansac  planar board, identity camera matrix, default arguments (TS.cpp:193)

Run from the repo root:  python tests/golden/make_golden_cvshim.py
"""
import os
import sys

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
OUT = os.path.dirname(os.path.abspath(__file__))


def main():
    rng = np.random.default_rng(2024)
    # Rodrigues: vectors incl. tiny and near-pi angles
    rv = np.concatenate([rng.normal(0, 1.0, (40, 3)), rng.normal(0, 1e-9, (4, 3)),
                         [np.array([np.pi - 1e-3, 0, 0]), np.array([0, 3.0, 0.5]), np.zeros(3)]])
    Rm = np.stack([cv2.Rodrigues(v.reshape(3, 1))[0] for v in rv])
    back = np.stack([cv2.Rodrigues(R)[0].reshape(3) for R in Rm])
    # planar PnP: 9x6 board, 45 mm, poses in front of the camera, pixel-ish noise on the normalised plane
    obj = np.array([[(j % 9) * 45.0, (j // 9) * 45.0, 0.0] for j in range(54)])
    poses, imgs, rvecs, tvecs, costs = [], [], [], [], []
    for n in range(24):
        r = rng.normal(0, 0.45, 3)
        t = np.array([rng.uniform(-300, 100), rng.uniform(-200, 100), rng.uniform(350, 900)])
        R = cv2.Rodrigues(r.reshape(3, 1))[0]
        P = obj @ R.T + t
        img = P[:, :2] / P[:, 2:3] + rng.normal(0, [0.0, 2e-4, 1e-3][n % 3], (54, 2))
        ok, rvec, tvec, inl = cv2.solvePnPRansac(obj.reshape(-1, 1, 3), img.reshape(-1, 1, 2), np.eye(3), None)
        assert ok and len(inl) == 54
        proj, _ = cv2.projectPoints(obj, rvec, tvec, np.eye(3), None)
        poses.append(np.concatenate([r, t]))
        imgs.append(img)
        rvecs.append(rvec.reshape(3))
        tvecs.append(tvec.reshape(3))
        costs.append(float(((proj.reshape(-1, 2) - img) ** 2).sum()))
    np.savez_compressed(os.path.join(OUT, "cv_shim.npz"), rodrigues_vec=rv, rodrigues_mat=Rm, rodrigues_back=back,
                        pnp_obj=obj, pnp_img=np.stack(imgs), pnp_true=np.stack(poses), pnp_rvec=np.stack(rvecs),
                        pnp_tvec=np.stack(tvecs), pnp_cost=np.array(costs))
    print("opencv", cv2.__version__, "pnp costs", np.array(costs).round(8)[:6])


def non_orthonormal():
    """cv_rodrigues_nonortho.npz: cv::Rodrigues of matrices that are not rotations, as the reference
    hands them over (r3 = r1 x r2 from float-truncated columns, chained pose-graph products)."""
    rng = np.random.default_rng(5)
    mats, backs = [], []
    for k in range(40):
        v = rng.normal(size=3) * rng.uniform(0.05, 2.5)
        R, _ = cv2.Rodrigues(v)
        if k % 2 == 0:
            M = R.astype(np.float32).astype(np.float64)            # float truncation, Rt_to_R_t style
            M[:, 2] = np.cross(M[:, 0], M[:, 1])
        else:
            M = R + rng.normal(scale=1e-4, size=(3, 3))            # accumulated error of chained products
        M = np.ascontiguousarray(M)
        mats.append(M)
        backs.append(cv2.Rodrigues(M)[0].reshape(3))
    np.savez_compressed(os.path.join(OUT, "cv_rodrigues_nonortho.npz"), mat=np.stack(mats), back=np.stack(backs))


if __name__ == "__main__":
    main()
    non_orthonormal()
