"""NumPy reference of orcvio_trajectory_nees (TEST INFRASTRUCTURE, not product code): the NEES of the IMU state of a
filter run against its truth, per run and frame, and the per-frame ANEES summary.

The error definitions follow the filter's own retraction, incrementState_IMUCam (oracle/filter.py): orientation
R = Exp(dtheta) R_est under use_larvio / left perturbation, R = R_est Exp(dtheta) otherwise; v, p and the biases additive.
tests/test_consistency_cpu.py checks this module against known answers, that retraction and the chi-square
distribution; tests/test_gpu_consistency.py checks the device kernels against it.
"""
import numpy as np

_PERM15 = np.array([0, 1, 2, 6, 7, 8, 3, 4, 5, 9, 10, 11, 12, 13, 14])   # [theta, v, p, bg, ba] -> [theta, p, v, bg, ba]


def so3_log(R):
    """Log of a rotation matrix: angle atan2(|w|, (tr - 1) / 2) with w = vee(R - R^T) / 2; near pi the axis comes from
    the symmetric part, R + R^T = 2 cos I + 2 (1 - cos) n n^T, with the sign of w."""
    w = 0.5 * np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]])
    c = 0.5 * (np.trace(R) - 1.0)
    s = float(np.linalg.norm(w))
    th = np.arctan2(s, c)
    if c > -0.9:
        return (th / s if s > 0.0 else 1.0) * w
    B = (0.5 * (R + R.T) - c * np.eye(3)) / (1.0 - c)
    k = int(np.argmax(np.diag(B)))
    n = B[k] / np.linalg.norm(B[k])
    return (-1.0 if n @ w < 0.0 else 1.0) * th * n


def error_state(est17, gt17, left):
    """15-vector [dtheta, dv, dp, dbg, dba] of the truth against the estimate under incrementState_IMUCam's retraction
    (oracle/filter.py): R = Exp(dtheta) R_est if `left` (use_larvio || use_left_perturbation), else R = R_est Exp(dtheta);
    the rest additive (true - est)."""
    Re = _q2R(est17[4:8])
    Rg = _q2R(gt17[4:8])
    dth = so3_log(Rg @ Re.T if left else Re.T @ Rg)
    return np.concatenate([dth, gt17[8:11] - est17[8:11], gt17[1:4] - est17[1:4], gt17[11:14] - est17[11:14],
                           gt17[14:17] - est17[14:17]])


def _q2R(q):
    """quaternionToRotation (x y z w, unit), math_utils.hpp:164-177."""
    x, y, z, w = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def nees_row(est17, gt17, P15, left):
    """One row of orcvio_trajectory_nees: NEES theta, v, p, pose [theta, p], nav [theta, p, v], full, |dtheta| deg,
    |dp| m; NaN where an input is not finite or the block is not positive definite.  Only the lower triangle of the
    permuted block is read (as the kernel's factorisation does)."""
    nan = np.full(8, np.nan)
    if not (np.all(np.isfinite(est17)) and np.all(np.isfinite(gt17)) and np.all(np.isfinite(P15))):
        return nan
    e = error_state(np.asarray(est17, float), np.asarray(gt17, float), left)
    A = np.asarray(P15, float).reshape(15, 15)[np.ix_(_PERM15, _PERM15)]
    A = np.tril(A) + np.tril(A, -1).T
    ep = e[_PERM15]
    try:
        L = np.linalg.cholesky(A)
    except np.linalg.LinAlgError:
        return nan
    if not np.all(np.diag(L) > 0):
        return nan
    y = np.linalg.solve(L, ep)
    cs = np.cumsum(y * y)

    def block(b0):
        B = A[b0:b0 + 3, b0:b0 + 3]
        return float(ep[b0:b0 + 3] @ np.linalg.solve(B, ep[b0:b0 + 3]))
    return np.array([cs[2], block(6), block(3), cs[5], cs[8], cs[14],
                     np.degrees(np.linalg.norm(e[0:3])), np.linalg.norm(e[6:9])])


def nees(est17, gt17, cov15, flags):
    """(n, F, 17), (n, F, 17), (n, F, 15, 15) -> (nees (n, F, 8), summary (F, 9)): what orcvio_trajectory_nees returns.
    flags: bit0 use_larvio, bit1 use_left_perturbation."""
    est17 = np.asarray(est17, float)
    gt17 = np.asarray(gt17, float)
    n, F = est17.shape[:2]
    cov = np.asarray(cov15, float).reshape(n, F, 15, 15)
    left = (int(flags) & 3) != 0
    out = np.zeros((n, F, 8))
    for i in range(n):
        for f in range(F):
            out[i, f] = nees_row(est17[i, f], gt17[i, f], cov[i, f], left)
    return out, nees_summary(out)


def nees_summary(rows):
    """Per frame over the trajectories with a finite full-state NEES: ANEES of the six blocks, RMS |dtheta| (deg), RMS
    |dp| (m), number of those trajectories (NaN statistics when there is none)."""
    rows = np.asarray(rows, float)
    F = rows.shape[1]
    out = np.zeros((F, 9))
    for f in range(F):
        r = rows[:, f]
        r = r[np.isfinite(r[:, 5])]
        if len(r) == 0:
            out[f, :8] = np.nan
            continue
        out[f, :6] = r[:, :6].mean(axis=0)
        out[f, 6] = np.sqrt(np.mean(r[:, 6] ** 2))
        out[f, 7] = np.sqrt(np.mean(r[:, 7] ** 2))
        out[f, 8] = len(r)
    return out
