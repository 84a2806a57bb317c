"""Numpy restatement of mpl_calibrate_rig (include/mpl_b200.h): bundle adjustment of a rig's extrinsics and the 3D joints
by Levenberg-Marquardt with a Gaussian prior on the given calibration.  The normal equations are formed and solved densely
(the device eliminates the points by a Schur complement; in exact arithmetic the step is the same), so the problem must be
small.  `residuals` / `jacobian` give the weighted residual vector whose squared norm is the cost, for a comparison with
scipy.optimize.least_squares.
"""
from __future__ import annotations

import numpy as np
from scipy.spatial.transform import Rotation


def left_jacobian(w):
    w = np.asarray(w, dtype=np.float64)
    t2 = float(w @ w)
    if t2 < 1e-2:
        b = 0.5 * (1.0 - t2 / 12.0 * (1.0 - t2 / 30.0 * (1.0 - t2 / 56.0 * (1.0 - t2 / 90.0))))
        c = (1.0 - t2 / 20.0 * (1.0 - t2 / 42.0 * (1.0 - t2 / 72.0 * (1.0 - t2 / 110.0)))) / 6.0
    else:
        t = np.sqrt(t2)
        b, c = (1.0 - np.cos(t)) / t2, (t - np.sin(t)) / (t2 * t)
    K = skew(w)
    return np.eye(3) + b * K + c * K @ K


def skew(w):
    return np.array([[0.0, -w[2], w[1]], [w[2], 0.0, -w[0]], [-w[1], w[0], 0.0]])


def select_items(pix, calib, init, view_mask=None, min_conf=0.0):
    """used [B, J] bitmask of the used views of every item, 0 for pairs that are not items."""
    pix = np.asarray(pix, dtype=np.float32)
    B, V, J, _ = pix.shape
    u, v, conf = (pix[..., k].astype(np.float64) for k in range(3))
    w, h = calib[:, 16][None, :, None], calib[:, 17][None, :, None]
    cand = (pix[..., 2] > np.float32(min_conf)) & (0.0 < u) & (u < w - 1.0) & (0.0 < v) & (v < h - 1.0)   # [B, V, J]
    bits = (cand.astype(np.int64) << np.arange(V)[None, :, None]).sum(1)
    if view_mask is not None:
        bits &= np.asarray(view_mask, dtype=np.int64)
    X = np.asarray(init, dtype=np.float32).astype(np.float64)
    used = np.zeros((B, J), dtype=np.int64)
    for b in range(B):
        for j in range(J):
            m = int(bits[b, j])
            if not np.isfinite(X[b, j]).all() or bin(m).count("1") < 2:
                continue
            ok = True
            for vv in range(V):
                if (m >> vv) & 1:
                    R, c = calib[vv, :9].reshape(3, 3), calib[vv, 9:12]
                    z = (R @ (X[b, j] - c))[2]
                    ok &= bool(z > 0.0 and np.isfinite(z))
            if ok:
                used[b, j] = m
    return used


class Problem:
    def __init__(self, pix, calib, init, used, sigma_px, sigma_rot, sigma_pos):
        self.pix = np.asarray(pix, dtype=np.float32).astype(np.float64)
        self.calib = np.asarray(calib, dtype=np.float64)
        self.V = self.calib.shape[0]
        self.items = [(b, j) for b, j in zip(*np.nonzero(used))]
        self.used = used
        self.obs = [(i, v) for i, (b, j) in enumerate(self.items) for v in range(self.V) if (used[b, j] >> v) & 1]
        self.X0 = np.asarray(init, dtype=np.float32).astype(np.float64)[tuple(np.array(self.items).T)] if self.items else \
            np.zeros((0, 3))
        self.s_px, self.s_rot, self.s_pos = sigma_px, sigma_rot, sigma_pos
        self.R0 = self.calib[:, :9].reshape(-1, 3, 3)
        self.c0 = self.calib[:, 9:12]
        self.np = 6 * self.V + 3 * len(self.items)

    def start(self):
        return np.concatenate([np.concatenate([np.zeros((self.V, 3)), self.c0], 1).ravel(), self.X0.ravel()])

    def unpack(self, x):
        cam = x[:6 * self.V].reshape(self.V, 6)
        return cam[:, :3], cam[:, 3:], x[6 * self.V:].reshape(-1, 3)

    def rotations(self, om):
        return [Rotation.from_rotvec(om[v]).as_matrix() @ self.R0[v] for v in range(self.V)]

    def residuals(self, x):
        om, c, X = self.unpack(x)
        R = self.rotations(om)
        r = np.empty(2 * len(self.obs) + 6 * self.V)
        for k, (i, v) in enumerate(self.obs):
            b, j = self.items[i]
            fx, fy, cx, cy = self.calib[v, 12:16]
            y = R[v] @ (X[i] - c[v])
            if not (y[2] > 0.0 and np.isfinite(y[2])):
                r[:] = np.inf
                return r
            s = self.pix[b, v, j, 2] / self.s_px
            r[2 * k] = s * (fx * y[0] / y[2] + cx - self.pix[b, v, j, 0])
            r[2 * k + 1] = s * (fy * y[1] / y[2] + cy - self.pix[b, v, j, 1])
        n = 2 * len(self.obs)
        r[n:] = np.concatenate([om / self.s_rot, (c - self.c0) / self.s_pos], 1).ravel()
        return r

    def jacobian(self, x):
        om, c, X = self.unpack(x)
        R = self.rotations(om)
        Jl = [left_jacobian(om[v]) for v in range(self.V)]
        Jm = np.zeros((2 * len(self.obs) + 6 * self.V, self.np))
        for k, (i, v) in enumerate(self.obs):
            b, j = self.items[i]
            fx, fy = self.calib[v, 12:14]
            y = R[v] @ (X[i] - c[v])
            P = np.array([[fx / y[2], 0.0, -fx * y[0] / y[2] ** 2], [0.0, fy / y[2], -fy * y[1] / y[2] ** 2]])
            s = self.pix[b, v, j, 2] / self.s_px
            Jm[2 * k:2 * k + 2, 6 * v:6 * v + 3] = s * (P @ (-skew(y) @ Jl[v]))
            Jm[2 * k:2 * k + 2, 6 * v + 3:6 * v + 6] = s * (P @ -R[v])
            Jm[2 * k:2 * k + 2, 6 * self.V + 3 * i:6 * self.V + 3 * i + 3] = s * (P @ R[v])
        n = 2 * len(self.obs)
        for v in range(self.V):
            Jm[n + 6 * v:n + 6 * v + 3, 6 * v:6 * v + 3] = np.eye(3) / self.s_rot
            Jm[n + 6 * v + 3:n + 6 * v + 6, 6 * v + 3:6 * v + 6] = np.eye(3) / self.s_pos
        return Jm

    def cost(self, x):
        r = self.residuals(x)
        return float(r @ r)

    def data_cost(self, x):
        r = self.residuals(x)[:2 * len(self.obs)]
        return float(r @ r)

    def calib_out(self, x):
        om, c, _ = self.unpack(x)
        out = self.calib.copy()
        for v in range(self.V):
            if np.any(om[v] != 0.0):
                out[v, :9] = self.rotations(om)[v].ravel()
            out[v, 9:12] = c[v]
        return out


def calibrate_rig(pix, calib, init, view_mask=None, sigma_px=1.0, sigma_rot=np.radians(1.0), sigma_pos=0.05, min_conf=0.0,
                  max_iters=30):
    """(calib_out [V, 18], points [B, J, 3] fp32, report [8]) by the LM of the header."""
    calib = np.asarray(calib, dtype=np.float64)
    used = select_items(pix, calib, init, view_mask, min_conf)
    pb = Problem(pix, calib, init, used, sigma_px, sigma_rot, sigma_pos)
    points = np.array(init, dtype=np.float32, copy=True)
    if not pb.items:
        return calib.copy(), points, np.zeros(8)
    x = pb.start()
    C = C0 = pb.cost(x)
    wsum = sum(pb.pix[pb.items[i][0], v, pb.items[i][1], 2] ** 2 for i, v in pb.obs)
    rms0 = np.sqrt(pb.data_cost(x) * sigma_px ** 2 / wsum)
    mu, iters, accepted = None, 0, 0
    n = 6 * pb.V
    for k in range(1, max_iters + 1):
        iters = k
        Jm, r = pb.jacobian(x), pb.residuals(x)
        A, g = Jm.T @ Jm, Jm.T @ r
        if mu is None:
            mu = 1e-3 * float(np.max(np.diag(A)))
        try:
            L = np.linalg.cholesky(A + mu * np.eye(pb.np))
        except np.linalg.LinAlgError:
            mu *= 10.0
            continue
        d = -np.linalg.solve(L.T, np.linalg.solve(L, g))
        cnorm = float(np.linalg.norm(pb.unpack(x)[1]))
        Cn = pb.cost(x + d)
        if Cn < C:
            x, C, mu, accepted = x + d, Cn, mu / 10.0, accepted + 1
        else:
            mu *= 10.0
        if np.linalg.norm(d[:n]) <= 1e-10 * (cnorm + 1e-10):
            break
    Xf = pb.unpack(x)[2]
    for i, (b, j) in enumerate(pb.items):
        points[b, j] = Xf[i].astype(np.float32)
    report = np.array([len(pb.items), len(pb.obs), C0, C, rms0, np.sqrt(pb.data_cost(x) * sigma_px ** 2 / wsum), iters,
                       accepted], dtype=np.float64)
    return pb.calib_out(x), points, report
