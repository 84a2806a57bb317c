"""numpy oracle of mpl_undistort_pixels (include/mpl_b200.h), written from the header's statement rather than from the kernel.

Per entry with conf != 0 whose raw pixel lies strictly inside the image: Newton's method on D(x) = x_d from x = x_d, at most
MAX_ITERS steps x -= J^-1 (D(x) - x_d) by Cramer's rule, stopping after a step with |dx| + |dy| not > STEP_TOL; success iff
the final residual |D(x) - x_d|_1 <= RESID_TOL and x passes the validity rule.  Each entry stops on its own, as a thread does.
Everything is elementwise: the coefficients k = (k1, k2, p1, p2, k3) may be scalars or arrays broadcasting against x.
"""
import numpy as np

MAX_ITERS = 20
STEP_TOL = 1e-14
RESID_TOL = 1e-12


def distort(k, x, y):
    """D(x, y) and the Jacobian entries (a, b, d) of J = [[a, b], [b, d]] of OpenCV's model."""
    k1, k2, p1, p2, k3 = k
    r2 = x * x + y * y
    rho = 1.0 + r2 * (k1 + r2 * (k2 + r2 * k3))
    drho = k1 + r2 * (2.0 * k2 + r2 * (3.0 * k3))
    xd = x * rho + 2.0 * p1 * x * y + p2 * (r2 + 2.0 * x * x)
    yd = y * rho + p1 * (r2 + 2.0 * y * y) + 2.0 * p2 * x * y
    a = rho + 2.0 * x * x * drho + 2.0 * p1 * y + 6.0 * p2 * x
    b = 2.0 * x * y * drho + 2.0 * p1 * x + 2.0 * p2 * y
    d = rho + 2.0 * y * y * drho + 6.0 * p1 * y + 2.0 * p2 * x
    return xd, yd, a, b, d


def valid(k, x, y):
    """det J > 0 and g(s) = 1 + 3 k1 s + 5 k2 s^2 + 7 k3 s^3 > 0 on [0, r^2]: at r^2 and at the roots of
    g'(s) = 3 k1 + 10 k2 s + 21 k3 s^2 strictly inside (0, r^2)."""
    k1, k2, _, _, k3 = k
    _, _, a, b, d = distort(k, x, y)
    r2 = x * x + y * y

    def g(s):
        return 1.0 + s * (3.0 * k1 + s * (5.0 * k2 + s * (7.0 * k3)))

    with np.errstate(all="ignore"):
        ok = (a * d - b * b > 0.0) & (g(r2) > 0.0) & np.isfinite(r2)
        disc = 100.0 * k2 * k2 - 252.0 * k1 * k3
        root = np.sqrt(np.maximum(disc, 0.0))
        crit = [np.where(k3 != 0.0, np.where(disc >= 0.0, (-10.0 * k2 - root) / (42.0 * k3), np.nan),
                         np.where(k2 != 0.0, -3.0 * k1 / (10.0 * k2), np.nan)),
                np.where((k3 != 0.0) & (disc >= 0.0), (-10.0 * k2 + root) / (42.0 * k3), np.nan)]
        for s in crit:
            ok = ok & (~((s > 0.0) & (s < r2)) | (g(s) > 0.0))
    return ok


def undistort_normalised(k, xd, yd):
    """(x, y, ok) for distorted normalised points: the Newton inversion of the header, elementwise."""
    xd, yd = np.asarray(xd, dtype=np.float64), np.asarray(yd, dtype=np.float64)
    x, y = xd.copy(), yd.copy()
    active = np.ones(x.shape, dtype=bool)
    with np.errstate(all="ignore"):
        for _ in range(MAX_ITERS):
            if not active.any():
                break
            px, py, a, b, d = distort(k, x, y)
            det = a * d - b * b
            rx, ry = px - xd, py - yd
            dx, dy = (d * rx - b * ry) / det, (a * ry - b * rx) / det
            x = np.where(active, x - dx, x)
            y = np.where(active, y - dy, y)
            active = active & (np.abs(dx) + np.abs(dy) > STEP_TOL)
        px, py, _, _, _ = distort(k, x, y)
        ok = (np.abs(px - xd) + np.abs(py - yd) <= RESID_TOL) & valid(k, x, y)
    return x, y, ok


def undistort_pixels(pix, calib, dist, margin_x=0.0, margin_y=0.0):
    """mpl_undistort_pixels in numpy: pix [B, V, J, 3], calib [V, 18] or [B, V, 18], dist [V, 5] or [B, V, 5].  Returns
    (float32 result [B, V, J, 3], float64 [B, V, J, 2] (u', v') before rounding)."""
    pix = np.asarray(pix, dtype=np.float32)
    calib = np.asarray(calib, dtype=np.float64)
    dist = np.asarray(dist, dtype=np.float64)
    c = (calib if calib.ndim == 3 else calib[None])[:, :, None, :]              # [B or 1, V, 1, 18]
    kk = (dist if dist.ndim == 3 else dist[None])[:, :, None, :]
    k = tuple(kk[..., m] for m in range(5))
    fx, fy, cx, cy, w, h = (c[..., m] for m in range(12, 18))
    u, v, conf = (pix[..., m].astype(np.float64) for m in range(3))
    live = conf != 0
    inside = (0.0 < u) & (u < w - 1.0) & (0.0 < v) & (v < h - 1.0)
    xd, yd = (u - cx) / fx, (v - cy) / fy
    x, y, ok = undistort_normalised(k, xd, yd)
    work = live & inside
    good, bad = work & ok, work & ~ok
    with np.errstate(all="ignore"):
        uu = np.where(good, u + fx * (x - xd) + margin_x, np.where(bad, np.nan, u))
        vv = np.where(good, v + fy * (y - yd) + margin_y, np.where(bad, np.nan, v))
    out = pix.copy()
    out[..., 0], out[..., 1] = uu.astype(np.float32), vv.astype(np.float32)
    out[..., 2] = np.where(live & ~good, np.float32(0.0), pix[..., 2])
    return out, np.stack([uu, vv], axis=-1)
