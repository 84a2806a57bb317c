"""Test-side reference for mpl_triangulate_robust: exhaustive-pair RANSAC with the MSAC cost, then a confidence-weighted
DLT refit over the inliers, in numpy float64 with one SVD per solve.  The reference has no robust triangulation; this
restates the library's own definition (include/mpl_b200.h).  The product path never imports it."""
from __future__ import annotations

import itertools

import numpy as np


def projections(R, t, f, c):
    """P_v = K_v [R_v | -R_v t_v], [V, 3, 4] float64."""
    V = len(R)
    P = np.zeros((V, 3, 4))
    for v in range(V):
        Rv, tv = np.asarray(R[v], dtype=np.float64), np.asarray(t[v], dtype=np.float64)
        K = np.array([[f[v][0], 0.0, c[v][0]], [0.0, f[v][1], c[v][1]], [0.0, 0.0, 1.0]], dtype=np.float64)
        P[v] = K @ np.concatenate([Rv, -(Rv @ tv)[:, None]], axis=1)
    return P


def _err2(P, X, u, w):
    """Squared pixel reprojection errors of homogeneous X through P [n, 3, 4] at pixels (u, w) [n]; inf where the depth
    (P3 . X) / X_4 is not > 0 or not finite."""
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        z = P[:, 2] @ X
        depth = z / X[3]
        e2 = (P[:, 0] @ X / z - u) ** 2 + (P[:, 1] @ X / z - w) ** 2
    return np.where((depth > 0) & np.isfinite(depth), e2, np.inf)


def triangulate_robust(pix, R, t, f, c, image_size, min_conf=0.0, inlier_px=10.0):
    """Per (pose, joint): candidates are the views with conf > min_conf and 0 < u < w-1, 0 < v < h-1.  Every candidate pair
    (a < b, lexicographic) gives the SVD solution of its two views' unweighted rows u P3 - P1, v P3 - P2; its MSAC cost is
    sum_c min(e_c^2, tau^2) over all candidates; the lowest cost wins (ties: the earlier pair).  Inliers: e_c < tau; with at
    least two, the point is the SVD solution of the inliers' rows each multiplied by its conf.

    Returns (points [B,J,3] NaN where undetermined, inliers [B,J] int32 bitmask, near_decision [B,J] bool).  near_decision
    flags items whose outcome float rounding can flip: a candidate of the winning hypothesis with |e_c - tau| < 1e-6 tau,
    or the two lowest pair costs within 1e-9 of each other relative to the larger.
    """
    pix = np.asarray(pix)
    w, h = image_size
    B, V, J, _ = pix.shape
    P = projections(R, t, f, c)
    tau = float(np.float32(inlier_px))
    tau2 = tau * tau
    u = pix[..., 0].astype(np.float64)
    vv = pix[..., 1].astype(np.float64)
    conf = pix[..., 2].astype(np.float64)
    cand = (pix[..., 2] > np.float32(min_conf)) & (0 < u) & (u < w - 1) & (0 < vv) & (vv < h - 1)   # [B,V,J]
    points = np.full((B, J, 3), np.nan)
    inliers = np.zeros((B, J), dtype=np.int32)
    near = np.zeros((B, J), dtype=bool)
    for b in range(B):
        for j in range(J):
            vs = np.flatnonzero(cand[b, :, j])
            if len(vs) < 2:
                continue
            rows = {v: np.stack([u[b, v, j] * P[v, 2] - P[v, 0], vv[b, v, j] * P[v, 2] - P[v, 1]]) for v in vs}
            pairs = list(itertools.combinations(vs, 2))
            Xs = np.linalg.svd(np.stack([np.concatenate([rows[a], rows[a2]]) for a, a2 in pairs]))[2][:, -1]   # [n,4]
            e2s = [_err2(P[vs], X, u[b, vs, j], vv[b, vs, j]) for X in Xs]
            costs = np.array([float(sum(min(e, tau2) for e in e2)) for e2 in e2s])
            k = int(np.argmin(costs))                      # first minimum: an exact tie keeps the earlier pair
            e2 = e2s[k]
            srt = np.sort(costs)
            near[b, j] = bool(np.any(np.abs(np.sqrt(e2) - tau) < 1e-6 * tau)) or (
                len(srt) > 1 and srt[1] - srt[0] <= 1e-9 * srt[1])
            inl = vs[e2 < tau2]
            if len(inl) < 2:
                continue
            X = np.linalg.svd(np.concatenate([conf[b, v, j] * rows[v] for v in inl]))[2][-1]
            points[b, j] = X[:3] / X[3]
            inliers[b, j] = int(sum(1 << int(v) for v in inl))
    return points, inliers, near
