"""Test-side reference for mpl_triangulate: the linear triangulation of MPL/lib/multiviews/triangulate.py:59-115 (pymvg's
find3d, called once per joint), restated in numpy float64 with one SVD per joint.  The product path never imports it."""
from __future__ import annotations

import numpy as np


def triangulate(pix, R, t, f, c, image_size, min_conf=0.0):
    """Linear (DLT) triangulation per (pose, joint), float64, one SVD per joint as pymvg's find3d does.

    pix [B,V,J,3] (u, v, conf) pixels; R [V,3,3] world->cam; t [V,3] camera position; f, c [V,2] pixels.
    View v is used iff conf > min_conf and 0 < u < w-1 and 0 < v < h-1.  P_v = K_v [R_v | -R_v t_v]; rows u P3 - P1 and
    v P3 - P2 per used view; X~ = last right singular vector, X = X~[:3] / X~[3].  Returns (points [B,J,3] with NaN where
    fewer than 2 views are used, views_used [B,J] int32).
    """
    pix = np.asarray(pix)
    w, h = image_size
    B, V, J, _ = pix.shape
    P = np.zeros((V, 3, 4))
    for v in range(V):
        Rv, tv = np.asarray(R[v], dtype=np.float64), np.asarray(t[v], dtype=np.float64)
        K = np.array([[f[v][0], 0.0, c[v][0]], [0.0, f[v][1], c[v][1]], [0.0, 0.0, 1.0]], dtype=np.float64)
        P[v] = K @ np.concatenate([Rv, -(Rv @ tv)[:, None]], axis=1)
    u = pix[..., 0].astype(np.float64)
    vv = pix[..., 1].astype(np.float64)
    use = (pix[..., 2] > np.float32(min_conf)) & (0 < u) & (u < w - 1) & (0 < vv) & (vv < h - 1)   # [B,V,J]
    points = np.full((B, J, 3), np.nan)
    views_used = use.sum(axis=1).astype(np.int32)
    for b in range(B):
        for j in range(J):
            vs = np.flatnonzero(use[b, :, j])
            if len(vs) < 2:
                continue
            A = np.concatenate([np.stack([u[b, v, j] * P[v, 2] - P[v, 0], vv[b, v, j] * P[v, 2] - P[v, 1]]) for v in vs])
            X = np.linalg.svd(A)[2][-1]
            points[b, j] = X[:3] / X[3]
    return points, views_used
