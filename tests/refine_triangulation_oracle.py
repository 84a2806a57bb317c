"""Test-side reference for mpl_triangulate_refine: Levenberg-Marquardt on the conf^2-weighted reprojection error, restated
in plain numpy float64 from its definition in include/mpl_b200.h, one (pose, joint) item at a time.  The reference has no
refinement; the product path never imports this module."""
from __future__ import annotations

import numpy as np


def projections(calib):
    """calib [..., V, 18] (R row-major, t, fx, fy, cx, cy, w, h) -> P = K [R | -R t] [..., V, 3, 4] and (w, h) [..., V, 2]."""
    calib = np.asarray(calib, dtype=np.float64)
    R = calib[..., :9].reshape(calib.shape[:-1] + (3, 3))
    t = calib[..., 9:12]
    K = np.zeros(calib.shape[:-1] + (3, 3))
    K[..., 0, 0], K[..., 1, 1] = calib[..., 12], calib[..., 13]
    K[..., 0, 2], K[..., 1, 2], K[..., 2, 2] = calib[..., 14], calib[..., 15], 1.0
    Rt = np.concatenate([R, -(R @ t[..., None])], axis=-1)
    return K @ Rt, calib[..., 16:18]


def candidates(pix, wh, min_conf=0.0):
    """[B, V, J] bool: the views mpl_triangulate uses (conf > min_conf, strictly inside the w x h image)."""
    pix = np.asarray(pix)
    u, v = pix[..., 0].astype(np.float64), pix[..., 1].astype(np.float64)
    w, h = wh[..., 0][..., None], wh[..., 1][..., None]                                  # [B or 1, V, 1]
    return (pix[..., 2] > np.float32(min_conf)) & (0 < u) & (u < w - 1) & (0 < v) & (v < h - 1)


def cost(P, X, uv, wts):
    """C(X) over the views P [n, 3, 4] with pixels uv [n, 2] and weights wts [n]: +inf where a view sees X at a depth that
    is not > 0 or not finite."""
    p = P @ np.append(X, 1.0)
    if not np.all((p[:, 2] > 0) & np.isfinite(p[:, 2])):
        return np.inf
    r = p[:, :2] / p[:, 2:3] - uv
    return float(np.sum(wts * np.sum(r * r, axis=1)))


def refine_item(P, X0, uv, wts, max_iters=20):
    """One item over its used views.  Returns (X fp64, C(X), stopped by the step rule, iterations run)."""
    X = np.asarray(X0, dtype=np.float64).copy()
    C = cost(P, X, uv, wts)
    mu, A, g, relin = 0.0, None, None, True
    for k in range(1, max_iters + 1):
        if relin:
            p = P @ np.append(X, 1.0)
            q = p[:, :2] / p[:, 2:3]
            D = (P[:, :2, :3] - q[:, :, None] * P[:, 2:3, :3]) / p[:, 2, None, None]    # [n, 2, 3]
            A = np.einsum("n,nri,nrk->ik", wts, D, D)
            g = np.einsum("n,nri,nr->i", wts, D, q - uv)
            relin = False
            if k == 1:
                mu = 1e-3 * A.diagonal().max()
        M = A + mu * np.eye(3)
        try:
            L = np.linalg.cholesky(M)
        except np.linalg.LinAlgError:
            L = None
        if L is None or not np.all(np.isfinite(L)):
            mu *= 10.0
            continue
        d = np.linalg.solve(L.T, np.linalg.solve(L, -g))
        step_small = np.linalg.norm(d) <= 1e-10 * (np.linalg.norm(X) + 1e-10)
        Cn = cost(P, X + d, uv, wts)
        if Cn < C:
            X, C, mu, relin = X + d, Cn, mu / 10.0, True
        else:
            mu *= 10.0
        if step_small:
            return X, C, True, k
    return X, C, False, max_iters


def refine(pix, calib, init, view_mask=None, min_conf=0.0, max_iters=20):
    """mpl_triangulate_refine over a batch.  pix [B, V, J, 3], calib [V, 18] or [B, V, 18], init [B, J, 3] fp32, view_mask
    None or [B, J] int.  Returns a dict of points [B, J, 3] fp32 (init where not refined), reproj_px [B, J] fp32 (NaN where
    not refined), refined [B, J] bool, X [B, J, 3] fp64, cost and cost0 [B, J] fp64, by_step [B, J] bool (the step rule
    stopped the item), iters [B, J]."""
    pix = np.asarray(pix)
    init = np.asarray(init, dtype=np.float32)
    B, V, J, _ = pix.shape
    P, wh = projections(calib)
    if P.ndim == 3:
        P, wh = np.broadcast_to(P, (B,) + P.shape), np.broadcast_to(wh, (B,) + wh.shape)
    use = candidates(pix, wh, min_conf)                                                  # [B, V, J]
    if view_mask is not None:
        bits = (np.asarray(view_mask, dtype=np.int64)[:, None, :] >> np.arange(V)[None, :, None]) & 1
        use &= bits.astype(bool)
    out = dict(points=init.copy(), reproj_px=np.full((B, J), np.nan, dtype=np.float32), refined=np.zeros((B, J), bool),
               X=init.astype(np.float64), cost=np.full((B, J), np.nan), cost0=np.full((B, J), np.nan),
               by_step=np.zeros((B, J), bool), iters=np.zeros((B, J), np.int32))
    for b in range(B):
        for j in range(J):
            vs = np.flatnonzero(use[b, :, j])
            X0 = init[b, j].astype(np.float64)
            if not np.all(np.isfinite(X0)) or len(vs) < 2:
                continue
            uv = pix[b, vs, j, :2].astype(np.float64)
            wts = pix[b, vs, j, 2].astype(np.float64) ** 2
            C0 = cost(P[b, vs], X0, uv, wts)
            if not np.isfinite(C0):
                continue
            X, C, by_step, k = refine_item(P[b, vs], X0, uv, wts, max_iters)
            out["points"][b, j] = X.astype(np.float32)
            out["reproj_px"][b, j] = np.float32(np.sqrt(C / wts.sum()))
            out["refined"][b, j], out["X"][b, j], out["cost"][b, j], out["cost0"][b, j] = True, X, C, C0
            out["by_step"][b, j], out["iters"][b, j] = by_step, k
    return out
