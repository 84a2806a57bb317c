"""Levenberg-Marquardt refinement of triangulated points without a GPU: the numpy oracle of mpl_triangulate_refine reaches
the optimum scipy's least_squares finds, never raises the cost, leaves exact points where they are, follows the
not-refined rules, lowers the error of the linear DLT on noisy detections, and the C entry points and the Python wrapper
reject bad arguments before any CUDA call."""
import ctypes

import numpy as np
import pytest
import torch
from scipy.optimize import least_squares

import refine_triangulation_oracle as rfo
import robust_triangulation_oracle as rto
import triangulation_oracle
from openmpl_b200 import _lib, inputs, synth


def _pixels(batch, rig):
    """make_batch's clipped pixels, recovered by inverting the screen normalisation, and its confidences."""
    w, h = rig.image_size
    px = (batch["poses"][..., :2].astype(np.float64) + np.array([1, h / w])) / 2 * w
    return np.concatenate([px, batch["poses"][..., 2:3]], axis=-1).astype(np.float32)


def _calib(rig):
    return inputs.pack_calibration(rig.R, rig.t, rig.f, rig.c, rig.image_size)


def _noisy(kind, V, B, seed, p_outlier=0.0):
    rig = synth.make_rig(V, kind)
    batch = synth.make_batch(B, rig, seed=seed)
    pix = synth.detector_noise(_pixels(batch, rig), rig.image_size, seed + 100, 0, 2.0, p_outlier, 0.0)
    return rig, pix, batch["target"].astype(np.float64)


def _linear(pix, rig):
    return triangulation_oracle.triangulate(pix, rig.R, rig.t, rig.f, rig.c, rig.image_size)


def _cost_at(pix, calib, X, use):
    """C at fp64 points X [B, J, 3] over the views of use [B, V, J], recomputed independently of the oracle's loop."""
    P, _ = rfo.projections(calib)
    p = np.einsum("vrk,bjk->bvjr", P, np.concatenate([X, np.ones(X.shape[:-1] + (1,))], axis=-1))
    r = p[..., :2] / p[..., 2:3] - pix[..., :2].astype(np.float64)
    behind = (p[..., 2] <= 0) & use
    c = np.where(use, pix[..., 2].astype(np.float64) ** 2 * (r * r).sum(-1), 0.0).sum(axis=1)
    return np.where(behind.any(axis=1), np.inf, c)


@pytest.mark.parametrize("kind,V", [("h36m", 4), ("cmu", 5)])
def test_oracle_reaches_the_least_squares_optimum(kind, V):
    rig, pix, _ = _noisy(kind, V, 30, seed=3)
    calib = _calib(rig)
    lin, _ = _linear(pix, rig)
    init = lin.astype(np.float32)
    res = rfo.refine(pix, calib, init, max_iters=100)
    P, wh = rfo.projections(calib)
    use = rfo.candidates(pix, wh[None])
    items = np.argwhere(res["refined"] & res["by_step"])
    assert res["refined"].mean() > 0.9 and len(items) > 0.8 * res["refined"].sum()
    for b, j in items:
        vs = np.flatnonzero(use[b, :, j])
        uv = pix[b, vs, j, :2].astype(np.float64)
        sw = pix[b, vs, j, 2].astype(np.float64)

        def resid(X):
            p = P[vs] @ np.append(X, 1.0)
            return ((p[:, :2] / p[:, 2:3] - uv) * sw[:, None]).ravel()

        ls = least_squares(resid, init[b, j].astype(np.float64), method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15)
        c_ls = float(resid(ls.x) @ resid(ls.x))
        assert abs(res["cost"][b, j] - c_ls) <= 1e-9 * c_ls + 1e-18, (b, j)
        assert np.abs(res["X"][b, j] - ls.x).max() <= 1e-6, (b, j)                      # metres


@pytest.mark.parametrize("kind,V,p_outlier", [("h36m", 4, 0.0), ("cmu", 5, 0.0), ("h36m", 4, 0.1)])
def test_refinement_never_raises_the_cost(kind, V, p_outlier):
    rig, pix, _ = _noisy(kind, V, 30, seed=5, p_outlier=p_outlier)
    calib = _calib(rig)
    lin, _ = _linear(pix, rig)
    res = rfo.refine(pix, calib, lin.astype(np.float32))
    use = rfo.candidates(pix, rfo.projections(calib)[1][None])
    ok = res["refined"]
    assert ok.mean() > 0.9
    c0 = _cost_at(pix, calib, lin.astype(np.float32).astype(np.float64), use)
    c1 = _cost_at(pix, calib, res["X"], use)
    assert np.all(c1[ok] <= c0[ok] * (1 + 1e-12))
    np.testing.assert_allclose(c1[ok], res["cost"][ok], rtol=1e-10)
    np.testing.assert_allclose(res["reproj_px"][ok], np.sqrt(res["cost"][ok] / np.where(use, pix[..., 2] ** 2.0, 0).sum(1)[ok]),
                               rtol=1e-6)


@pytest.mark.parametrize("kind,V", [("h36m", 4), ("cmu", 5), ("h36m", 8)])
def test_exact_points_stay_where_they_are(kind, V):
    """The pixels are the targets' projections rounded to fp32, so the optimum is the target up to that rounding.  (With
    two views it is amplified near the baseline: up to 2e-6 m, so V = 2 is left out.)"""
    rig = synth.make_rig(V, kind)
    batch = synth.make_batch(40, rig, seed=7)
    pix = _pixels(batch, rig)
    res = rfo.refine(pix, _calib(rig), batch["target"])
    ok = res["refined"]
    assert ok.mean() > 0.9
    assert np.abs(res["X"][ok] - batch["target"][ok]).max() <= 1e-6                        # metres
    assert res["reproj_px"][ok].max() < 1e-3


def test_items_that_are_not_refined_keep_their_init():
    V = 4
    rig = synth.make_rig(V, "h36m")
    calib = _calib(rig)
    batch = synth.make_batch(1, rig, seed=2, conf_mode="ones")
    pix = _pixels(batch, rig)[:, :, :5].copy()
    init = batch["target"][:, :5].astype(np.float32).copy()
    assert rfo.candidates(pix, rfo.projections(calib)[1][None]).all()
    init[0, 0] = [np.nan, 1.0, 2.0]                                   # init not finite
    pix[0, 1:, 1, 2] = 0.0                                            # one candidate view left
    mask = np.full((1, 5), 0xF, dtype=np.int32)
    mask[0, 2] = 0b0100                                               # a mask that leaves one view
    mask[0, 4] = 0x7FFFFFF0 | 0b0011                                  # bits >= V are ignored: views 0, 1 used
    # behind camera 0: the target mirrored through its centre
    init[0, 3] = 2 * rig.t[0] - batch["target"][0, 3]
    res = rfo.refine(pix, calib, init, view_mask=mask)
    np.testing.assert_array_equal(res["refined"][0], [False, False, False, False, True])
    np.testing.assert_array_equal(res["points"][0, :4].view(np.int32), init[0, :4].view(np.int32))
    assert np.isnan(res["reproj_px"][0, :4]).all() and np.isfinite(res["reproj_px"][0, 4])


@pytest.mark.parametrize("kind,V", [("h36m", 4), ("cmu", 5)])
def test_refinement_lowers_the_error_of_the_linear_dlt(kind, V):
    """Gaussian noise of std 2 px / conf: the conf^2-weighted optimum is the maximum-likelihood point, the DLT is not."""
    rig, pix, target = _noisy(kind, V, 120, seed=11)
    lin, used = _linear(pix, rig)
    res = rfo.refine(pix, _calib(rig), lin.astype(np.float32))
    ok = (used >= 2) & res["refined"]
    e0 = np.linalg.norm(lin[ok] - target[ok], axis=-1).mean()
    e1 = np.linalg.norm(res["X"][ok] - target[ok], axis=-1).mean()
    assert e1 <= 0.9 * e0, (e0, e1)


def test_refining_the_robust_point_over_its_inliers_does_not_raise_the_error():
    rig, pix, target = _noisy("h36m", 4, 60, seed=13, p_outlier=0.1)
    rob, inl, _ = rto.triangulate_robust(pix, rig.R, rig.t, rig.f, rig.c, rig.image_size)
    res = rfo.refine(pix, _calib(rig), rob.astype(np.float32), view_mask=inl)
    ok = inl != 0
    np.testing.assert_array_equal(res["refined"], ok)
    e0 = np.linalg.norm(rob[ok] - target[ok], axis=-1).mean()
    e1 = np.linalg.norm(res["X"][ok] - target[ok], axis=-1).mean()
    assert e1 <= e0, (e0, e1)


def test_triangulate_refine_rejects_bad_arguments_before_any_cuda_call():
    L = _lib.lib()
    buf = ctypes.create_string_buffer(64)      # host memory: never dereferenced on the rejected paths
    p = ctypes.cast(buf, ctypes.c_void_p)

    def call(pix=p, calib=p, stride=None, batch=4, V=4, J=17, mask=None, init=p, iters=20, points=p, rp=p):
        if stride is None:
            return L.mpl_triangulate_refine(pix, calib, batch, V, J, 0.0, mask, init, iters, points, rp, None)
        return L.mpl_triangulate_refine_strided(pix, calib, stride, batch, V, J, 0.0, mask, init, iters, points, rp, None)

    bad = [dict(pix=None), dict(calib=None), dict(init=None), dict(points=None), dict(rp=None), dict(batch=-1), dict(V=0),
           dict(V=17), dict(J=0), dict(J=-3), dict(iters=0), dict(iters=101), dict(iters=-1), dict(stride=-18),
           dict(stride=1), dict(stride=18 * 4 - 1), dict(batch=0, V=17), dict(batch=0, iters=0), dict(batch=0, stride=5)]
    for kw in bad:
        for stride in ([None, 0] if "stride" not in kw else [kw.pop("stride")]):
            assert call(stride=stride, **kw) == _lib.MPL_ERR_INVALID_ARGUMENT, (kw, stride)
            assert L.mpl_last_error().startswith(b"mpl_triangulate_refine_strided"), (kw, stride)
    assert call(batch=0) == _lib.MPL_OK
    assert call(batch=0, pix=None, calib=None, init=None, points=None, rp=None) == _lib.MPL_OK   # empty tensors
    assert call(batch=0, stride=18 * 4, iters=100) == _lib.MPL_OK


def test_wrapper_rejects_badly_shaped_init_and_view_mask():
    B, V, J = 3, 4, 17
    pix = torch.zeros(B, V, J, 3)
    calib = np.zeros((V, 18))
    for init in (torch.zeros(B, J), torch.zeros(B, J + 1, 3), torch.zeros(B + 1, J, 3), torch.zeros(B, J, 4)):
        with pytest.raises(ValueError, match="init"):
            inputs.refine_triangulation(pix, calib, init)
    init = torch.zeros(B, J, 3)
    for mask in (torch.zeros(B, J, dtype=torch.int64), torch.zeros(B, J), torch.zeros(B, J - 1, dtype=torch.int32),
                 torch.zeros(B, J, 1, dtype=torch.int32), torch.zeros(B, dtype=torch.int32)):
        with pytest.raises(ValueError, match="view_mask"):
            inputs.refine_triangulation(pix, calib, init, view_mask=mask)
