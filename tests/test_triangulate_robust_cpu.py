"""Robust multi-view triangulation (pair RANSAC with the MSAC cost + confidence-weighted refit) without a GPU: the numpy
oracle recovers the generator's targets, rejects a confident false detection that breaks the linear DLT, reduces to the
linear DLT when every view agrees, does not depend on view order, and the C entry point rejects bad arguments before any
CUDA call."""
import ctypes

import numpy as np
import pytest

import robust_triangulation_oracle as rto
import triangulation_oracle
from openmpl_b200 import _lib, synth


def _pixels(batch, rig):
    """make_batch's clipped pixels, recovered by inverting the screen normalisation, and its confidences."""
    w, h = rig.image_size
    px = (batch["poses"][..., :2].astype(np.float64) + np.array([1, h / w])) / 2 * w
    return np.concatenate([px, batch["poses"][..., 2:3]], axis=-1).astype(np.float32)


def _candidates(pix, rig, min_conf=0.0):
    w, h = rig.image_size
    u, v = pix[..., 0].astype(np.float64), pix[..., 1].astype(np.float64)
    cand = (pix[..., 2] > np.float32(min_conf)) & (0 < u) & (u < w - 1) & (0 < v) & (v < h - 1)          # [B,V,J]
    return (cand * (1 << np.arange(pix.shape[1]))[None, :, None]).sum(axis=1).astype(np.int32)


def _robust(pix, rig, perm=None, **kw):
    R, t, f, c = (a if perm is None else a[perm] for a in (rig.R, rig.t, rig.f, rig.c))
    return rto.triangulate_robust(pix if perm is None else pix[:, perm], R, t, f, c, rig.image_size, **kw)


@pytest.mark.parametrize("kind,V", [("h36m", 2), ("h36m", 4), ("cmu", 5)])
def test_oracle_recovers_the_generator_targets(kind, V):
    rig = synth.make_rig(V, kind)
    batch = synth.make_batch(60, rig, seed=7)
    pix = _pixels(batch, rig)
    points, inliers, _ = _robust(pix, rig)
    cand = _candidates(pix, rig)
    ok = np.array([bin(m).count("1") >= 2 for m in cand.ravel()]).reshape(cand.shape)
    assert ok.mean() > 0.9
    np.testing.assert_array_equal(inliers, np.where(ok, cand, 0))
    assert np.isnan(points[~ok]).all() and not np.isnan(points[ok]).any()
    assert np.abs(points[ok] - batch["target"][ok]).max() <= 1e-4                                        # metres


@pytest.mark.parametrize("kind,V", [("h36m", 4), ("cmu", 5), ("h36m", 8)])
def test_one_confident_false_detection_is_rejected(kind, V):
    """One candidate view per joint moved half the image away with conf 1: the robust point stays on the target and its
    mask drops exactly that view, while the linear DLT is pulled off by more than 10 cm."""
    rig = synth.make_rig(V, kind)
    w, h = rig.image_size
    batch = synth.make_batch(40, rig, seed=3)
    pix = _pixels(batch, rig)
    cand = _candidates(pix, rig)
    B, _, J, _ = pix.shape
    bad = np.zeros((B, J), dtype=np.int64)
    for b in range(B):
        for j in range(J):
            views = [v for v in range(V) if (cand[b, j] >> v) & 1]
            if views:
                v = views[(b + j) % len(views)]
                bad[b, j] = v
                pix[b, v, j, 0] = (pix[b, v, j, 0] + w / 2) % (w - 2) + 1
                pix[b, v, j, 1] = (pix[b, v, j, 1] + h / 2) % (h - 2) + 1
                pix[b, v, j, 2] = 1.0
    items = np.array([bin(m).count("1") >= 3 for m in cand.ravel()]).reshape(cand.shape)   # the outlier is identifiable
    assert items.mean() > 0.5
    points, inliers, _ = _robust(pix, rig)
    lin, _ = triangulation_oracle.triangulate(pix, rig.R, rig.t, rig.f, rig.c, rig.image_size)
    target = batch["target"].astype(np.float64)
    np.testing.assert_array_equal(inliers[items], (cand & ~(1 << bad).astype(np.int32))[items])
    assert np.linalg.norm(points[items] - target[items], axis=-1).max() < 0.01
    assert np.linalg.norm(lin[items] - target[items], axis=-1).min() > 0.10


def test_all_inliers_with_unit_confidence_is_the_linear_dlt():
    rig = synth.make_rig(4, "h36m")
    batch = synth.make_batch(40, rig, seed=5, conf_mode="ones")
    pix = _pixels(batch, rig)
    rng = np.random.default_rng(1)
    pix[..., :2] += rng.normal(0, 1.0, pix[..., :2].shape).astype(np.float32)         # well inside the 10 px threshold
    points, inliers, _ = _robust(pix, rig)
    lin, used = triangulation_oracle.triangulate(pix, rig.R, rig.t, rig.f, rig.c, rig.image_size)
    full = inliers == _candidates(pix, rig)
    assert (full | (used < 2)).mean() > 0.99
    ok = full & (used >= 2)
    np.testing.assert_array_equal(points[ok], lin[ok])


@pytest.mark.parametrize("min_conf", [0.0, 0.5])
def test_view_order_permutes_the_mask_and_keeps_the_points(min_conf):
    rig = synth.make_rig(5, "cmu")
    w, h = rig.image_size
    batch = synth.make_batch(30, rig, seed=9)
    pix = _pixels(batch, rig)
    rng = np.random.default_rng(2)
    pix[..., :2] += (rng.normal(0, 2.0, pix[..., :2].shape) / np.maximum(pix[..., 2:3], 0.3)).astype(np.float32)
    out = rng.random(pix.shape[:3]) < 0.15                                                # confident false detections
    pix[..., 0] = np.where(out, rng.uniform(1, w - 2, out.shape), pix[..., 0])
    pix[..., 1] = np.where(out, rng.uniform(1, h - 2, out.shape), pix[..., 1])
    pix[..., 2] = np.where(out, rng.uniform(0.3, 1.0, out.shape), pix[..., 2])
    base, mask, near = _robust(pix, rig, min_conf=min_conf)
    perm = np.array([3, 0, 4, 1, 2])
    got, gmask, gnear = _robust(pix, rig, perm=perm, min_conf=min_conf)
    # bit k of the permuted mask is view perm[k]
    unperm = sum(((gmask >> k) & 1) << int(perm[k]) for k in range(5))
    sure = ~(near | gnear)
    assert sure.mean() > 0.9 and (mask[sure] != 0).mean() > 0.5
    np.testing.assert_array_equal(unperm[sure], mask[sure])
    det = sure & (mask != 0)
    assert np.isnan(got[sure & (mask == 0)]).all()
    rel = np.linalg.norm(got[det] - base[det], axis=-1) / np.linalg.norm(base[det], axis=-1)
    assert rel.max() <= 1e-12


def test_triangulate_robust_rejects_bad_arguments_before_any_cuda_call():
    L = _lib.lib()
    buf = ctypes.create_string_buffer(64)      # host memory: never dereferenced on the rejected paths
    p = ctypes.cast(buf, ctypes.c_void_p)

    def call(pix=p, calib=p, batch=4, V=4, J=17, tau=10.0, points=p, inl=p):
        return L.mpl_triangulate_robust(pix, calib, batch, V, J, 0.0, tau, points, inl, None)

    bad = [dict(pix=None), dict(calib=None), dict(points=None), dict(inl=None), dict(batch=-1), dict(V=0), dict(V=17),
           dict(J=0), dict(J=-3), dict(tau=0.0), dict(tau=-1.0), dict(tau=float("nan")), dict(tau=float("inf")),
           dict(batch=0, V=17), dict(batch=0, tau=0.0)]
    for kw in bad:
        assert call(**kw) == _lib.MPL_ERR_INVALID_ARGUMENT, kw
        assert L.mpl_last_error().startswith(b"mpl_triangulate_robust"), kw
    assert call(batch=0) == _lib.MPL_OK
    assert call(batch=0, pix=None, calib=None, points=None, inl=None) == _lib.MPL_OK     # an empty tensor has no storage
