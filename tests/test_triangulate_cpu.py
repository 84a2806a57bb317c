"""Linear multi-view triangulation (MPL/lib/multiviews/triangulate.py:59-115) without a GPU: the oracle recovers the
synthetic generator's 3D targets from its own pixels, ignores views it must ignore, does not depend on view order, and the
C entry point rejects bad arguments before any CUDA call."""
import ctypes

import numpy as np
import pytest

import triangulation_oracle
from oracle import mpl_oracle
from openmpl_b200 import _lib, synth


def _pixels(batch, rig):
    """make_batch's clipped pixels, recovered by inverting the screen normalisation, and its confidences."""
    w, h = rig.image_size
    px = (batch["poses"][..., :2].astype(np.float64) + np.array([1, h / w])) / 2 * w
    return np.concatenate([px, batch["poses"][..., 2:3]], axis=-1).astype(np.float32)


def _tri(pix, rig, R=None, t=None, f=None, c=None, min_conf=0.0):
    return triangulation_oracle.triangulate(pix, rig.R if R is None else R, rig.t if t is None else t,
                                            rig.f if f is None else f, rig.c if c is None else c, rig.image_size, min_conf)


@pytest.mark.parametrize("kind,V", [("h36m", 2), ("h36m", 4), ("cmu", 5)])
def test_oracle_recovers_the_generator_targets(kind, V):
    rig = synth.make_rig(V, kind)
    batch = synth.make_batch(100, rig, seed=7)
    pix = _pixels(batch, rig)
    points, used = _tri(pix, rig)
    np.testing.assert_array_equal(used, (batch["poses"][..., 2] > 0).sum(axis=1))
    ok = used >= 2
    assert ok.mean() > 0.9
    assert np.isnan(points[~ok]).all() and not np.isnan(points[ok]).any()
    assert np.abs(points[ok] - batch["target"][ok]).max() <= 1e-4           # metres


def test_unused_views_change_nothing_and_view_order_does_not_matter():
    rig = synth.make_rig(4, "h36m")
    batch = synth.make_batch(40, rig, seed=2)
    rng = np.random.default_rng(0)
    pix = _pixels(batch, rig)
    pix[..., :2] += rng.normal(0, 2.0, pix[..., :2].shape).astype(np.float32)       # noisy: the solve is not exact
    pix[..., 2] = np.where(pix[..., 2] > 0, rng.uniform(0.05, 1.0, pix[..., 2].shape), 0).astype(np.float32)
    min_conf = 0.3
    base, used = _tri(pix, rig, min_conf=min_conf)
    R, t, f, c = (np.concatenate([a, a[:1]]) for a in (rig.R, rig.t, rig.f, rig.c))   # a fifth camera = view 0
    for extra in ("outside", "low_conf"):
        more = np.concatenate([pix, pix[:, :1]], axis=1)
        if extra == "outside":
            more[:, 4, :, 0] = -3.0                                                       # left of the image
        else:
            more[:, 4, :, 2] = min_conf                                                   # conf <= min_conf
        got, got_used = _tri(more, rig, R, t, f, c, min_conf)
        np.testing.assert_array_equal(got, base)
        np.testing.assert_array_equal(got_used, used)
    perm = [2, 0, 3, 1]
    got, got_used = _tri(pix[:, perm], rig, rig.R[perm], rig.t[perm], rig.f[perm], rig.c[perm], min_conf)
    np.testing.assert_array_equal(got_used, used)
    ok = used >= 2
    assert np.isnan(got[~ok]).all()
    rel = np.linalg.norm(got[ok] - base[ok], axis=-1) / np.linalg.norm(base[ok], axis=-1)     # relative to the point
    assert rel.max() <= 1e-12


def test_triangulate_rejects_bad_arguments_before_any_cuda_call():
    L = _lib.lib()
    buf = ctypes.create_string_buffer(64)      # host memory: never dereferenced on the rejected paths
    p = ctypes.cast(buf, ctypes.c_void_p)

    def call(pix=p, calib=p, batch=4, V=4, J=17, points=p, used=p):
        return L.mpl_triangulate(pix, calib, batch, V, J, 0.0, points, used, None)

    bad = [dict(pix=None), dict(calib=None), dict(points=None), dict(used=None), dict(batch=-1), dict(V=0), dict(V=17),
           dict(J=0), dict(J=-3), dict(batch=0, V=17)]
    for kw in bad:
        assert call(**kw) == _lib.MPL_ERR_INVALID_ARGUMENT, kw
        assert L.mpl_last_error().startswith(b"mpl_triangulate")
    assert call(batch=0) == _lib.MPL_OK
    assert call(batch=0, pix=None, calib=None, points=None, used=None) == _lib.MPL_OK   # an empty tensor has no storage


def test_triangulation_summary_of_the_evaluation_line():
    """evaluate.py's triangulation entry from the masked MPJPE sums: the reference's masked means, the mean over
    triangulated joints only, and the number of under-determined joints."""
    from openmpl_b200 import evaluate
    rng = np.random.default_rng(5)
    B, J = 60, 17
    target = rng.normal(size=(B, J, 3)).astype(np.float32)
    points = (target + rng.normal(0, 0.01, size=(B, J, 3))).astype(np.float32)
    used = rng.integers(0, 4, size=(B, J))
    used[:, 5] = 0                                               # a joint never triangulated
    points[used < 2] = np.nan
    acc = mpl_oracle.metric_sums(points, target, (used >= 2).astype(np.float32))
    s = evaluate.triangulation_summary(acc, J)
    ev = mpl_oracle.evaluate(points, target, True, np.broadcast_to((used >= 2)[..., None], (B, J, 3)))
    assert abs(s["mpjpe_cm"]["absolute"] - ev["mpjpe"]) < 1e-9
    ok = used >= 2
    err = np.linalg.norm(points.astype(np.float64) - target, axis=-1) * 100
    want = np.mean([err[ok[:, j], j].mean() for j in range(J) if ok[:, j].any()])
    assert abs(s["mpjpe_cm"]["triangulated_joints"] - want) < 1e-9
    assert s["under_determined_joints"] == int((~ok).sum())
