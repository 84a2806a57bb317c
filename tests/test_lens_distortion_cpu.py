"""Lens distortion without a GPU: the distortion's numpy twin (synth.distort_pixels) against cv2.projectPoints, the
undistortion oracle (tests/lens_oracle.py) against cv2.undistortPointsIter, the round trip, the fold rule in both directions,
zero coefficients as an exact copy, and the argument checks of the C entry points and the Python wrappers."""
import ctypes

import numpy as np
import pytest
import torch

from openmpl_b200 import _lib, inputs, synth

from lens_oracle import distort, undistort_normalised, undistort_pixels, valid

cv2 = pytest.importorskip("cv2")

# (k1, k2, p1, p2, k3): H36M-like magnitudes, a stronger CMU-like set, and a strong barrel whose fold lies inside the image
LENSES = {"h36m": ((-0.207, 0.248, -0.0009, -0.0016, -0.0031), "h36m"),
          "cmu": ((-0.30, 0.10, 0.001, -0.001, 0.0), "cmu"),
          "fold": ((-0.5, 0.05, 0.001, -0.001, 0.0), "h36m")}


def _camera(kind):
    f0, (w, h), _ = synth.rig_kind(kind)
    return f0, w, h, np.array([[f0, 0, w / 2], [0, f0, h / 2], [0, 0, 1.0]])


def _grid(w, h, n=161):
    u, v = np.meshgrid(np.linspace(0.5, w - 1.5, n), np.linspace(0.5, h - 1.5, n))
    return u.ravel(), v.ravel()


@pytest.mark.parametrize("name", sorted(LENSES))
def test_distortion_twin_matches_opencv_project_points(name):
    k, kind = LENSES[name]
    f0, w, h, K = _camera(kind)
    P = np.random.default_rng(3).uniform(-0.7, 0.7, (4000, 2))
    calib = inputs.pack_calibration(np.eye(3)[None], np.zeros((1, 3)), [[f0, f0]], [[w / 2, h / 2]], (w, h))
    pix = np.stack([f0 * P[:, 0] + w / 2, f0 * P[:, 1] + h / 2, np.ones(len(P))], -1)[None, None].astype(np.float32)
    out = synth.distort_pixels(pix, calib, np.array([k]))[0, 0]
    x = (pix[0, 0, :, 0].astype(np.float64) - w / 2) / f0          # the normalised point of the fp32 pixel
    y = (pix[0, 0, :, 1].astype(np.float64) - h / 2) / f0
    ok = out[:, 2] != 0
    assert ok.mean() > 0.9 and (ok == valid(k, x, y)).all()
    img, _ = cv2.projectPoints(np.stack([x, y, np.ones_like(x)], -1), np.zeros(3), np.zeros(3), K, np.array(k))
    xd, yd, *_ = synth.lens_map(k, x, y)
    np.testing.assert_allclose(np.stack([f0 * xd + w / 2, f0 * yd + h / 2], -1), img[:, 0], rtol=0, atol=1e-9)
    # the fp32 output is the fp64 pixel rounded once: within one fp32 ulp of OpenCV's
    ulp = np.spacing(np.abs(img[ok, 0]).astype(np.float32)).astype(np.float64)
    assert (np.abs(out[ok, :2].astype(np.float64) - img[ok, 0]) <= ulp).all()
    np.testing.assert_array_equal(out[~ok, :2], pix[0, 0, ~ok, :2])


@pytest.mark.parametrize("name", sorted(LENSES))
def test_undistortion_oracle_matches_opencv_over_the_image(name):
    k, kind = LENSES[name]
    f0, w, h, K = _camera(kind)
    u, v = _grid(w, h)
    x, y, ok = undistort_normalised(k, (u - w / 2) / f0, (v - h / 2) / f0)
    ocv = cv2.undistortPointsIter(np.stack([u, v], -1)[:, None], K, np.array(k), None, None,
                                  (cv2.TERM_CRITERIA_COUNT | cv2.TERM_CRITERIA_EPS, 1000, 1e-16))[:, 0]
    px, py, *_ = distort(k, ocv[:, 0], ocv[:, 1])
    converged = f0 * np.hypot(px - (u - w / 2) / f0, py - (v - h / 2) / f0) < 1e-9   # OpenCV's own fixed point reached
    good = converged & valid(k, ocv[:, 0], ocv[:, 1])
    assert good.mean() > 0.95
    assert ok[good].all()                                          # every valid preimage OpenCV finds, Newton finds
    err = f0 * np.abs(np.stack([x, y], -1) - ocv).max(-1)
    assert err[good].max() <= 1e-6
    if name == "fold":
        assert (~ok).sum() > 100 and not good[~ok].any()           # the corners beyond the fold's image have no valid preimage
    else:
        assert ok.all()


@pytest.mark.parametrize("name", ["h36m", "cmu"])
def test_round_trip_recovers_every_valid_point_inside_the_frame(name):
    k, kind = LENSES[name]
    rig = synth.make_rig(5, kind)
    f0, w, h, _ = _camera(kind)
    b = synth.make_batch(300, rig, seed=4)
    px = (b["poses"][..., :2].astype(np.float64) + np.array([1, h / w])) / 2 * w
    x, y = (px[..., 0] - w / 2) / f0, (px[..., 1] - h / 2) / f0
    xd, yd, *_ = distort(k, x, y)
    ud, vd = f0 * xd + w / 2, f0 * yd + h / 2
    keep = valid(k, x, y) & (0 < ud) & (ud < w - 1) & (0 < vd) & (vd < h - 1)
    assert keep.mean() > 0.5
    xr, yr, ok = undistort_normalised(k, xd[keep], yd[keep])
    assert ok.all()
    assert f0 * max(np.abs(xr - x[keep]).max(), np.abs(yr - y[keep]).max()) <= 1e-6
    # through the fp32 pixels of the twin and the oracle: fp32 rounding of the distorted pixel is the only loss
    calib = inputs.pack_calibration(rig.R, rig.t, rig.f, rig.c, rig.image_size)
    pix = np.concatenate([px, np.ones(px.shape[:-1] + (1,))], -1).astype(np.float32)
    dist = np.tile(np.array(k), (5, 1))
    back, _ = undistort_pixels(synth.distort_pixels(pix, calib, dist), calib, dist)
    sel = keep & (back[..., 2] != 0)
    assert sel.sum() == keep.sum()
    assert np.abs(back[sel][:, :2].astype(np.float64) - pix[sel][:, :2]).max() <= 1e-3


def test_points_past_a_fold_are_invalid_both_ways():
    k, kind = LENSES["fold"]
    f0, w, h, _ = _camera(kind)
    k1, k2 = k[0], k[1]
    s_fold = (1.5 - np.sqrt(2.25 - 4 * 0.25)) / (2 * 0.25)          # g(s) = 1 - 1.5 s + 0.25 s^2 = 0
    assert abs(1 + 3 * k1 * s_fold + 5 * k2 * s_fold ** 2) < 1e-12
    r_fold = np.sqrt(s_fold)
    t = np.linspace(0, 2 * np.pi, 64, endpoint=False)
    for r, want in ((0.97 * r_fold, True), (1.03 * r_fold, False), (1.5 * r_fold, False)):
        x, y = r * np.cos(t), r * np.sin(t)
        assert (valid(k, x, y) == want).all() and (synth.lens_valid(k, x, y) == want).all(), r
        calib = inputs.pack_calibration(np.eye(3)[None], np.zeros((1, 3)), [[f0, f0]], [[w / 2, h / 2]], (w, h))
        pix = np.stack([f0 * x + w / 2, f0 * y + h / 2, np.ones_like(x)], -1)[None, None].astype(np.float32)
        out = synth.distort_pixels(pix, calib, np.array([k]))
        assert ((out[..., 2] != 0) == want).all()
    # detected pixels beyond the image of the fold circle have no preimage: the inversion fails
    r_max = r_fold * (1 + k1 * s_fold + k2 * s_fold ** 2)
    xd, yd = 1.02 * r_max * np.cos(t), 1.02 * r_max * np.sin(t)
    assert not undistort_normalised(k, xd, yd)[2].any()
    xd, yd = 0.98 * r_max * np.cos(t), 0.98 * r_max * np.sin(t)
    x, y, ok = undistort_normalised(k, xd, yd)
    assert ok.all() and (np.hypot(x, y) < r_fold).all()


def test_zero_coefficients_copy_the_pixels():
    rig = synth.make_rig(4, "cmu")
    b = synth.make_batch(200, rig, seed=8)
    w, h = rig.image_size
    px = (b["poses"][..., :2].astype(np.float64) + np.array([1, h / w])) / 2 * w
    pix = np.concatenate([px, b["poses"][..., 2:3]], -1).astype(np.float32)
    pix[::5, 1, :, :2] += np.float32(900.0)                          # some outside the frame
    calib = inputs.pack_calibration(rig.R, rig.t, rig.f, rig.c, rig.image_size)
    zero = np.zeros((4, 5))
    np.testing.assert_array_equal(synth.distort_pixels(pix, calib, zero), pix)
    odd = pix.copy()
    odd[::7, :, 3, 0], odd[::11, 1, :, 1], odd[..., 2] = -0.0, np.nan, 0.5         # -0 and NaN pixels with conf > 0
    out = synth.distort_pixels(odd, calib, zero)
    assert out.tobytes() == odd.tobytes()
    lens = np.zeros((4, 5))
    lens[0] = LENSES["cmu"][0]                                                       # a lens on view 0 only
    out = synth.distort_pixels(odd, calib, lens)
    assert out[:, 1:].tobytes() == odd[:, 1:].tobytes()
    odd[::11, 0, :, 1] = np.nan                                                      # under a lens a NaN pixel is not valid
    out = synth.distort_pixels(odd, calib, lens)
    assert (out[::11, 0, :, 2] == 0).all()
    out, _ = undistort_pixels(pix, calib, zero)
    np.testing.assert_array_equal(out[..., :2], pix[..., :2])
    inside = (0 < pix[..., 0]) & (pix[..., 0] < w - 1) & (0 < pix[..., 1]) & (pix[..., 1] < h - 1)
    np.testing.assert_array_equal(out[..., 2], np.where(inside, pix[..., 2], 0))


def test_entry_points_reject_bad_arguments_before_any_cuda_call():
    L = _lib.lib()
    buf = ctypes.create_string_buffer(64)                            # host memory: never dereferenced on the rejected paths
    p = ctypes.cast(buf, ctypes.c_void_p)
    nan, inf = float("nan"), float("inf")

    def calls(batch=4, V=4, J=17, pin=p, pout=p, calib=p, dist=p, cs=0, ds=0, mx=0.0, my=0.0, distort=True):
        # distort=False for margin cases: the distortion has no margin, so those arguments are valid for it and it would
        # launch on the host buffer
        if distort:
            yield "mpl_distort_pixels_strided", L.mpl_distort_pixels_strided(pin, pout, calib, cs, dist, ds, batch, V, J, None)
        yield "mpl_undistort_pixels_strided", L.mpl_undistort_pixels_strided(pin, pout, calib, cs, dist, ds, mx, my, batch, V,
                                                                           J, None)
        if cs == 0 and ds == 0:                                      # the plain forms forward with both strides 0
            if distort:
                yield "mpl_distort_pixels_strided", L.mpl_distort_pixels(pin, pout, calib, dist, batch, V, J, None)
            yield "mpl_undistort_pixels_strided", L.mpl_undistort_pixels(pin, pout, calib, dist, mx, my, batch, V, J, None)

    bad = [dict(pin=None), dict(pout=None), dict(calib=None), dict(dist=None), dict(batch=-1), dict(V=0), dict(V=17),
           dict(J=0), dict(cs=-18), dict(cs=1), dict(cs=18 * 4 - 1), dict(ds=-5), dict(ds=1), dict(ds=5 * 4 - 1),
           dict(batch=0, V=17), dict(batch=0, ds=3)]
    bad_margin = [dict(mx=-1.0, distort=False), dict(my=-0.5, distort=False), dict(mx=nan, distort=False),
                  dict(my=inf, distort=False), dict(batch=0, mx=-1.0, distort=False)]
    for kw in bad + bad_margin:
        for name, status in calls(**kw):
            assert status == _lib.MPL_ERR_INVALID_ARGUMENT, (name, kw)
            assert L.mpl_last_error().decode().startswith(name), (name, kw)
    for kw in (dict(batch=0), dict(batch=0, pin=None, pout=None, calib=None, dist=None), dict(batch=0, cs=72, ds=20),
               dict(batch=0, cs=100, ds=33, mx=500.0, my=0.0)):
        for name, status in calls(**kw):
            assert status == _lib.MPL_OK, (name, kw)


def test_wrappers_reject_bad_arguments_before_any_cuda_call():
    rig = synth.make_rig(4, "h36m")
    calib = inputs.pack_calibration(rig.R, rig.t, rig.f, rig.c, rig.image_size)
    pix = torch.zeros((3, 4, 17, 3))
    dist = np.zeros((4, 5))
    for d in (np.zeros((3, 5)), np.zeros((4, 4)), np.zeros((2, 4, 5)), np.zeros(5), np.zeros((3, 4, 5, 1))):
        with pytest.raises(ValueError, match="dist must be"):
            inputs.distort_pixels(pix, calib, d)
        with pytest.raises(ValueError, match="dist must be"):
            inputs.undistort_pixels(pix, calib, d, margin=0.0)
    with pytest.raises(ValueError, match="per-pose calibration"):
        inputs.undistort_pixels(pix, np.zeros((2, 4, 18)), dist, margin=0.0)
    for m in (-1.0, (0.0, -2.0), float("nan"), (float("inf"), 0.0)):
        with pytest.raises(ValueError, match="margin"):
            inputs.undistort_pixels(pix, calib, dist, margin=m)
    for bad in (pix.double(), pix.transpose(1, 2), pix[..., :2]):
        with pytest.raises(ValueError, match="in place"):
            inputs.distort_pixels(bad, calib, dist)
    for bad in (pix[..., :2], pix[0], pix[None]):
        with pytest.raises(ValueError, match=r"\[B, V, J, 3\]"):
            inputs.undistort_pixels(bad, calib, dist, margin=0.0)


def test_evaluation_rejects_bad_lens_coefficients_on_the_command_line():
    from openmpl_b200 import evaluate
    for arg in ("--lens-distortion=nan,0,0,0,0", "--lens-distortion=0,inf,0,0,0", "--lens-distortion=1,2",
                "--lens-distortion=a,b,c,d,e"):
        with pytest.raises(SystemExit):
            evaluate.main([arg])
