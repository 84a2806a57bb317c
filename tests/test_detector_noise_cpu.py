"""The detector-error model's numpy twin (synth.detector_noise) without a GPU: it depends only on (seed, global pose index),
zero parameters are the identity, entries behind the camera stay, the miss / outlier rates and the confidence-scaled
Gaussian have the stated statistics, and the C entry point rejects bad arguments before any CUDA call."""
import ctypes

import numpy as np
import pytest

from openmpl_b200 import _lib, synth


def _raw(n, rig, seed=1, start=0):
    """Raw (u, v, conf) pixels of make_batch, with conf 0 on a few entries as the device generator writes behind-camera ones."""
    b = synth.make_batch(n, rig, seed=seed, start=start)
    w, h = rig.image_size
    px = (b["poses"][..., :2].astype(np.float64) + np.array([1, h / w])) / 2 * w
    return np.concatenate([px, b["poses"][..., 2:3]], axis=-1).astype(np.float32)


def test_noise_depends_only_on_seed_and_global_index():
    rig = synth.make_rig(4, "h36m")
    pix = _raw(50, rig)
    whole = synth.detector_noise(pix, rig.image_size, 3, 0, 2.0, 0.1, 0.05)
    for s, n in ((0, 7), (7, 20), (27, 23), (49, 1)):
        part = synth.detector_noise(pix[s:s + n], rig.image_size, 3, s, 2.0, 0.1, 0.05)
        np.testing.assert_array_equal(part, whole[s:s + n])
    other = synth.detector_noise(pix, rig.image_size, 4, 0, 2.0, 0.1, 0.05)
    assert not np.array_equal(other, whole)


def test_zero_parameters_are_the_identity_and_conf_zero_is_untouched():
    rig = synth.make_rig(5, "cmu")
    pix = _raw(40, rig)
    pix[::3, 1, :, 2] = 0.0                                        # behind the camera
    np.testing.assert_array_equal(synth.detector_noise(pix, rig.image_size, 1, 10, 0.0, 0.0, 0.0), pix)
    noisy = synth.detector_noise(pix, rig.image_size, 1, 10, 3.0, 0.3, 0.3)
    dead = pix[..., 2] == 0
    assert dead.any()
    np.testing.assert_array_equal(noisy[dead], pix[dead])
    assert (noisy[~dead] != pix[~dead]).any(axis=-1).all()


def test_rates_and_noise_statistics():
    rig = synth.make_rig(4, "h36m")
    w, h = rig.image_size
    n = 16000                                                      # 16000 x 4 x 17 = 1.09e6 entries
    pix = np.zeros((n, 4, 17, 3), dtype=np.float32)
    pix[..., 0], pix[..., 1] = 400.0, 600.0
    pix[..., 2] = np.float32(0.3) + np.float32(0.7) * np.linspace(0, 1, n * 68, dtype=np.float32).reshape(n, 4, 17)
    sigma, po, pm = 2.0, 0.1, 0.05
    out = synth.detector_noise(pix, rig.image_size, 11, 5, sigma, po, pm)
    N = pix[..., 0].size
    miss = out[..., 2] == 0
    moved = ~miss & (out[..., 2] != pix[..., 2])                   # an outlier draws a new confidence
    for k, p in ((miss.sum(), pm), (moved.sum(), po)):
        assert abs(k - N * p) < 5 * np.sqrt(N * p * (1 - p)), (k, N * p)
    assert (out[moved, 0] >= 0).all() and (out[moved, 0] <= w - 1).all()
    assert (out[moved, 1] >= 0).all() and (out[moved, 1] <= h - 1).all()
    assert (out[moved, 2] >= 0.3).all() and (out[moved, 2] <= 1.0).all()
    np.testing.assert_array_equal(out[miss][:, :2], pix[miss][:, :2])
    keep = ~miss & ~moved
    z = np.concatenate([(out[keep, 0].astype(np.float64) - 400.0) * pix[keep, 2] / sigma,
                        (out[keep, 1].astype(np.float64) - 600.0) * pix[keep, 2] / sigma])
    assert abs(z.std() - 1) < 0.01 and abs(z.mean()) < 0.01


def test_noise_rejects_bad_arguments_before_any_cuda_call():
    L = _lib.lib()
    buf = ctypes.create_string_buffer(64)      # host memory: never dereferenced on the rejected paths
    p = ctypes.cast(buf, ctypes.c_void_p)
    nan, inf = float("nan"), float("inf")

    def call(batch=4, start=0, V=4, J=17, calib=p, sigma=2.0, po=0.1, pm=0.1, pix=p):
        return L.mpl_synth_detector_noise(1, start, batch, V, J, calib, sigma, po, pm, pix, None)

    bad = [dict(calib=None), dict(pix=None), dict(batch=-1), dict(start=-1), dict(V=0), dict(V=17), dict(J=0),
           dict(sigma=-0.5), dict(sigma=nan), dict(sigma=inf), dict(po=-0.1), dict(po=1.5), dict(po=nan), dict(pm=-0.1),
           dict(pm=1.5), dict(pm=nan), dict(po=0.6, pm=0.5), dict(batch=0, V=17), dict(batch=0, sigma=-1.0),
           dict(batch=0, po=0.7, pm=0.7)]
    for kw in bad:
        assert call(**kw) == _lib.MPL_ERR_INVALID_ARGUMENT, kw
        assert L.mpl_last_error().startswith(b"mpl_synth_detector_noise"), kw
    assert call(batch=0) == _lib.MPL_OK
    assert call(batch=0, po=0.5, pm=0.5) == _lib.MPL_OK                        # a sum of exactly 1 is allowed
    assert call(batch=0, calib=None, pix=None) == _lib.MPL_OK                  # an empty tensor has no storage
