"""mpl_synth_calib_noise on the device: it matches the numpy twin (synth.calibration_noise) per pose and for a fixed rig, keeps
the intrinsics (and a field whose sigma is 0) bit for bit, works in place, and checks its arguments."""
import ctypes

import numpy as np
import pytest
import torch

from openmpl_b200 import _lib, inputs, synth

pytestmark = pytest.mark.gpu


def _check(got, want, sigma_pos):
    np.testing.assert_array_equal(got[..., 12:].view(np.int64), want[..., 12:].view(np.int64))
    # R: entries <= 1, a few roundings of the Rodrigues and product sums apart; t: the trig of Box-Muller within 1 ulp
    assert np.abs(got[..., :9] - want[..., :9]).max() <= 8e-16
    tol = 2 * np.spacing(np.abs(want[..., 9:12])) + 4e-16 * 6 * sigma_pos
    assert (np.abs(got[..., 9:12] - want[..., 9:12]) <= tol).all()


@pytest.mark.parametrize("V", [1, 4, 16])
def test_per_pose_matches_the_twin(V):
    cal = synth.random_cameras(1000, V, seed=V)
    sr, sp = np.radians(0.7), 0.03
    got = inputs.calibration_noise(torch.from_numpy(cal).cuda(), seed=5, start=37, sigma_rot=sr, sigma_pos=sp).cpu().numpy()
    _check(got, synth.calibration_noise(cal, 5, 37, sr, sp), sp)


@pytest.mark.parametrize("V", [2, 5])
def test_rig_matches_the_twin(V):
    r = synth.make_rig(V, "cmu")
    rig = inputs.pack_calibration(r.R, r.t, r.f, r.c, r.image_size)
    got = inputs.calibration_noise(rig, seed=1, start=0, sigma_rot=0.02, sigma_pos=0.05, device="cuda").cpu().numpy()
    assert got.shape == (V, 18)
    _check(got, synth.calibration_noise(rig, 1, 0, 0.02, 0.05), 0.05)


def test_zero_sigmas_and_in_place():
    cal = torch.from_numpy(synth.random_cameras(300, 4, seed=1)).cuda()
    for sr, sp in ((0.0, 0.0), (0.0, 0.1), (0.1, 0.0)):
        out = inputs.calibration_noise(cal, 3, 0, sr, sp)
        if sr == 0:
            assert torch.equal(out[..., :9].view(torch.int64), cal[..., :9].view(torch.int64))
        if sp == 0:
            assert torch.equal(out[..., 9:12].view(torch.int64), cal[..., 9:12].view(torch.int64))
        assert torch.equal(out[..., 12:].view(torch.int64), cal[..., 12:].view(torch.int64))
    ref = inputs.calibration_noise(cal, 3, 0, 0.01, 0.02)
    buf = cal.clone()
    L = _lib.lib()
    _lib.check(L.mpl_synth_calib_noise(3, 0, 300, 4, buf.data_ptr(), 72, 0.01, 0.02, buf.data_ptr(), None))
    torch.cuda.synchronize()
    assert torch.equal(buf, ref)


def test_argument_checks():
    L = _lib.lib()
    cal = torch.from_numpy(synth.random_cameras(4, 3, seed=1)).cuda()
    out = torch.empty_like(cal)
    p, o = cal.data_ptr(), out.data_ptr()
    bad = [(0, 0, 4, 0, p, 0, 0.1, 0.1, o), (0, 0, 4, 17, p, 0, 0.1, 0.1, o), (0, -1, 4, 3, p, 0, 0.1, 0.1, o),
           (0, 0, 4, 3, p, 0, -0.1, 0.1, o), (0, 0, 4, 3, p, 0, 0.1, float("inf"), o), (0, 0, 4, 3, p, 0, float("nan"), 0.1, o),
           (0, 0, 4, 3, p, 53, 0.1, 0.1, o), (0, 0, -1, 3, p, 0, 0.1, 0.1, o), (0, 0, 4, 3, None, 0, 0.1, 0.1, o),
           (0, 0, 4, 3, p, 54, 0.1, 0.1, None), (0, 0, 4, 3, p, 0, 0.1, 0.1, p), (0, 0, 4, 3, p, 108, 0.1, 0.1, p)]
    for args in bad:
        assert L.mpl_synth_calib_noise(*args, None) == _lib.MPL_ERR_INVALID_ARGUMENT, args
    assert L.mpl_synth_calib_noise(0, 0, 0, 3, None, 0, 0.1, 0.1, None, None) == _lib.MPL_OK
    assert L.mpl_synth_calib_noise(0, 0, 4, 3, p, 54, 0.1, 0.1, p, None) == _lib.MPL_OK
    torch.cuda.synchronize()
