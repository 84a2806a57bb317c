"""mpl_synth_detector_noise on the device: it draws the numpy twin's uniforms (miss / outlier decisions and outlier
confidences exactly, pixels to 1e-3 px), does not depend on how the batch is split, and is the identity at zero noise."""
import numpy as np
import pytest
import torch

from openmpl_b200 import inputs, synth

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("kind,V", [("h36m", 4), ("cmu", 5)])
def test_device_noise_matches_the_numpy_twin(kind, V):
    rig = synth.make_rig(V, kind)
    pix, _, calib = inputs.synth_project(3000, rig, seed=6, start=1000)
    raw = pix.cpu().numpy()
    inputs.add_detector_noise(pix, calib, 9, 1000, 2.0, 0.15, 0.05)
    got = pix.cpu().numpy()
    want = synth.detector_noise(raw, rig.image_size, 9, 1000, 2.0, 0.15, 0.05)
    np.testing.assert_array_equal(got[..., 2], want[..., 2])          # miss and outlier decisions, outlier confidences
    outlier = (want[..., 2] != raw[..., 2]) & (want[..., 2] != 0)
    assert outlier.mean() > 0.1
    np.testing.assert_array_equal(got[outlier], want[outlier])       # a uniform point of the image, exact arithmetic
    assert np.abs(got[..., :2].astype(np.float64) - want[..., :2]).max() <= 1e-3


def test_batch_split_and_start_are_bitwise_invariant_and_zero_noise_is_identity():
    rig = synth.make_rig(4, "h36m")
    pix, _, calib = inputs.synth_project(5000, rig, seed=2)
    clean = pix.clone()
    inputs.add_detector_noise(pix, calib, 1, 0, 0.0, 0.0, 0.0)
    assert torch.equal(pix.view(torch.int32), clean.view(torch.int32))
    whole = inputs.add_detector_noise(clean.clone(), calib, 4, 0, 2.0, 0.1, 0.1)
    for s, n in ((0, 1), (1, 4097), (4098, 902)):
        part = inputs.add_detector_noise(clean[s:s + n].clone(), calib, 4, s, 2.0, 0.1, 0.1)
        assert torch.equal(part.view(torch.int32), whole[s:s + n].view(torch.int32))
    shifted, _, _ = inputs.synth_project(1000, rig, seed=2, start=3000)
    inputs.add_detector_noise(shifted, calib, 4, 3000, 2.0, 0.1, 0.1)
    assert torch.equal(shifted.view(torch.int32), whole[3000:4000].view(torch.int32))
    empty = torch.empty((0, 4, 17, 3), device="cuda")
    assert inputs.add_detector_noise(empty, calib, 4, 0, 2.0, 0.1, 0.1).shape == (0, 4, 17, 3)
