"""Per-pose calibrations and the random camera generator without a GPU: the numpy twin of mpl_synth_cameras reduces to
make_rig at the centre of its ranges, gives proper rotations that see the room, stays in its stated focal range and depends
only on (seed, global pose index); the *_strided entry points and mpl_synth_cameras reject bad arguments before any CUDA
call; the Python wrappers reject a per-pose calibration whose batch does not match the pixels'."""
import ctypes

import numpy as np
import pytest
import torch

from openmpl_b200 import _lib, inputs, synth


@pytest.mark.parametrize("kind", ["h36m", "cmu"])
def test_centre_of_every_range_is_the_ring_rig(kind):
    f0, image_size, room = synth.rig_kind(kind)
    for V in range(1, 17):
        rig = synth.make_rig(V, kind)
        want = inputs.pack_calibration(rig.R, rig.t, rig.f, rig.c, rig.image_size)
        got = synth.cameras_from_uniforms(np.full((V, 6), 0.5), f0, image_size, room)
        assert np.abs(got - want).max() <= 1e-12, V


@pytest.mark.parametrize("kind,V", [("h36m", 4), ("cmu", 5), ("h36m", 16), ("cmu", 2)])
def test_random_cameras_are_proper_and_see_the_room_centre(kind, V):
    n = 10000
    f0, (w, h), room = synth.rig_kind(kind)
    cal = synth.random_cameras(n, V, kind, seed=7, start=1000)
    assert cal.shape == (n, V, 18) and cal.dtype == np.float64
    R = cal[..., :9].reshape(n, V, 3, 3)
    np.testing.assert_allclose(R @ np.swapaxes(R, -1, -2), np.broadcast_to(np.eye(3), R.shape), rtol=0, atol=1e-12)
    np.testing.assert_allclose(np.linalg.det(R), 1.0, rtol=0, atol=1e-12)
    centre = np.array([(room[0] + room[1]) / 2, (room[2] + room[3]) / 2, 0.9])
    xc = np.einsum("bvij,bvj->bvi", R, centre - cal[..., 9:12])
    assert (xc[..., 2] > 0).all()
    u = xc[..., 0] / xc[..., 2] * cal[..., 12] + cal[..., 14]
    v = xc[..., 1] / xc[..., 2] * cal[..., 13] + cal[..., 15]
    assert ((0 < u) & (u < w - 1) & (0 < v) & (v < h - 1)).all()
    f = cal[..., 12:14]
    assert (f >= 0.8 * f0).all() and (f <= 1.2 * f0).all() and (cal[..., 12] == cal[..., 13]).all()
    assert f.min() < 0.81 * f0 and f.max() > 1.19 * f0                  # the range is used, not just its centre
    np.testing.assert_array_equal(cal[..., 14:18], np.broadcast_to([w / 2, h / 2, w, h], (n, V, 4)))
    # horizontal distance from the room centre: 4.5 (0.75 .. 1.25) m, give or take the look-at shift (<= 0.36 m)
    d = np.hypot(*(cal[..., 9:11] - centre[:2]).transpose(2, 0, 1))
    assert (d > 4.5 * 0.75 - 0.4).all() and (d < 4.5 * 1.25 + 0.4).all()


def test_random_cameras_depend_only_on_seed_and_global_index():
    whole = synth.random_cameras(60, 5, "cmu", seed=3, start=20)
    for s, n in ((0, 1), (1, 12), (13, 40), (53, 7)):
        np.testing.assert_array_equal(synth.random_cameras(n, 5, "cmu", seed=3, start=20 + s), whole[s:s + n])
    assert not np.array_equal(synth.random_cameras(60, 5, "cmu", seed=4, start=20), whole)


def test_pack_calibration_takes_leading_batch_dimensions():
    cal = synth.random_cameras(6, 3, "h36m", seed=1)
    R, t, f, c = cal[..., :9].reshape(6, 3, 3, 3), cal[..., 9:12], cal[..., 12:14], cal[..., 14:16]
    np.testing.assert_array_equal(inputs.pack_calibration(R, t, f, c, (1000, 1000)), cal)
    for b in range(6):
        np.testing.assert_array_equal(inputs.pack_calibration(R[b], t[b], f[b], c[b], (1000, 1000)), cal[b])


def _host():
    buf = ctypes.create_string_buffer(64)      # host memory: never dereferenced on the rejected paths
    return buf, ctypes.cast(buf, ctypes.c_void_p)


def _calls(p):
    """name -> (call(batch, V, stride, **pointers) -> status, pointer argument names)"""
    L = _lib.lib()
    return {
        "mpl_build_inputs_strided": (
            lambda batch=4, V=4, stride=0, pix=p, calib=p, poses=p, rays=p, centers=p:
            L.mpl_build_inputs_strided(pix, calib, stride, batch, V, 17, poses, rays, centers, None),
            ("pix", "calib", "poses", "rays", "centers")),
        "mpl_synth_project_strided": (
            lambda batch=4, V=4, stride=0, calib=p, room=p, pix=p, target=p:
            L.mpl_synth_project_strided(1, 0, batch, V, 17, calib, stride, room, 0, pix, target, None),
            ("calib", "room", "pix", "target")),
        "mpl_synth_detector_noise_strided": (
            lambda batch=4, V=4, stride=0, calib=p, pix=p:
            L.mpl_synth_detector_noise_strided(1, 0, batch, V, 17, calib, stride, 2.0, 0.1, 0.1, pix, None),
            ("calib", "pix")),
        "mpl_triangulate_strided": (
            lambda batch=4, V=4, stride=0, pix=p, calib=p, points=p, used=p:
            L.mpl_triangulate_strided(pix, calib, stride, batch, V, 17, 0.0, points, used, None),
            ("pix", "calib", "points", "used")),
        "mpl_triangulate_robust_strided": (
            lambda batch=4, V=4, stride=0, pix=p, calib=p, points=p, inliers=p:
            L.mpl_triangulate_robust_strided(pix, calib, stride, batch, V, 17, 0.0, 10.0, points, inliers, None),
            ("pix", "calib", "points", "inliers")),
    }


@pytest.mark.parametrize("name", ["mpl_build_inputs_strided", "mpl_synth_project_strided", "mpl_synth_detector_noise_strided",
                                  "mpl_triangulate_strided", "mpl_triangulate_robust_strided"])
def test_strided_entry_points_reject_bad_arguments_before_any_cuda_call(name):
    buf, p = _host()
    call, ptrs = _calls(p)[name]
    L = _lib.lib()
    bad = [dict(stride=-1), dict(stride=-72), dict(stride=1), dict(stride=17), dict(stride=18 * 4 - 1), dict(V=5, stride=72),
           dict(batch=0, stride=-1), dict(batch=0, stride=5), dict(batch=-1, stride=72)]
    bad += [{k: None} for k in ptrs] + [{k: None, "stride": 72} for k in ptrs]
    for kw in bad:
        assert call(**kw) == _lib.MPL_ERR_INVALID_ARGUMENT, kw
        assert L.mpl_last_error().startswith(name.encode()), (kw, L.mpl_last_error())
    for stride in (0, 72, 73, 1000):
        assert call(batch=0, stride=stride) == _lib.MPL_OK
    assert call(batch=0, stride=72, **{k: None for k in ptrs}) == _lib.MPL_OK   # an empty batch touches nothing


def test_synth_cameras_rejects_bad_arguments_before_any_cuda_call():
    buf, p = _host()
    L = _lib.lib()
    nan, inf = float("nan"), float("inf")

    def call(batch=4, start=0, V=4, f0=1145.0, w=1000.0, h=1000.0, room=p, out=p):
        return L.mpl_synth_cameras(1, start, batch, V, f0, w, h, room, out, None)

    bad = [dict(batch=-1), dict(start=-1), dict(V=0), dict(V=17), dict(f0=0.0), dict(f0=-1.0), dict(f0=nan), dict(f0=inf),
           dict(w=1.0), dict(w=nan), dict(h=0.5), dict(h=inf), dict(room=None), dict(out=None), dict(batch=0, V=0)]
    for kw in bad:
        assert call(**kw) == _lib.MPL_ERR_INVALID_ARGUMENT, kw
        assert L.mpl_last_error().startswith(b"mpl_synth_cameras"), kw
    assert call(batch=0) == _lib.MPL_OK
    assert call(batch=0, room=None, out=None) == _lib.MPL_OK


def test_wrappers_reject_a_per_pose_calibration_of_another_batch():
    B, V, J = 6, 4, 17
    pix = torch.zeros((B, V, J, 3), dtype=torch.float32)
    rig = synth.make_rig(V, "h36m")
    for bad in (synth.random_cameras(B - 1, V), synth.random_cameras(B + 1, V), synth.random_cameras(B, V + 1),
                np.zeros((B, V, 17))):
        with pytest.raises(ValueError):
            inputs.build_inputs(pix, bad)
        with pytest.raises(ValueError):
            inputs.triangulate(pix, bad)
        with pytest.raises(ValueError):
            inputs.triangulate_robust(pix, bad)
        with pytest.raises(ValueError):
            inputs.add_detector_noise(pix, bad, 1, 0, 2.0, 0.1, 0.0)
        with pytest.raises(ValueError):
            inputs.synth_project(B, rig, device="cpu", cameras=bad)
    with pytest.raises(ValueError):
        inputs.synth_project(B, rig, device="cpu", cameras=inputs.pack_calibration(rig.R, rig.t, rig.f, rig.c, rig.image_size))
