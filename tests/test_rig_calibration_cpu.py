"""Calibration errors and rig calibration without a GPU: the numpy twin of mpl_synth_calib_noise (synth.calibration_noise),
the numpy restatement of mpl_calibrate_rig (tests/rig_calibration_oracle.py) against scipy.optimize.least_squares, and the
argument checks of evaluate.py's --calib-noise / --calibrate-rig."""
import numpy as np
import pytest
from scipy.optimize import least_squares
from scipy.spatial.transform import Rotation

from openmpl_b200 import evaluate, inputs, synth

import rig_calibration_oracle as oracle


def _rig(V, kind="h36m"):
    r = synth.make_rig(V, kind)
    return inputs.pack_calibration(r.R, r.t, r.f, r.c, r.image_size)


def test_zero_sigma_keeps_the_calibration_bit_for_bit():
    cal = synth.random_cameras(7, 5, seed=3)
    for sr, sp in ((0.0, 0.0), (0.0, 0.02), (0.01, 0.0)):
        out = synth.calibration_noise(cal, seed=1, start=11, sigma_rot=sr, sigma_pos=sp)
        np.testing.assert_array_equal(out[..., 12:].view(np.int64), cal[..., 12:].view(np.int64))
        if sr == 0:
            np.testing.assert_array_equal(out[..., :9].view(np.int64), cal[..., :9].view(np.int64))
        if sp == 0:
            np.testing.assert_array_equal(out[..., 9:12].view(np.int64), cal[..., 9:12].view(np.int64))


def test_rotations_stay_orthonormal():
    cal = synth.random_cameras(500, 4, seed=2)
    out = synth.calibration_noise(cal, seed=5, start=0, sigma_rot=0.3, sigma_pos=0.1)
    R = out[..., :9].reshape(-1, 3, 3)
    assert np.abs(R @ R.transpose(0, 2, 1) - np.eye(3)).max() < 1e-15 * 8
    assert np.abs(np.linalg.det(R) - 1.0).max() < 1e-14


def test_draws_have_the_stated_distribution():
    V, B = 4, 25_000                                             # 100 k draws per component
    cal = np.broadcast_to(_rig(V), (B, V, 18)).copy()
    sr, sp = np.radians(0.5), 0.02
    out = synth.calibration_noise(cal, seed=9, start=1000, sigma_rot=sr, sigma_pos=sp)
    R, R0 = out[..., :9].reshape(-1, 3, 3), cal[..., :9].reshape(-1, 3, 3)
    w = Rotation.from_matrix(R @ R0.transpose(0, 2, 1)).as_rotvec()          # R' = Exp(w) R
    dc = (out[..., 9:12] - cal[..., 9:12]).reshape(-1, 3)
    for x, s in ((w, sr), (dc, sp)):
        n = len(x)
        assert np.abs(x.mean(0)).max() < 5 * s / np.sqrt(n)
        assert np.abs(x.std(0) / s - 1.0).max() < 5 / np.sqrt(2 * n)
    assert np.abs(np.corrcoef(np.concatenate([w, dc], 1).T) - np.eye(6)).max() < 5 / np.sqrt(len(w))


def test_rows_depend_only_on_the_global_pose_index():
    cal = synth.random_cameras(40, 3, seed=4)
    full = synth.calibration_noise(cal, seed=2, start=100, sigma_rot=0.01, sigma_pos=0.03)
    for cut in (1, 17, 39):
        a = synth.calibration_noise(cal[:cut], seed=2, start=100, sigma_rot=0.01, sigma_pos=0.03)
        b = synth.calibration_noise(cal[cut:], seed=2, start=100 + cut, sigma_rot=0.01, sigma_pos=0.03)
        np.testing.assert_array_equal(np.concatenate([a, b]), full)
    rig = _rig(3)
    np.testing.assert_array_equal(synth.calibration_noise(rig, 2, 100, 0.01, 0.03),
                                  synth.calibration_noise(rig[None], 2, 100, 0.01, 0.03)[0])


def small_problem(V=3, B=4, J=5, seed=0, rot_deg=1.0, pos_mm=50.0, pixel_noise=0.5):
    """Pixels of B poses through a true rig, a perturbed rig and starting points near the truth."""
    true = _rig(V)
    rng = np.random.default_rng(seed)
    X = np.array([0.0, 0.25, 0.9]) + 0.3 * rng.standard_normal((B, J, 3))
    pix = np.empty((B, V, J, 3), dtype=np.float32)
    for v in range(V):
        R, c = true[v, :9].reshape(3, 3), true[v, 9:12]
        y = (X - c) @ R.T
        pix[:, v, :, 0] = true[v, 12] * y[..., 0] / y[..., 2] + true[v, 14] + pixel_noise * rng.standard_normal((B, J))
        pix[:, v, :, 1] = true[v, 13] * y[..., 1] / y[..., 2] + true[v, 15] + pixel_noise * rng.standard_normal((B, J))
    pix[..., 2] = rng.uniform(0.4, 1.0, (B, V, J))
    noisy = synth.calibration_noise(true, seed + 1, 0, np.radians(rot_deg), pos_mm / 1000.0)
    init = (X + 0.01 * rng.standard_normal(X.shape)).astype(np.float32)
    return pix, noisy, init, true


def test_oracle_agrees_with_scipy_least_squares():
    pix, noisy, init, _ = small_problem()
    sr, sp = np.radians(1.0), 0.05
    cal, pts, rep = oracle.calibrate_rig(pix, noisy, init, sigma_px=0.5, sigma_rot=sr, sigma_pos=sp, max_iters=100)
    assert rep[0] == 4 * 5 and rep[1] == 4 * 5 * 3 and rep[3] <= rep[2] and rep[5] < rep[4] and rep[7] >= 1
    assert rep[6] < 100                                          # converged by the step test
    used = oracle.select_items(pix, noisy, init)
    pb = oracle.Problem(pix, noisy, init, used, 0.5, sr, sp)
    ls = least_squares(pb.residuals, pb.start(), jac=pb.jacobian, method="trf", xtol=1e-15, ftol=1e-15, gtol=1e-15,
                       max_nfev=1000)
    ref = pb.calib_out(ls.x)
    Xs = pb.unpack(ls.x)[2]
    assert np.abs(cal[:, :9] - ref[:, :9]).max() < 1e-8
    assert np.abs(cal[:, 9:12] - ref[:, 9:12]).max() < 1e-8
    assert np.abs(pts.reshape(-1, 3).astype(np.float64) - Xs).max() < 1e-6          # points rounded to fp32
    assert abs(rep[3] - float(ls.fun @ ls.fun)) <= 1e-10 * rep[3]


def test_oracle_without_items_returns_its_inputs():
    pix, noisy, init, _ = small_problem()
    pix[:, 1:, :, 2] = 0.0                                       # one view left per joint
    cal, pts, rep = oracle.calibrate_rig(pix, noisy, init)
    np.testing.assert_array_equal(cal, noisy)
    np.testing.assert_array_equal(pts, init)
    assert not rep.any()


@pytest.mark.parametrize("argv,msg", [
    (["--calib-noise", "0.5"], "--calib-noise"),
    (["--calib-noise", "0.5,x"], "--calib-noise"),
    (["--calib-noise", "-1,10"], "--calib-noise"),
    (["--calib-noise", "nan,10"], "--calib-noise"),
    (["--calibrate-rig", "1024"], "--calibrate-rig"),
    (["--calib-noise", "0,10", "--calibrate-rig", "1024"], "--calibrate-rig"),
    (["--calib-noise", "0.5,10", "--calibrate-rig", "1024", "--random-cameras"], "--random-cameras"),
    (["--calib-noise", "0.5,10", "--calibrate-rig", "4096", "--micro-batch", "2048"], "--micro-batch"),
])
def test_evaluate_flag_checks(argv, msg, capsys):
    with pytest.raises(SystemExit) as e:
        evaluate.main(argv)
    assert e.value.code == 2
    assert msg in capsys.readouterr().err


def test_rig_errors_after_similarity_alignment():
    true = _rig(4)
    moved = true.copy()
    Q = Rotation.from_rotvec([0.01, -0.02, 0.015]).as_matrix()
    moved[:, 9:12] = 1.01 * true[:, 9:12] @ Q.T + np.array([0.03, -0.02, 0.01])   # c' = s Q c + t
    moved[:, :9] = (true[:, :9].reshape(-1, 3, 3) @ Q.T).reshape(-1, 9)              # R' = R Q^T: the same images
    ang, pos = evaluate.rig_errors(moved, true)
    assert min(ang) > 0.5 and min(pos) > 10
    ang, pos = evaluate.rig_errors(moved, true, align=True)
    assert max(ang) < 1e-10 and max(pos) < 1e-9


def test_oracle_jacobian_matches_finite_differences():
    """The oracle's analytic Jacobian (d y / d omega = -[y]x J_l(omega), the form the device uses too) against central
    differences of its residuals, at a point away from omega = 0 and on both sides of the Taylor switch of J_l."""
    pix, noisy, init, _ = small_problem()
    used = oracle.select_items(pix, noisy, init)
    pb = oracle.Problem(pix, noisy, init, used, 0.5, np.radians(1.0), 0.05)
    rng = np.random.default_rng(7)
    for om_scale in (0.02, 0.3):                                  # |omega|^2 below and above 1e-2
        x = pb.start()
        x[:6 * pb.V].reshape(pb.V, 6)[:, :3] += om_scale * rng.standard_normal((pb.V, 3)) / np.sqrt(3)
        x[6 * pb.V:] += 1e-3 * rng.standard_normal(x.size - 6 * pb.V)
        J = pb.jacobian(x)
        h = 1e-6
        Jn = np.empty_like(J)
        for k in range(x.size):
            e = np.zeros_like(x)
            e[k] = h
            Jn[:, k] = (pb.residuals(x + e) - pb.residuals(x - e)) / (2 * h)
        assert np.abs(J - Jn).max() <= 1e-6 * np.abs(J).max()
