"""mpl_calibrate_rig on the device: it matches the numpy oracle (tests/rig_calibration_oracle.py) at 2 to 16 views, with and
without a view mask; recovers a perturbed rig from exact pixels up to the similarity gauge; leaves an exact rig where it is;
returns init bit for bit where a pair is not an item; is bitwise reproducible, also under CUDA-graph replay; checks its
arguments; and the evaluation's --calib-noise / --calibrate-rig paths behave as documented."""
import math

import numpy as np
import pytest
import torch

from openmpl_b200 import _lib, evaluate, inputs, synth

import rig_calibration_oracle as oracle

pytestmark = pytest.mark.gpu


def _rig(V, kind="h36m"):
    r = synth.make_rig(V, kind)
    return inputs.pack_calibration(r.R, r.t, r.f, r.c, r.image_size)


def _problem(V, J, B, seed, pixel_noise=0.5, rot_deg=0.5, pos_mm=20.0, conf_ones=False):
    """Detections of B poses of J joints through the true rig, a perturbed rig, and init = the triangulation under it."""
    true = _rig(V)
    rng = np.random.default_rng(seed)
    X = np.array([0.0, 0.25, 0.9]) + 0.4 * rng.standard_normal((B, J, 3))
    pix = np.empty((B, V, J, 3), dtype=np.float32)
    for v in range(V):
        R, c = true[v, :9].reshape(3, 3), true[v, 9:12]
        y = (X - c) @ R.T
        for k in range(2):
            pix[:, v, :, k] = (true[v, 12 + k] * y[..., k] / y[..., 2] + true[v, 14 + k]
                               + pixel_noise * rng.standard_normal((B, J)))
    pix[..., 2] = 1.0 if conf_ones else np.where(rng.random((B, V, J)) < 0.1, 0.0, rng.uniform(0.4, 1.0, (B, V, J)))
    noisy = synth.calibration_noise(true, seed + 1, 0, math.radians(rot_deg), pos_mm / 1000.0) if rot_deg or pos_mm else true
    init = inputs.triangulate(torch.from_numpy(pix).cuda(), noisy)[0].cpu().numpy()
    return pix, noisy, init, true, X


def _run(pix, calib, init, mask=None, **kw):
    cal, pts, rep = inputs.calibrate_rig(torch.from_numpy(pix).cuda(), calib, torch.from_numpy(init).cuda(),
                                         None if mask is None else torch.from_numpy(mask).cuda(), **kw)
    return cal.cpu().numpy(), pts.cpu().numpy(), rep.cpu().numpy()


@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("J", [1, 17])
@pytest.mark.parametrize("V", [2, 4, 8, 16])
def test_matches_the_oracle(V, J, masked):
    B = 48 if J == 1 else 5
    pix, noisy, init, _, _ = _problem(V, J, B, seed=10 * V + J)
    init[0, 0] = np.nan                                          # never an item
    mask = None
    if masked:
        mask = np.random.default_rng(V + J).integers(0, 1 << V, (B, J)).astype(np.int32)
        mask[mask == 0] = (1 << V) - 1
    kw = dict(sigma_px=0.5, sigma_rot=math.radians(0.5), sigma_pos=0.02, max_iters=40)
    cal, pts, rep = _run(pix, noisy, init, mask, **kw)
    ocal, opts, orep = oracle.calibrate_rig(pix, noisy, init, mask, **kw)
    dr, dc = np.abs(cal[:, :9] - ocal[:, :9]).max(), np.abs(cal[:, 9:12] - ocal[:, 9:12]).max()
    items = oracle.select_items(pix, noisy, init, mask) != 0
    dp = np.abs(pts - opts)[items].max()
    print(f"V={V} J={J} masked={masked}: items {int(rep[0])} obs {int(rep[1])} iters {int(rep[6])}/{int(orep[6])} "
          f"accepted {int(rep[7])}/{int(orep[7])} rms {rep[4]:.4f} -> {rep[5]:.4f} px; |dR| {dr:.2e} |dc| {dc:.2e} m "
          f"|dX| {dp:.2e} m")
    np.testing.assert_array_equal(rep[:2], orep[:2])
    # both stop once a camera step is <= 1e-10 (|c|_2 + 1e-10); where rounding makes them accept or reject a different
    # step, they stop at different points of that size around the minimum (measured: up to 2.6e-9 m at |c|_2 = 13 m)
    tol = 4e-10 * (np.linalg.norm(noisy[:, 9:12]) + 1e-10)
    assert dr <= tol and dc <= tol
    # points: fp32 rounding, plus the shift a camera difference of that size causes in a weakly constrained point (measured:
    # 6e-8 m for 2.6e-9 m of camera difference, masked V = 8)
    ptol = 2 * np.spacing(np.abs(opts[items])) + 50 * max(dr, dc)
    assert (np.abs(pts - opts)[items] <= ptol).all()
    np.testing.assert_array_equal(pts[~items].view(np.int32), init[~items].view(np.int32))
    np.testing.assert_array_equal(cal[:, 12:].view(np.int64), noisy[:, 12:].view(np.int64))
    assert rep[3] <= rep[2] and rep[5] < rep[4]
    assert abs(rep[3] - orep[3]) <= 1e-9 * orep[3] and abs(rep[2] - orep[2]) <= 1e-12 * orep[2]


def _umeyama(src, dst):
    """s, Q, t with dst ~ s Q src + t (least squares)."""
    ms, md = src.mean(0), dst.mean(0)
    a, b = src - ms, dst - md
    U, S, Vt = np.linalg.svd(b.T @ a)
    D = np.diag([1.0, 1.0, np.sign(np.linalg.det(U @ Vt))])
    Q = U @ D @ Vt
    s = np.trace(np.diag(S) @ D) / (a * a).sum()
    return s, Q, md - s * Q @ ms


def test_recovers_a_perturbed_rig_from_exact_pixels():
    V = 4
    pix, noisy, init, true, _ = _problem(V, 17, 2048, seed=3, pixel_noise=0.0, rot_deg=1.0, pos_mm=50.0, conf_ones=True)
    cal, _, rep = _run(pix, noisy, init, sigma_px=1.0, sigma_rot=math.radians(1.0), sigma_pos=0.05)
    s, Q, t = _umeyama(true[:, 9:12], cal[:, 9:12])
    c_back = (cal[:, 9:12] - t) @ Q / s                           # the calibrated centres in the true frame
    R_back = cal[:, :9].reshape(V, 3, 3) @ Q                      # R_est = R_true Q^T in the aligned frame
    ang = np.degrees([np.arccos(np.clip((np.trace(R_back[v] @ true[v, :9].reshape(3, 3).T) - 1) / 2, -1, 1))
                      for v in range(V)])
    pos = 1000 * np.linalg.norm(c_back - true[:, 9:12], axis=1)
    print(f"rms {rep[4]:.3f} -> {rep[5]:.2e} px in {int(rep[6])} iterations ({int(rep[7])} accepted); after a similarity "
          f"alignment (scale {s:.6f}): rotation {ang.max():.2e} deg, centre {pos.max():.2e} mm")
    assert rep[5] < 0.01
    assert ang.max() < 0.01 and pos.max() < 1.0


def test_exact_rig_stays_put():
    pix, cal0, init, true, _ = _problem(4, 17, 256, seed=4, pixel_noise=0.0, rot_deg=0.0, pos_mm=0.0)
    cal, _, rep = _run(pix, cal0, init)
    dr, dc = np.abs(cal[:, :9] - true[:, :9]).max(), np.abs(cal[:, 9:12] - true[:, 9:12]).max()
    print(f"exact start: |dR| {dr:.2e}, |dc| {dc:.2e} m, rms {rep[4]:.2e} -> {rep[5]:.2e} px")
    assert dr < 1e-7 and dc < 1e-6 and rep[3] <= rep[2]


def test_no_item_returns_the_inputs():
    pix, noisy, init, _, _ = _problem(3, 17, 8, seed=5)
    pix[:, 1:, :, 2] = 0.0
    cal, pts, rep = _run(pix, noisy, init)
    np.testing.assert_array_equal(cal.view(np.int64), noisy.view(np.int64))
    np.testing.assert_array_equal(pts.view(np.int32), init.view(np.int32))
    assert not rep.any()


def test_bitwise_reproducible_and_graph_replay():
    pix, noisy, init, _, _ = _problem(8, 17, 300, seed=6)
    p, i = torch.from_numpy(pix).cuda(), torch.from_numpy(init).cuda()
    a = inputs.calibrate_rig(p, noisy, i)
    b = inputs.calibrate_rig(p, noisy, i)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    L = _lib.lib()
    B, V, J = 300, 8, 17
    nb = L.mpl_calibrate_rig_workspace_bytes(B, V, J)
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    cal = torch.as_tensor(noisy).cuda()
    out = torch.empty_like(cal)
    pts = torch.empty_like(i)
    rep = torch.empty(8, dtype=torch.float64, device="cuda")
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        L.mpl_calibrate_rig(p.data_ptr(), cal.data_ptr(), B, V, J, 0.0, None, i.data_ptr(), 1.0, math.radians(1.0), 0.05, 30,
                            out.data_ptr(), pts.data_ptr(), rep.data_ptr(), ws.data_ptr(), nb, s.cuda_stream)   # warm up
        s.synchronize()
        with torch.cuda.graph(g, stream=s):
            _lib.check(L.mpl_calibrate_rig(p.data_ptr(), cal.data_ptr(), B, V, J, 0.0, None, i.data_ptr(), 1.0,
                                           math.radians(1.0), 0.05, 30, out.data_ptr(), pts.data_ptr(), rep.data_ptr(),
                                           ws.data_ptr(), nb, s.cuda_stream))
    out.zero_(); pts.zero_(); rep.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, a[0]) and torch.equal(pts, a[1]) and torch.equal(rep, a[2])


def test_argument_checks():
    L = _lib.lib()
    B, V, J = 4, 3, 5
    pix = torch.zeros((B, V, J, 3), device="cuda")
    cal = torch.as_tensor(_rig(V)).cuda()
    init = torch.zeros((B, J, 3), device="cuda")
    out = torch.empty_like(cal)
    rep = torch.empty(8, dtype=torch.float64, device="cuda")
    nb = L.mpl_calibrate_rig_workspace_bytes(B, V, J)
    assert nb > 0
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    base = dict(pix=pix.data_ptr(), calib=cal.data_ptr(), batch=B, V=V, J=J, min_conf=0.0, mask=None, init=init.data_ptr(),
                spx=1.0, srot=0.01, spos=0.05, iters=10, out=out.data_ptr(), pts=None, rep=rep.data_ptr(),
                ws=ws.data_ptr(), nb=nb)

    def call(**kw):
        a = dict(base, **kw)
        return L.mpl_calibrate_rig(*a.values(), None)

    inf, nan = float("inf"), float("nan")
    for kw in (dict(V=1), dict(V=17), dict(J=0), dict(batch=0), dict(spx=0.0), dict(srot=-1.0), dict(spos=inf),
               dict(spx=nan), dict(iters=0), dict(iters=101), dict(pix=None), dict(calib=None), dict(init=None),
               dict(out=None), dict(rep=None), dict(ws=None)):
        assert call(**kw) == _lib.MPL_ERR_INVALID_ARGUMENT, kw
    assert call(nb=nb - 1) == _lib.MPL_ERR_WORKSPACE
    assert call() == _lib.MPL_OK
    torch.cuda.synchronize()
    assert L.mpl_calibrate_rig_workspace_bytes(B, 1, J) == 0


def _metrics(line):
    return line["mpjpe_cm"], line["triangulation"]["mpjpe_cm"]


def test_evaluate_calib_noise_zero_is_the_plain_line():
    kw = dict(arch="hm0", views=4, depth=2, poses=8192, micro_batch=4096, precision="fp32", triangulate=True, pixel_noise=1.0)
    plain = evaluate.run(**kw)
    zero = evaluate.run(**kw, calib_noise=(0.0, 0.0))
    # the calibration is bitwise the rig (test_calib_noise_gpu.py), so every kernel sees the same inputs; the fp64 atomics of
    # the metric accumulators make the last bits of a sum vary from run to run of the same command
    for a, b in zip(_metrics(plain), _metrics(zero)):
        for k, v in a.items():
            if isinstance(v, float):
                assert v == pytest.approx(b[k], rel=1e-12, abs=0), k
    assert zero["data"]["calibration_noise"]["rotation_deg"] == 0.0


def test_evaluate_calibrate_rig():
    kw = dict(arch="hm0", views=4, depth=2, poses=8192, micro_batch=4096, precision="fp32", triangulate=True, pixel_noise=1.0)
    noisy = evaluate.run(**kw, calib_noise=(0.5, 20.0))
    line = evaluate.run(**kw, calib_noise=(0.5, 20.0), calibrate_rig=1024)
    rc = line["rig_calibration"]
    print({k: rc[k] for k in ("items", "iterations", "accepted_steps", "rms_px", "rotation_error_deg", "centre_error_mm",
                              "after_similarity_alignment", "ms")})
    assert rc["poses"] == 1024 and rc["items"] > 0.9 * 1024 * 17
    assert rc["rms_px"]["after"] < rc["rms_px"]["before"]
    for errs in (rc, rc["after_similarity_alignment"]):
        for key in ("rotation_error_deg", "centre_error_mm"):
            assert all(c < n for c, n in zip(errs[key]["calibrated"], errs[key]["noisy"])), (key, errs[key])
    print("triangulation MPJPE cm: noisy", noisy["triangulation"]["mpjpe_cm"]["absolute"], "calibrated",
          line["triangulation"]["mpjpe_cm"]["absolute"])
    assert line["triangulation"]["mpjpe_cm"]["absolute"] < noisy["triangulation"]["mpjpe_cm"]["absolute"]
