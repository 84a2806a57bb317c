"""mpl_distort_pixels / mpl_undistort_pixels on the device: they match the numpy twin (synth.distort_pixels) and the oracle
(tests/lens_oracle.py) at every view count, joint count, rig and stride combination up to a million poses, and make the
same validity decisions on lenses that fold inside the tested range; zero coefficients
copy, in place equals out of place, batch splits and CUDA-graph replay are bitwise invariant; distorted exact pixels
undistorted for the three triangulations recover the 3D poses; and the evaluation's --lens-distortion path is the
step-by-step pipeline."""
import ctypes

import numpy as np
import pytest
import torch

from openmpl_b200 import _lib, evaluate, inputs, metric, synth

from lens_oracle import undistort_pixels as oracle_undistort

pytestmark = pytest.mark.gpu

LENS = {"h36m": (-0.207, 0.248, -0.0009, -0.0016, -0.0031), "cmu": (-0.30, 0.10, 0.001, -0.001, 0.0)}
# lenses whose validity rule fails inside the range tested: a strong barrel folding at r^2 = 0.76 (k3 = 0: the critical point
# of g is -3 k1 / (10 k2)), and one whose g dips below 0 on (0.5, 1.3) and rises again (k3 != 0: the roots of the quadratic
# g'), so points beyond r^2 = 1.3 fail on the interior critical point alone, with g(r^2) > 0
FOLDS = {"fold": (-0.5, 0.05, 0.001, -0.001, 0.0), "unfold": (-0.9, 0.3, 0.0005, -0.0005, 0.01)}


def _bits(t):
    return t.contiguous().view(torch.int32)


def _case(kind, B, V, J, per_pose_calib, per_pose_dist, seed=0, lens=None, spread=0.08):
    """Random pixels around the frame, up to `spread` of its size outside it (some conf 0), a calibration and a lens (that of
    the rig kind, or `lens`): shared or per pose."""
    rng = np.random.default_rng(seed)
    rig = synth.make_rig(V, kind)
    w, h = rig.image_size
    pix = np.empty((B, V, J, 3), dtype=np.float32)
    pix[..., 0] = rng.uniform(-spread * w, (1 + spread) * w, (B, V, J))
    pix[..., 1] = rng.uniform(-spread * h, (1 + spread) * h, (B, V, J))
    pix[..., 2] = np.where(rng.random((B, V, J)) < 0.1, 0.0, rng.uniform(0.3, 1.0, (B, V, J)))
    if per_pose_calib:
        calib = synth.random_cameras(B, V, kind, seed=seed + 1)
    else:
        calib = inputs.pack_calibration(rig.R, rig.t, rig.f, rig.c, rig.image_size)
    k = np.array(LENS[kind] if lens is None else lens)
    dist = np.tile(k, (V, 1))
    if per_pose_dist:
        dist = k * (1.0 + 0.3 * (rng.random((B, V, 5)) - 0.5))
    return pix, calib, dist, rig


def _check_distortion(got, want):
    np.testing.assert_array_equal(got[..., 2], want[..., 2])
    tol = np.maximum(1e-4, np.spacing(np.abs(want[..., :2])).astype(np.float64))
    assert (np.abs(got[..., :2].astype(np.float64) - want[..., :2]) <= tol).all()


def _check_undistortion(got, want, exact):
    np.testing.assert_array_equal(got[..., 2], want[..., 2])                     # conf and validity decisions
    np.testing.assert_array_equal(np.isnan(got[..., :2]), np.isnan(want[..., :2]))
    fin = np.isfinite(exact)
    tol = np.maximum(1e-4, np.spacing(np.abs(want[..., :2])).astype(np.float64))
    assert (np.abs(got[..., :2].astype(np.float64)[fin] - exact[fin]) <= tol[fin]).all()


VJ = [(1, 17), (2, 1), (4, 40), (5, 17), (8, 1), (16, 40)]


@pytest.mark.parametrize("per_pose_calib,per_pose_dist", [(False, False), (True, False), (False, True), (True, True)])
@pytest.mark.parametrize("kind", ["h36m", "cmu"])
@pytest.mark.parametrize("V,J", VJ)
def test_device_matches_the_numpy_twin_and_oracle(V, J, kind, per_pose_calib, per_pose_dist):
    pix, calib, dist, rig = _case(kind, 257, V, J, per_pose_calib, per_pose_dist, seed=V * 100 + J)
    dev = torch.from_numpy(pix).cuda()
    d = inputs.distort_pixels(dev.clone(), calib, dist).cpu().numpy()
    _check_distortion(d, synth.distort_pixels(pix, calib, dist))
    w, h = rig.image_size
    got, calib_u = inputs.undistort_pixels(torch.from_numpy(d).cuda(), calib, dist, margin=(w / 2, h / 2))
    want, exact = oracle_undistort(d, calib, dist, w / 2, h / 2)
    inside = (d[..., 2] != 0) & (d[..., 0] > 0) & (d[..., 0] < w - 1) & (d[..., 1] > 0) & (d[..., 1] < h - 1)
    assert (want[..., 2][inside] != 0).mean() > 0.95                                # candidates undistort
    _check_undistortion(got.cpu().numpy(), want, exact)
    shifted = np.array(calib, dtype=np.float64, copy=True)
    shifted[..., 14:18] += [w / 2, h / 2, w, h]
    np.testing.assert_array_equal(calib_u.cpu().numpy(), shifted)


@pytest.mark.parametrize("per_pose_calib,per_pose_dist", [(False, False), (True, False), (False, True), (True, True)])
@pytest.mark.parametrize("lens", sorted(FOLDS))
@pytest.mark.parametrize("V,J", [(1, 17), (4, 40), (16, 17)])
def test_device_decides_folds_like_the_numpy_twin_and_oracle(V, J, lens, per_pose_calib, per_pose_dist):
    # ideal pixels far beyond the frame: many lie past the fold, and the distortion must give them conf 0
    pix, calib, dist, rig = _case("h36m", 512, V, J, per_pose_calib, per_pose_dist, seed=V * 10 + J, lens=FOLDS[lens],
                                  spread=0.6)
    d = inputs.distort_pixels(torch.from_numpy(pix).cuda(), calib, dist).cpu().numpy()
    want = synth.distort_pixels(pix, calib, dist)
    _check_distortion(d, want)
    folded = (pix[..., 2] != 0) & (want[..., 2] == 0)
    assert folded.sum() >= 0.05 * (pix[..., 2] != 0).sum(), folded.sum()
    np.testing.assert_array_equal(d[folded][:, :2], pix[folded][:, :2])             # pixel kept
    c = calib[..., None, :] if calib.ndim == 3 else calib[None, :, None, :]
    kk = dist[..., None, :] if dist.ndim == 3 else dist[None, :, None, :]
    k = tuple(kk[..., m] for m in range(5))
    x = (pix[..., 0].astype(np.float64) - c[..., 14]) / c[..., 12]
    y = (pix[..., 1].astype(np.float64) - c[..., 15]) / c[..., 13]
    _, _, a, b, dd = synth.lens_map(k, x, y)
    r2 = x * x + y * y
    g = 1.0 + r2 * (3.0 * k[0] + r2 * (5.0 * k[1] + r2 * (7.0 * k[4])))
    interior_only = folded & (a * dd - b * b > 0) & (g > 0)                       # rejected by a root of g' inside (0, r^2)
    assert interior_only.sum() >= (10 if lens == "unfold" else 0), interior_only.sum()
    # detections around the frame: those in its corners lie beyond the fold's image and have no valid preimage
    det, _, _, _ = _case("h36m", 512, V, J, per_pose_calib, per_pose_dist, seed=V * 10 + J + 1, lens=FOLDS[lens])
    w, h = rig.image_size
    got, _ = inputs.undistort_pixels(torch.from_numpy(det).cuda(), calib, dist, margin=(w / 2, h / 2))
    want_u, exact = oracle_undistort(det, calib, dist, w / 2, h / 2)
    failed = np.isnan(want_u[..., 0])
    assert failed.sum() >= 10, failed.sum()
    assert (want_u[failed][:, 2] == 0).all()
    _check_undistortion(got.cpu().numpy(), want_u, exact)


def test_a_million_poses_with_per_pose_cameras():
    B, V, J = 1 << 20, 2, 17
    rig = synth.make_rig(V, "h36m")
    cams = inputs.synth_cameras(B, V, "h36m", seed=3)
    pix, _, calib = inputs.synth_project(B, rig, seed=3, cameras=cams)
    ideal = pix.clone()
    dist = np.tile(LENS["h36m"], (V, 1))
    inputs.distort_pixels(pix, calib, dist)
    und, _ = inputs.undistort_pixels(pix, calib, dist, margin=(500.0, 500.0))
    torch.cuda.synchronize()
    sel = torch.from_numpy(np.concatenate([np.arange(0, B, 61), np.arange(B - 3000, B)])).cuda()  # spread, and the end
    c = calib[sel].cpu().numpy()
    raw, d = ideal[sel].cpu().numpy(), pix[sel].cpu().numpy()
    _check_distortion(d, synth.distort_pixels(raw, c, dist))
    want, exact = oracle_undistort(d, c, dist, 500.0, 500.0)
    _check_undistortion(und[sel].cpu().numpy(), want, exact)


def _undistort_c(pin, pout, calib, cstride, dist, dstride, mx, my):
    B, V, J, _ = pin.shape
    _lib.check(_lib.lib().mpl_undistort_pixels_strided(pin.data_ptr(), pout.data_ptr(), calib.data_ptr(), cstride,
                                                       dist.data_ptr(), dstride, mx, my, B, V, J,
                                                       torch.cuda.current_stream().cuda_stream))


def _distort_c(pin, pout, calib, cstride, dist, dstride):
    B, V, J, _ = pin.shape
    _lib.check(_lib.lib().mpl_distort_pixels_strided(pin.data_ptr(), pout.data_ptr(), calib.data_ptr(), cstride,
                                                     dist.data_ptr(), dstride, B, V, J, torch.cuda.current_stream().cuda_stream))


def test_bitwise_invariants():
    pix, calib, dist, rig = _case("cmu", 5000, 4, 17, True, True, seed=5)
    w, h = rig.image_size
    pix_t = torch.from_numpy(pix).cuda()
    cal = torch.from_numpy(calib).cuda()
    dst = torch.from_numpy(dist).cuda()
    # zero coefficients (and zero margins): u, v copied; conf too except outside the frame
    zero = torch.zeros_like(dst)
    assert torch.equal(_bits(inputs.distort_pixels(pix_t.clone(), cal, zero)), _bits(pix_t))
    odd = pix_t.clone()
    odd[::7, :, 3, 0] = -0.0                                                         # -0 and non-finite pixels, conf > 0
    odd[::11, 1, :, 1] = float("nan")
    odd[::13, 2, 5, 0] = float("inf")
    odd[..., 2] = 0.5
    assert torch.equal(_bits(inputs.distort_pixels(odd.clone(), cal, zero)), _bits(odd))
    mixed = zero.clone()
    mixed[:, 0] = dst[:, 0]                                                          # a lens on view 0 only
    out = inputs.distort_pixels(odd.clone(), cal, mixed)
    assert torch.equal(_bits(out[:, 1:]), _bits(odd[:, 1:]))
    und, cal_u = inputs.undistort_pixels(pix_t, cal, zero, margin=0.0)
    assert torch.equal(_bits(und[..., :2]), _bits(pix_t[..., :2])) and torch.equal(cal_u, cal)
    inside = (pix[..., 0] > 0) & (pix[..., 0] < w - 1) & (pix[..., 1] > 0) & (pix[..., 1] < h - 1)
    np.testing.assert_array_equal(und[..., 2].cpu().numpy(), np.where(inside, pix[..., 2], 0))
    # in place == out of place, for both kernels and both instantiations
    for cs, ds, c, d in ((72, 20, cal, dst), (0, 0, cal[0], dst[0]), (72, 0, cal, dst[0]), (0, 20, cal[0], dst)):
        out = torch.empty_like(pix_t)
        _undistort_c(pix_t, out, c, cs, d, ds, 17.0, 3.5)
        same = pix_t.clone()
        _undistort_c(same, same, c, cs, d, ds, 17.0, 3.5)
        assert torch.equal(_bits(out), _bits(same))
        _distort_c(pix_t, out, c, cs, d, ds)
        same = pix_t.clone()
        _distort_c(same, same, c, cs, d, ds)
        assert torch.equal(_bits(out), _bits(same))
    # batch splits
    whole = inputs.undistort_pixels(pix_t, cal, dst, margin=(w / 2, h / 2))[0]
    wd = inputs.distort_pixels(pix_t.clone(), cal, dst)
    for s, n in ((0, 1), (1, 2047), (2048, 2952)):
        part = inputs.undistort_pixels(pix_t[s:s + n], cal[s:s + n], dst[s:s + n], margin=(w / 2, h / 2))[0]
        assert torch.equal(_bits(part), _bits(whole[s:s + n]))
        pd = inputs.distort_pixels(pix_t[s:s + n].clone(), cal[s:s + n], dst[s:s + n])
        assert torch.equal(_bits(pd), _bits(wd[s:s + n]))
    # CUDA-graph replay == direct calls
    gi, go, gd = pix_t.clone(), torch.empty_like(pix_t), torch.empty_like(pix_t)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s), torch.cuda.graph(g, stream=s):
        _undistort_c(gi, go, cal, 72, dst, 20, w / 2, h / 2)
        _distort_c(gi, gd, cal, 72, dst, 20)
    torch.cuda.current_stream().wait_stream(s)
    go.zero_()
    gd.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(_bits(go), _bits(whole)) and torch.equal(_bits(gd), _bits(wd))
    empty = torch.empty((0, 4, 17, 3), device="cuda")
    assert inputs.undistort_pixels(empty, cal[:0], dst[:0], margin=1.0)[0].shape == (0, 4, 17, 3)
    assert inputs.distort_pixels(empty, cal[:0], dst[:0]).shape == (0, 4, 17, 3)


def _triangulations(pix, calib):
    lin, used = inputs.triangulate(pix, calib)
    rob, inl = inputs.triangulate_robust(pix, calib, inlier_px=10.0)
    ref, _ = inputs.refine_triangulation(pix, calib, lin, max_iters=20)
    return (lin, rob, ref), (used >= 2, inl != 0, used >= 2)


@pytest.mark.parametrize("kind,V,cameras", [("h36m", 4, False), ("cmu", 5, True)])
def test_undistorted_exact_pixels_recover_the_poses(kind, V, cameras):
    rig = synth.make_rig(V, kind)
    n = 4000
    cams = inputs.synth_cameras(n, V, kind, seed=2) if cameras else None
    pix, target, calib = inputs.synth_project(n, rig, seed=2, conf_mode="ones", cameras=cams)
    dist = np.tile(LENS[kind], (V, 1))
    inputs.distort_pixels(pix, calib, dist)
    und, calib_u = inputs.undistort_pixels(pix, calib, dist)
    tgt = target.cpu().numpy()
    for (pts, mask), (raw_pts, raw_mask) in zip(zip(*_triangulations(und, calib_u)), zip(*_triangulations(pix, calib))):
        m = mask.cpu().numpy()
        assert m.mean() > 0.5
        err = np.linalg.norm(pts.cpu().numpy() - tgt, axis=-1)[m]
        assert err.max() <= 1e-5, err.max()
        raw_err = np.linalg.norm(raw_pts.cpu().numpy() - tgt, axis=-1)[raw_mask.cpu().numpy()]
        assert np.mean(raw_err) > 2e-3, np.mean(raw_err)                # the distorted pixels are off by millimetres to cm


def test_zero_distortion_leaves_every_triangulation_bitwise_unchanged():
    rig = synth.make_rig(4, "h36m")
    pix, _, calib = inputs.synth_project(3000, rig, seed=9)
    inputs.add_detector_noise(pix, calib, 9, 0, 2.0, 0.1, 0.05)
    und, calib_u = inputs.undistort_pixels(pix, calib, np.zeros((4, 5)), margin=0.0)
    for a, b in zip(_triangulations(und, calib_u), _triangulations(pix, calib)):
        for x, y in zip(a, b):
            assert torch.equal(_bits(x.to(torch.float32)), _bits(y.to(torch.float32)))


def test_evaluation_with_lens_distortion():
    lens = LENS["h36m"]
    kw = dict(arch="cmu0", views=4, poses=3000, micro_batch=1024, precision="fp32", rig="h36m", pixel_noise=2,
              outlier_rate=0.1, triangulate=True, triangulate_robust=True, refine_triangulations=True)
    line = evaluate.run(**kw, lens_distortion=lens)
    assert line["data"]["lens_distortion"]["coefficients"] == dict(zip(("k1", "k2", "p1", "p2", "k3"), lens))
    # step by step: project, distort, noise, lifter inputs from the distorted pixels, triangulations on the undistorted ones
    J = 17
    accs = {k: metric.MpjpeAccumulator(J, output_in_meter=True) for k in ("t", "r", "tf", "rf")}
    rig = synth.make_rig(4, "h36m")
    for s0 in range(0, 3000, 1024):
        n = min(1024, 3000 - s0)
        pix, target, calib = inputs.synth_project(n, rig, seed=1, start=s0)
        inputs.distort_pixels(pix, calib, np.tile(lens, (4, 1)))
        inputs.add_detector_noise(pix, calib, 1, s0, 2.0, 0.1, 0.0)
        und, calib_u = inputs.undistort_pixels(pix, calib, np.tile(lens, (4, 1)), margin=(500.0, 500.0))
        lin, used = inputs.triangulate(und, calib_u)
        rob, inl = inputs.triangulate_robust(und, calib_u, inlier_px=10.0)
        accs["t"].update(lin, target, used >= 2)
        accs["r"].update(rob, target, inl != 0)
        accs["tf"].update(inputs.refine_triangulation(und, calib_u, lin, max_iters=20)[0], target, used >= 2)
        accs["rf"].update(inputs.refine_triangulation(und, calib_u, rob, view_mask=inl, max_iters=20)[0], target, inl != 0)
    for key, entry, sub in (("t", "triangulation", None), ("r", "triangulation_robust", None),
                            ("tf", "triangulation", "refined"), ("rf", "triangulation_robust", "refined")):
        got = line[entry] if sub is None else line[entry][sub]
        want = evaluate.triangulation_summary(accs[key].acc.cpu().numpy(), J)
        for m in ("absolute", "root_relative", "triangulated_joints"):
            assert abs(got["mpjpe_cm"][m] - want["mpjpe_cm"][m]) <= 1e-9 * abs(want["mpjpe_cm"][m]), (entry, sub, m)
        assert got["under_determined_joints"] == want["under_determined_joints"]
    # the lifter saw the distorted pixels: its error differs from the run without a lens; the rest of the line keeps its keys
    plain = evaluate.run(**kw)
    assert "lens_distortion" not in plain["data"] and set(plain) == set(line)
    assert line["mpjpe_cm"]["absolute"] != plain["mpjpe_cm"]["absolute"]
    assert line["triangulation"]["mpjpe_cm"]["triangulated_joints"] < 1.5 * plain["triangulation"]["mpjpe_cm"]["triangulated_joints"]
    with pytest.raises(ValueError, match="lens_distortion"):
        evaluate.run(arch="cmu0", views=4, poses=100, lens_distortion=(0.1, 0.2))
