"""mpl_triangulate_refine on the device: it matches the numpy oracle from the linear and the robust points, returns init
bit for bit where it does not refine, never raises the cost, gives the same bits in place, for any batch split, with a
calibration per pose and from a CUDA graph, and the evaluation reports the refined triangulations."""
import numpy as np
import pytest
import torch

import refine_triangulation_oracle as rfo
from openmpl_b200 import _lib, evaluate, inputs, synth

pytestmark = pytest.mark.gpu


def _bits(x):
    return x.contiguous().view(torch.int32)


def _random_pix(B, V, J, seed, w=1000.0, h=1000.0):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    scale = torch.tensor([w + 100.0, h + 100.0, 1.2], device="cuda")
    return torch.rand(B, V, J, 3, device="cuda", generator=gen) * scale - torch.tensor([50.0, 50.0, 0.1], device="cuda")


def _refine_c(pix, calib, stride, init, mask, points, reproj, max_iters=20, min_conf=0.0):
    B, V, J, _ = pix.shape
    _lib.check(_lib.lib().mpl_triangulate_refine_strided(
        pix.data_ptr(), calib.data_ptr(), stride, B, V, J, min_conf, None if mask is None else mask.data_ptr(), init.data_ptr(),
        max_iters, points.data_ptr(), reproj.data_ptr(), torch.cuda.current_stream().cuda_stream))


def _cost(pix, calib, X, use):
    """fp64 C at points X [B, J, 3] over use [B, V, J]; +inf where a used view sees X at depth <= 0."""
    P, _ = rfo.projections(calib)
    p = np.einsum("vrk,bjk->bvjr", P, np.concatenate([X, np.ones(X.shape[:-1] + (1,))], axis=-1))
    with np.errstate(divide="ignore", invalid="ignore"):
        r = p[..., :2] / p[..., 2:3] - pix[..., :2].astype(np.float64)
        c = np.where(use, pix[..., 2].astype(np.float64) ** 2 * (r * r).sum(-1), 0.0).sum(axis=1)
    return np.where(((p[..., 2] <= 0) & use).any(axis=1), np.inf, c)


@pytest.mark.parametrize("kind,V", [("h36m", 2), ("h36m", 4), ("h36m", 8), ("h36m", 16), ("cmu", 5)])
@pytest.mark.parametrize("min_conf", [0.0, 0.5])
def test_device_matches_the_oracle_from_both_inits(kind, V, min_conf):
    rig = synth.make_rig(V, kind)
    pix, _, calib = inputs.synth_project(300, rig, seed=4)
    inputs.add_detector_noise(pix, calib, 8, 0, 2.0, 0.1, 0.05)
    lin, _ = inputs.triangulate(pix, calib, min_conf=min_conf)
    rob, inl = inputs.triangulate_robust(pix, calib, min_conf=min_conf)
    cal, npix = calib.cpu().numpy(), pix.cpu().numpy()
    # The linear point with its outliers needs up to ~80 iterations on these detections (a fifth of the items reach a cap
    # of 20), the robust point over its inliers at most ~16.  Where the cap cuts an iteration off, the point depends on the
    # rounding of every step taken, so the caps are chosen to let (almost) every item stop by the step rule.
    for init, mask, iters in ((lin, None, 100), (rob, inl, 20)):
        got, rp = inputs.refine_triangulation(pix, calib, init, view_mask=mask, min_conf=min_conf, max_iters=iters)
        got, rp, x0 = got.cpu().numpy(), rp.cpu().numpy(), init.cpu().numpy()
        want = rfo.refine(npix, cal, x0, None if mask is None else mask.cpu().numpy(), min_conf, iters)
        np.testing.assert_array_equal(np.isnan(rp), ~want["refined"])
        ok = want["refined"]
        assert ok.mean() > 0.2
        np.testing.assert_array_equal(got[~ok].view(np.int32), x0[~ok].view(np.int32))        # init bit for bit
        sure = ok & want["by_step"]
        assert sure.sum() >= 0.995 * ok.sum()
        # metres, plus one fp32 ulp: the fp64 points may straddle a rounding boundary of the output
        assert np.all(np.abs(got[sure] - want["points"][sure]) <= 1e-6 + 2.0 ** -23 * np.abs(want["points"][sure]))
        np.testing.assert_allclose(rp[sure], want["reproj_px"][sure], rtol=1e-5, atol=1e-6)
        # C(refined) <= C(init), both recomputed in fp64 from the outputs; slack for rounding the refined X to fp32
        use = rfo.candidates(npix, rfo.projections(cal)[1][None], min_conf)
        if mask is not None:
            use &= ((mask.cpu().numpy()[:, None, :] >> np.arange(V)[None, :, None]) & 1).astype(bool)
        c0 = _cost(npix, cal, x0.astype(np.float64), use)
        c1 = _cost(npix, cal, got.astype(np.float64), use)
        assert np.all(c1[ok] <= c0[ok] * (1 + 1e-6) + 1e-6)


def test_in_place_is_bitwise_out_of_place():
    rig = synth.make_rig(5, "cmu")
    pix, _, calib = inputs.synth_project(3000, rig, seed=6)
    inputs.add_detector_noise(pix, calib, 6, 0, 2.0, 0.1, 0.05)
    rob, inl = inputs.triangulate_robust(pix, calib)
    for mask in (None, inl):
        out, rp = inputs.refine_triangulation(pix, calib, rob, view_mask=mask)
        buf, rp2 = rob.clone(), torch.empty_like(rp)
        _refine_c(pix, calib, 0, buf, mask, buf, rp2)
        assert torch.equal(_bits(buf), _bits(out)) and torch.equal(_bits(rp2), _bits(rp))


@pytest.mark.parametrize("B", [0, 1, 4097, 65536])
@pytest.mark.parametrize("J", [17, 40])
def test_batch_split_is_bitwise_invariant(B, J):
    V = 4
    rig = synth.make_rig(V, "h36m")
    calib = inputs.pack_calibration(rig.R, rig.t, rig.f, rig.c, rig.image_size)
    pix = _random_pix(B, V, J, B + J)
    init, _ = inputs.triangulate(pix, calib, min_conf=0.2)
    _, inl = inputs.triangulate_robust(pix, calib, min_conf=0.2, inlier_px=200.0)
    for mask in (None, inl):
        whole = inputs.refine_triangulation(pix, calib, init, view_mask=mask, min_conf=0.2)
        k = B // 3
        parts = [inputs.refine_triangulation(pix[s], calib, init[s], view_mask=None if mask is None else mask[s], min_conf=0.2)
                 for s in (slice(0, k), slice(k, B))]
        for n in range(2):
            assert torch.equal(_bits(whole[n]), _bits(torch.cat([p[n] for p in parts])))           # NaNs included
        if B >= 4097:
            refined = ~torch.isnan(whole[1])
            assert bool(refined.any()) and bool((~refined).any())


@pytest.mark.parametrize("B", [1, 4097])
@pytest.mark.parametrize("J", [1, 17, 40])
@pytest.mark.parametrize("V", [2, 5, 16])
def test_repeated_rig_is_bitwise_the_shared_calibration(B, J, V):
    rig = synth.make_rig(V, "h36m")
    calib = torch.as_tensor(inputs.pack_calibration(rig.R, rig.t, rig.f, rig.c, rig.image_size)).cuda()
    tiled = calib.expand(B, V, 18).contiguous()
    pix = _random_pix(B, V, J, B + 31 * J + V)
    init, _ = inputs.triangulate(pix, calib, min_conf=0.2)
    _, inl = inputs.triangulate_robust(pix, calib, min_conf=0.2, inlier_px=200.0)
    for mask in (None, inl):
        shared = inputs.refine_triangulation(pix, calib, init, view_mask=mask, min_conf=0.2)
        per_pose = inputs.refine_triangulation(pix, tiled, init, view_mask=mask, min_conf=0.2)
        for a, b in zip(shared, per_pose):
            assert torch.equal(_bits(a), _bits(b))


@pytest.mark.parametrize("V,J,kind", [(5, 17, "cmu"), (16, 1, "h36m"), (4, 5, "h36m"), (16, 40, "h36m")])
def test_each_pose_gets_its_own_calibration(V, J, kind):
    B, start = 4097, 300
    cams = inputs.synth_cameras(B, V, kind, seed=9, start=start)
    rig = synth.make_rig(V, kind)
    pix, _, calib = inputs.synth_project(B, rig, seed=9, start=start, cameras=cams)
    pix = torch.cat([inputs.add_detector_noise(pix, calib, 9, start, 2.0, 0.1, 0.05)] * 3, dim=2)[:, :, :J].contiguous()
    init, inl = inputs.triangulate_robust(pix, calib)
    got = inputs.refine_triangulation(pix, calib, init, view_mask=inl)
    assert float((~torch.isnan(got[1])).float().mean()) > 0.5
    # first, last, the poses that straddle an item tile of either tile size, and random ones
    edge = {0, B - 1} | {min(B - 1, (t * k) // J) for t in (128, 12, 32) for k in range(1, 40)}
    rest = np.random.default_rng(0).choice(np.setdiff1d(np.arange(B), sorted(edge)), 128 - len(edge), replace=False)
    for b in sorted(edge) + [int(r) for r in rest]:
        one = inputs.refine_triangulation(pix[b:b + 1], cams[b], init[b:b + 1], view_mask=inl[b:b + 1])
        for a, full in zip(one, got):
            assert torch.equal(_bits(a[0]), _bits(full[b])), b


@pytest.mark.parametrize("per_pose", [False, True])
def test_refinement_replays_from_a_cuda_graph(per_pose):
    B, V = 3000, 5
    rig = synth.make_rig(V, "cmu")
    cams = inputs.synth_cameras(B, V, "cmu", seed=8) if per_pose else None
    pix, _, calib = inputs.synth_project(B, rig, seed=8, cameras=cams)
    inputs.add_detector_noise(pix, calib, 8, 0, 2.0, 0.1, 0.05)
    lin, _ = inputs.triangulate(pix, calib)
    rob, inl = inputs.triangulate_robust(pix, calib)
    eager = inputs.refine_triangulation(pix, calib, lin) + inputs.refine_triangulation(pix, calib, rob, view_mask=inl)
    stride = 18 * V if per_pose else 0
    out = [torch.full_like(lin, 7.0), torch.full_like(eager[1], 7.0), torch.full_like(rob, 7.0), torch.full_like(eager[3], 7.0)]
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        _refine_c(pix, calib, stride, lin, None, out[0], out[1])                 # warm-up outside the capture
        for o in out:
            o.fill_(7.0)
        with torch.cuda.graph(g, stream=s):
            _refine_c(pix, calib, stride, lin, None, out[0], out[1])
            _refine_c(pix, calib, stride, rob, inl, out[2], out[3])
    torch.cuda.current_stream().wait_stream(s)
    g.replay()
    torch.cuda.synchronize()
    for a, b in zip(out, eager):
        assert torch.equal(_bits(a), _bits(b))


def test_evaluation_reports_the_refined_triangulations():
    kw = dict(arch="cmu0", views=4, poses=2000, precision="fp32")
    line = evaluate.run(**kw, pixel_noise=2, triangulate=True, triangulate_robust=True, refine_triangulations=True)
    for entry in ("triangulation", "triangulation_robust"):
        ref = line[entry]["refined"]
        assert set(ref) == {"mpjpe_cm", "under_determined_joints", "method", "note"}
        assert ref["under_determined_joints"] == line[entry]["under_determined_joints"]     # the parent entry's mask
        assert "Levenberg-Marquardt" in ref["method"] and "conf^2" in ref["method"] and "20 iterations" in ref["method"]
    lin = line["triangulation"]
    assert lin["refined"]["mpjpe_cm"]["triangulated_joints"] < lin["mpjpe_cm"]["triangulated_joints"]
    # without the flag the line is today's, key for key
    plain = evaluate.run(**kw, pixel_noise=2, triangulate=True, triangulate_robust=True)
    assert set(plain) == set(line) == {"metric", "value", "unit", "n_gpus", "ms_total", "poses", "dtype", "data", "config",
                                       "mpjpe_cm", "tflops", "triangulation", "triangulation_robust"}
    for entry in ("triangulation", "triangulation_robust"):
        assert set(plain[entry]) == {"mpjpe_cm", "under_determined_joints", "method", "note"}
        assert set(line[entry]) == set(plain[entry]) | {"refined"}
    with pytest.raises(ValueError, match="refine_triangulations"):
        evaluate.run(**kw, refine_triangulations=True)
