"""mpl_triangulate_robust on the device: on noiseless pixels it is bitwise the linear triangulation, on noisy detections
with confident false detections it agrees with the numpy oracle and beats the linear DLT, results do not depend on how
the batch is split or whether they come from a CUDA graph, and the evaluation reports it next to the linear baseline."""
import numpy as np
import pytest
import torch

import robust_triangulation_oracle as rto
from openmpl_b200 import evaluate, inputs, synth

pytestmark = pytest.mark.gpu


def _candidates(pix, calib, min_conf=0.0):
    """[B, J] int32 bitmask of the views mpl_triangulate uses."""
    u, v, c = pix[..., 0].double(), pix[..., 1].double(), pix[..., 2]
    w, h = calib[:, 16].view(1, -1, 1), calib[:, 17].view(1, -1, 1)
    cand = (c > min_conf) & (0 < u) & (u < w - 1) & (0 < v) & (v < h - 1)                   # [B,V,J]
    bits = (1 << torch.arange(pix.shape[1], device=pix.device, dtype=torch.int32)).view(1, -1, 1)
    return (cand.int() * bits).sum(dim=1, dtype=torch.int32)


@pytest.mark.parametrize("kind,V", [("h36m", 2), ("h36m", 4), ("h36m", 8), ("h36m", 16), ("cmu", 5)])
def test_noiseless_unit_confidence_is_bitwise_the_linear_triangulation(kind, V):
    rig = synth.make_rig(V, kind)
    pix, target, calib = inputs.synth_project(4096, rig, seed=11, start=123, conf_mode="ones")
    points, inliers = inputs.triangulate_robust(pix, calib)
    lin, used = inputs.triangulate(pix, calib)
    assert inliers.dtype == torch.int32
    full = (inliers == _candidates(pix, calib)) & (used >= 2)
    assert float(full.sum()) >= 0.99 * float((used >= 2).sum())
    assert torch.equal(points[full].view(torch.int32), lin[full].view(torch.int32))
    ok = inliers != 0
    assert torch.isnan(points[~ok]).all() and not torch.isnan(points[ok]).any()
    assert float((points[ok] - target[ok]).abs().max()) <= 1e-5                               # metres


@pytest.mark.parametrize("kind,V", [("h36m", 4), ("cmu", 5)])
@pytest.mark.parametrize("min_conf", [0.0, 0.5])
def test_noisy_detections_match_the_oracle_and_beat_the_linear_dlt(kind, V, min_conf):
    rig = synth.make_rig(V, kind)
    pix, target, calib = inputs.synth_project(300, rig, seed=4)
    raw = pix.cpu().numpy()
    inputs.add_detector_noise(pix, calib, 8, 0, 2.0, 0.15, 0.05)
    noisy = pix.cpu().numpy()
    points, inliers = inputs.triangulate_robust(pix, calib, min_conf=min_conf)
    lin, used = inputs.triangulate(pix, calib, min_conf=min_conf)
    points, inliers, lin = points.cpu().numpy(), inliers.cpu().numpy(), lin.cpu().numpy()
    want, want_inl, near = rto.triangulate_robust(noisy, rig.R, rig.t, rig.f, rig.c, rig.image_size, min_conf)
    sure = ~near
    assert sure.mean() > 0.9
    np.testing.assert_array_equal(inliers[sure], want_inl[sure])
    np.testing.assert_array_equal(np.isnan(points), np.isnan(want))
    det = sure & (inliers != 0)
    assert det.mean() > 0.5
    assert np.abs(points[det] - want[det]).max() <= 1e-6
    # items with a confident false detection among >= 3 candidates
    cand = _candidates(pix, calib, min_conf).cpu().numpy()
    outlier = (noisy[..., 2] != raw[..., 2]) & (noisy[..., 2] != 0)                            # [B,V,J]
    bits = (outlier * (1 << np.arange(V))[None, :, None]).sum(axis=1)
    n_cand = np.vectorize(lambda m: bin(m).count("1"))(cand)
    hit = ((bits & cand) != 0) & (n_cand >= 3)
    assert hit.sum() > 50
    t = target.cpu().numpy().astype(np.float64)
    err_r = np.linalg.norm(points[hit] - t[hit], axis=-1)
    err_l = np.linalg.norm(lin[hit] - t[hit], axis=-1)
    assert np.nanmedian(err_r) < 0.1 * np.nanmedian(err_l)


@pytest.mark.parametrize("B", [0, 1, 4097, 65536])
@pytest.mark.parametrize("J", [17, 40])
def test_batch_split_is_bitwise_invariant(B, J):
    V = 4
    rig = synth.make_rig(V, "h36m")
    calib = inputs.pack_calibration(rig.R, rig.t, rig.f, rig.c, rig.image_size)
    gen = torch.Generator(device="cuda").manual_seed(B + J)
    scale = torch.tensor([1100.0, 1100.0, 1.2], device="cuda")
    pix = torch.rand(B, V, J, 3, device="cuda", generator=gen) * scale - torch.tensor([50.0, 50.0, 0.1], device="cuda")
    whole = inputs.triangulate_robust(pix, calib, min_conf=0.2, inlier_px=200.0)
    k = B // 3
    parts = [inputs.triangulate_robust(pix[s], calib, min_conf=0.2, inlier_px=200.0) for s in (slice(0, k), slice(k, B))]
    assert torch.equal(whole[0].view(torch.int32), torch.cat([p[0] for p in parts]).view(torch.int32))   # NaNs included
    assert torch.equal(whole[1], torch.cat([p[1] for p in parts]))
    if B >= 4097:
        assert bool((whole[1] != 0).any()) and bool((whole[1] == 0).any())


def test_noise_and_robust_triangulation_replay_from_a_cuda_graph():
    """Neither call allocates or synchronises, so both can be captured and replayed."""
    rig = synth.make_rig(5, "cmu")
    clean, _, calib = inputs.synth_project(3000, rig, seed=2)
    eager_pix = inputs.add_detector_noise(clean.clone(), calib, 3, 0, 2.0, 0.1, 0.05)
    eager = inputs.triangulate_robust(eager_pix, calib)
    buf = torch.empty_like(clean)
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        buf.copy_(clean)                                              # warm-up outside the capture
        inputs.triangulate_robust(inputs.add_detector_noise(buf, calib, 3, 0, 2.0, 0.1, 0.05), calib)
        with torch.cuda.graph(g):
            buf.copy_(clean)
            out = inputs.triangulate_robust(inputs.add_detector_noise(buf, calib, 3, 0, 2.0, 0.1, 0.05), calib)
    torch.cuda.current_stream().wait_stream(s)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(buf.view(torch.int32), eager_pix.view(torch.int32))
    assert torch.equal(out[0].view(torch.int32), eager[0].view(torch.int32)) and torch.equal(out[1], eager[1])


def test_evaluation_reports_the_robust_triangulation_on_noisy_detections():
    n = 2000
    kw = dict(arch="cmu0", views=4, poses=n, precision="fp32")
    line = evaluate.run(**kw, pixel_noise=2, outlier_rate=0.1, triangulate=True, triangulate_robust=True)
    lin, rob = line["triangulation"], line["triangulation_robust"]
    assert rob["mpjpe_cm"]["triangulated_joints"] < lin["mpjpe_cm"]["triangulated_joints"]
    assert line["data"]["pixel_noise_px"] == 2 and line["data"]["outlier_rate"] == 0.1 and line["data"]["miss_rate"] == 0
    assert rob["method"] != lin["method"] == "linear DLT, pixel-space rows, views with conf > 0 inside the image"
    # without the new arguments nothing changes: same keys, same data string, same lifter numbers
    plain = evaluate.run(**kw)
    zero = evaluate.run(**kw, pixel_noise=0, outlier_rate=0, miss_rate=0)
    assert set(plain) == {"metric", "value", "unit", "n_gpus", "ms_total", "poses", "dtype", "data", "config", "mpjpe_cm",
                          "tflops"}
    assert plain["data"] == "synthetic (device generator keyed by global pose index)" and set(zero) == set(plain)
    for k, v in plain["mpjpe_cm"].items():                 # fp64 atomics may add the same terms in another order
        if isinstance(v, float):
            assert abs(zero["mpjpe_cm"][k] - v) <= 1e-12 * abs(v), k
            assert line["mpjpe_cm"][k] != v, k                  # the lifter saw the noisy detections
