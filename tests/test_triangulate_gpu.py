"""mpl_triangulate on the device: noiseless synthetic projections triangulate back to the generator's 3D targets (which
checks the camera model of synth_project_kernel and the calibration layout it shares with mpl_build_inputs end to end),
noisy pixels agree with the per-joint SVD of the oracle, and results do not depend on how the batch is split."""
import numpy as np
import pytest
import torch

import triangulation_oracle
from openmpl_b200 import evaluate, inputs, synth

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("conf_mode", ["uniform", "ones"])
@pytest.mark.parametrize("kind,V", [("h36m", 2), ("h36m", 4), ("h36m", 8), ("h36m", 16), ("cmu", 5)])
def test_noiseless_device_pipeline_recovers_the_targets(kind, V, conf_mode):
    rig = synth.make_rig(V, kind)
    pix, target, calib = inputs.synth_project(4096, rig, seed=11, start=123, conf_mode=conf_mode)
    points, used = inputs.triangulate(pix, calib)
    seen = (inputs.build_inputs(pix, calib)[0][..., 2] > 0).sum(dim=1, dtype=torch.int32)
    assert used.dtype == torch.int32 and torch.equal(used, seen)
    ok = used >= 2
    assert ok.float().mean() > 0.5
    assert torch.isnan(points[~ok]).all() and not torch.isnan(points[ok]).any()
    assert float((points[ok] - target[ok]).abs().max()) <= 1e-5                     # metres


@pytest.mark.parametrize("kind,V", [("h36m", 4), ("cmu", 5)])
@pytest.mark.parametrize("min_conf", [0.0, 0.5])
def test_noisy_pixels_match_the_oracle(kind, V, min_conf):
    rig = synth.make_rig(V, kind)
    pix, _, calib = inputs.synth_project(300, rig, seed=4, conf_mode="uniform")
    pix = pix.cpu().numpy()
    rng = np.random.default_rng(V * 10 + int(min_conf * 10))
    pix[..., :2] += rng.normal(0, 2.0, pix[..., :2].shape).astype(np.float32)            # sigma = 2 px
    low = rng.random(pix[..., 2].shape) < 0.3
    pix[..., 2] = np.where(low, pix[..., 2] * rng.random(pix[..., 2].shape), pix[..., 2]).astype(np.float32)
    points, used = inputs.triangulate(torch.from_numpy(pix).cuda(), calib, min_conf=min_conf)
    want, want_used = triangulation_oracle.triangulate(pix, rig.R, rig.t, rig.f, rig.c, rig.image_size, min_conf)
    points, used = points.cpu().numpy(), used.cpu().numpy()
    np.testing.assert_array_equal(used, want_used)
    ok = used >= 2
    assert ok.mean() > 0.5
    assert np.isnan(points[~ok]).all()
    assert np.abs(points[ok] - want[ok]).max() <= 1e-6


@pytest.mark.parametrize("B", [0, 1, 4097, 65536])
@pytest.mark.parametrize("J", [17, 40])
def test_batch_split_is_bitwise_invariant(B, J):
    V = 4
    rig = synth.make_rig(V, "h36m")
    calib = inputs.pack_calibration(rig.R, rig.t, rig.f, rig.c, rig.image_size)
    gen = torch.Generator(device="cuda").manual_seed(B + J)
    scale = torch.tensor([1100.0, 1100.0, 1.2], device="cuda")
    pix = torch.rand(B, V, J, 3, device="cuda", generator=gen) * scale - torch.tensor([50.0, 50.0, 0.1], device="cuda")
    whole = inputs.triangulate(pix, calib, min_conf=0.2)
    k = B // 3
    parts = [inputs.triangulate(pix[s], calib, min_conf=0.2) for s in (slice(0, k), slice(k, B))]
    assert torch.equal(whole[0].view(torch.int32), torch.cat([p[0] for p in parts]).view(torch.int32))   # NaNs included
    assert torch.equal(whole[1], torch.cat([p[1] for p in parts]))


def test_triangulation_replays_from_a_cuda_graph():
    """Nothing is allocated or synchronised inside the call, so it can be captured and replayed."""
    rig = synth.make_rig(5, "cmu")
    pix, _, calib = inputs.synth_project(3000, rig, seed=2)
    eager = inputs.triangulate(pix, calib)
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        inputs.triangulate(pix, calib)                                # warm-up outside the capture
        with torch.cuda.graph(g):
            out = inputs.triangulate(pix, calib)
    torch.cuda.current_stream().wait_stream(s)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out[0].view(torch.int32), eager[0].view(torch.int32)) and torch.equal(out[1], eager[1])


def test_evaluation_reports_the_triangulation_baseline():
    n = 300
    line = evaluate.run(arch="cmu0", views=2, poses=n, precision="fp32", triangulate=True)
    plain = evaluate.run(arch="cmu0", views=2, poses=n, precision="fp32")
    tri = line["triangulation"]
    assert tri["mpjpe_cm"]["triangulated_joints"] <= 1e-3                    # noiseless data
    pix, _, calib = inputs.synth_project(n, synth.make_rig(2, "cmu"), seed=1)
    seen = (inputs.build_inputs(pix, calib)[0][..., 2] > 0).sum(dim=1)
    assert tri["under_determined_joints"] == int((seen < 2).sum())
    # the lifter's numbers do not change; fp64 atomics may add the same terms in another order
    assert "triangulation" not in plain and line["poses"] == plain["poses"]
    for k, v in plain["mpjpe_cm"].items():
        if isinstance(v, float):
            assert abs(line["mpjpe_cm"][k] - v) <= 1e-12 * abs(v), k
