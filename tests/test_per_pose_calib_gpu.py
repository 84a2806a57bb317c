"""A calibration per pose on the device: with one rig repeated in every row the per-pose path is bitwise the shared one for
all five consumers; with distinct calibrations each pose gets what a one-pose call with its own calibration gives; the input
builder matches the reference's per-sample construction; mpl_synth_cameras matches its numpy twin, shards freely and
replays from a CUDA graph; random camera setups triangulate back to the targets; the evaluation runs on them."""
import numpy as np
import pytest
import torch

from openmpl_b200 import _lib, evaluate, inputs, synth
from oracle import mpl_oracle

pytestmark = pytest.mark.gpu


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _bits(x):
    return x.contiguous().view(torch.int32)


def _room(kind="h36m"):
    return torch.tensor(synth.rig_kind(kind)[2], dtype=torch.float64, device="cuda")


def _consumers(pix, calib, stride, seed=5, start=0):
    """Outputs of all five consumers for pixels pix [B, V, J, 3] and calibrations at the given stride, as int32 bit views."""
    L = _lib.lib()
    B, V, J, _ = pix.shape
    s = _stream()
    out = {}
    poses, rays = torch.empty_like(pix), torch.empty_like(pix)
    centers = torch.empty((B, V, 1, 3), dtype=torch.float32, device="cuda")
    _lib.check(L.mpl_build_inputs_strided(pix.data_ptr(), calib.data_ptr(), stride, B, V, J, poses.data_ptr(), rays.data_ptr(),
                                          centers.data_ptr(), s))
    out["build_inputs"] = (poses, rays, centers)
    pts, used = torch.empty((B, J, 3), device="cuda"), torch.empty((B, J), dtype=torch.int32, device="cuda")
    _lib.check(L.mpl_triangulate_strided(pix.data_ptr(), calib.data_ptr(), stride, B, V, J, 0.2, pts.data_ptr(), used.data_ptr(),
                                         s))
    out["triangulate"] = (pts, used)
    rpts, inl = torch.empty((B, J, 3), device="cuda"), torch.empty((B, J), dtype=torch.int32, device="cuda")
    _lib.check(L.mpl_triangulate_robust_strided(pix.data_ptr(), calib.data_ptr(), stride, B, V, J, 0.2, 200.0, rpts.data_ptr(),
                                                inl.data_ptr(), s))
    out["triangulate_robust"] = (rpts, inl)
    noisy = pix.clone()
    _lib.check(L.mpl_synth_detector_noise_strided(seed, start, B, V, J, calib.data_ptr(), stride, 2.0, 0.2, 0.1,
                                                  noisy.data_ptr(), s))
    out["detector_noise"] = (noisy,)
    spix, target = torch.empty_like(pix), torch.empty((B, J, 3), device="cuda")
    _lib.check(L.mpl_synth_project_strided(seed, start, B, V, J, calib.data_ptr(), stride, _room().data_ptr(), 0,
                                           spix.data_ptr(), target.data_ptr(), s))
    out["synth_project"] = (spix, target)
    return {k: tuple(_bits(t) for t in v) for k, v in out.items()}


def _random_pix(B, V, J, seed, w=1000.0, h=1000.0):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    scale = torch.tensor([w + 100.0, h + 100.0, 1.2], device="cuda")
    return torch.rand(B, V, J, 3, device="cuda", generator=gen) * scale - torch.tensor([50.0, 50.0, 0.1], device="cuda")


@pytest.mark.parametrize("B", [1, 4097, 65536])
@pytest.mark.parametrize("J", [1, 5, 17, 40])
@pytest.mark.parametrize("V", [2, 5, 16])
def test_repeated_rig_is_bitwise_the_shared_calibration(B, J, V):
    rig = synth.make_rig(V, "h36m")
    calib = torch.as_tensor(inputs.pack_calibration(rig.R, rig.t, rig.f, rig.c, rig.image_size)).cuda()
    tiled = calib.expand(B, V, 18).contiguous()
    pix = _random_pix(B, V, J, B + 31 * J + V)
    shared = _consumers(pix, calib, 0)
    per_pose = _consumers(pix, tiled, 18 * V)
    for k in shared:
        for a, b in zip(shared[k], per_pose[k]):
            assert torch.equal(a, b), k
    if B >= 4097:                                                    # the triangulations produced points
        used, inl = shared["triangulate"][1], shared["triangulate_robust"][1]
        assert bool((used >= 2).any()) and bool((inl != 0).any())
        if V < 16:                                                   # ... and NaNs (16 random views leave no item under-determined)
            assert bool((used < 2).any())


@pytest.mark.parametrize("V,J,kind", [(5, 17, "cmu"), (16, 1, "h36m"), (4, 5, "h36m"), (16, 40, "h36m")])
def test_each_pose_gets_its_own_calibration(V, J, kind):
    B, start = 4097, 300
    cams = inputs.synth_cameras(B, V, kind, seed=9, start=start)
    w, h = synth.rig_kind(kind)[1]
    pix = _random_pix(B, V, J, 17, w, h)
    got = _consumers(pix, cams, 18 * V, start=start)
    # first, last, the poses that straddle an item tile of either tile size, and random ones
    edge = {0, B - 1} | {min(B - 1, (t * k) // J) for t in (128, 12, 32) for k in range(1, 40)}
    rest = np.random.default_rng(0).choice(np.setdiff1d(np.arange(B), sorted(edge)), 256 - len(edge), replace=False)
    sample = sorted(edge) + [int(b) for b in rest]
    assert len(sample) == 256
    for b in sample:
        one = _consumers(pix[b:b + 1].contiguous(), cams[b].contiguous(), 0, start=start + b)
        for k in one:
            for a, full in zip(one[k], got[k]):
                assert torch.equal(a[0], full[b]), (k, b)


def test_input_builder_matches_the_reference_pose_by_pose():
    V, B = 4, 64
    cams = inputs.synth_cameras(B, V, "cmu", seed=2)
    rig = synth.make_rig(V, "cmu")
    pix, _, calib = inputs.synth_project(B, rig, seed=3, cameras=cams)
    inputs.add_detector_noise(pix, calib, 3, 0, 3.0, 0.2, 0.0)
    poses, rays, centers = (x.cpu().numpy() for x in inputs.build_inputs(pix, calib))
    pix, cal = pix.cpu().numpy(), calib.cpu().numpy()
    assert len({cal[b, 0, 12] for b in range(B)}) == B                          # every pose has its own cameras
    for b in range(B):
        c = cal[b]
        want = mpl_oracle.build_inputs(pix[b:b + 1], c[:, :9].reshape(V, 3, 3), c[:, 9:12], c[:, 12:14], c[:, 14:16],
                                       tuple(c[0, 16:18]))
        np.testing.assert_array_equal(poses[b:b + 1], want[0])
        np.testing.assert_array_equal(centers[b:b + 1], want[2])
        np.testing.assert_allclose(rays[b:b + 1], want[1], rtol=0, atol=1e-6)


@pytest.mark.parametrize("kind,V", [("h36m", 4), ("cmu", 5), ("h36m", 16), ("cmu", 1)])
def test_device_cameras_match_the_twin_and_shard_freely(kind, V):
    B, start = 3000, 12345
    got = inputs.synth_cameras(B, V, kind, seed=6, start=start)
    want = synth.random_cameras(B, V, kind, seed=6, start=start)
    assert got.shape == (B, V, 18) and got.dtype == torch.float64
    assert np.abs(got.cpu().numpy() - want).max() <= 1e-12
    k = 1234
    parts = torch.cat([inputs.synth_cameras(k, V, kind, seed=6, start=start),
                       inputs.synth_cameras(B - k, V, kind, seed=6, start=start + k)])
    assert torch.equal(parts, got)
    assert torch.equal(inputs.synth_cameras(10, V, kind, seed=6, start=start + 100), got[100:110])


def test_synth_cameras_replays_from_a_cuda_graph():
    B, V = 5000, 8
    eager = inputs.synth_cameras(B, V, "h36m", seed=4, start=77)
    room = _room("h36m")
    out = torch.zeros_like(eager)
    f0, (w, h), _ = synth.rig_kind("h36m")
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        args = (4, 77, B, V, f0, float(w), float(h), room.data_ptr(), out.data_ptr())
        _lib.check(_lib.lib().mpl_synth_cameras(*args, s.cuda_stream))
        out.zero_()
        with torch.cuda.graph(g, stream=s):
            _lib.check(_lib.lib().mpl_synth_cameras(*args, s.cuda_stream))
    torch.cuda.current_stream().wait_stream(s)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)


@pytest.mark.parametrize("kind", ["h36m", "cmu"])
@pytest.mark.parametrize("V", [2, 4, 5, 8, 16])
def test_random_cameras_triangulate_back_to_the_targets(kind, V):
    B = 4096
    cams = inputs.synth_cameras(B, V, kind, seed=5, start=50)
    pix, target, calib = inputs.synth_project(B, synth.make_rig(V, kind), seed=5, start=50, conf_mode="ones", cameras=cams)
    assert calib.data_ptr() == cams.data_ptr()
    points, used = inputs.triangulate(pix, calib)
    ok = used >= 2
    assert float(ok.float().mean()) > 0.8                                              # random cameras may not all see a joint
    # metres.  With V = 2 the two cameras can face each other at about a joint's height, which puts the joint near the
    # baseline, where the fp32 rounding of the pixels is amplified (measured up to 5e-5 m); more views bound it to 1e-5 m
    assert float((points[ok] - target[ok]).abs().max()) <= (1e-4 if V == 2 else 1e-5)
    rob, inl = inputs.triangulate_robust(pix, calib)
    full = inl != 0
    assert torch.equal(full, ok)
    assert torch.equal(_bits(rob[full]), _bits(points[full]))


def test_per_pose_triangulations_replay_from_a_cuda_graph():
    B, V = 3000, 5
    cams = inputs.synth_cameras(B, V, "cmu", seed=8)
    clean, _, calib = inputs.synth_project(B, synth.make_rig(V, "cmu"), seed=8, cameras=cams)
    pix = inputs.add_detector_noise(clean.clone(), calib, 8, 0, 2.0, 0.1, 0.05)
    eager = inputs.triangulate(pix, calib) + inputs.triangulate_robust(pix, calib)
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        inputs.triangulate(pix, calib)
        inputs.triangulate_robust(pix, calib)
        with torch.cuda.graph(g, stream=s):
            out = inputs.triangulate(pix, calib) + inputs.triangulate_robust(pix, calib)
    torch.cuda.current_stream().wait_stream(s)
    g.replay()
    torch.cuda.synchronize()
    for a, b in zip(out, eager):
        assert torch.equal(_bits(a), _bits(b))


def test_evaluation_with_random_cameras():
    kw = dict(arch="cmu0", views=4, poses=2000, precision="fp32")
    line = evaluate.run(**kw, random_cameras=True, triangulate=True)
    assert line["triangulation"]["mpjpe_cm"]["triangulated_joints"] <= 1e-3
    assert line["data"]["source"] == "synthetic (device generator keyed by global pose index)"
    assert line["data"]["cameras"]["rig_kind"] == "cmu"
    # without the flag the line is that of the shared rig: same keys, same data string, same numbers
    plain = evaluate.run(**kw, triangulate=True)
    again = evaluate.run(**kw, triangulate=True, random_cameras=False)
    assert set(plain) == set(again) == {"metric", "value", "unit", "n_gpus", "ms_total", "poses", "dtype", "data", "config",
                                        "mpjpe_cm", "tflops", "triangulation"}
    assert plain["data"] == again["data"] == "synthetic (device generator keyed by global pose index)"
    for k, v in plain["mpjpe_cm"].items():                 # fp64 atomics may add the same terms in another order
        if isinstance(v, float):
            assert abs(again["mpjpe_cm"][k] - v) <= 1e-12 * abs(v), k
            assert line["mpjpe_cm"][k] != v, k                  # the lifter saw other cameras
