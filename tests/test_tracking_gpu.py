"""Tracking across frames on the device: mpl_synth_motion matches its numpy twin (the same uniforms bit for bit; the fp64
libm differences stay below an fp32 ulp in all but a few entries) and does not depend on the sequence split; on the noisy
pipeline motion -> detector noise -> slots -> association -> gather -> robust triangulation, mpl_track_people is bitwise
tests/tracking_oracle.py, and so is mpl_tracking_score; the ids do not depend on chunking the frames, on the sequence split
or on CUDA-graph capture; noiseless sequences are tracked without ID switches; evaluate.run(frames=...) reports the
tracking."""
import numpy as np
import pytest
import torch

from openmpl_b200 import _lib, evaluate, inputs, synth

import tracking_oracle as oracle

pytestmark = pytest.mark.gpu

J = 17


def _np(*ts):
    return [t.cpu().numpy() for t in ts]


def _check_twin(pix, target, want_pix, want_target):
    got_pix, got_target = _np(pix, target)
    np.testing.assert_array_equal(got_pix[..., 2], want_pix[..., 2])
    np.testing.assert_allclose(got_target, want_target, rtol=0, atol=2e-6)
    np.testing.assert_allclose(got_pix[..., :2], want_pix[..., :2], rtol=2e-6, atol=2e-4)
    same = (got_pix.view(np.int32) == want_pix.view(np.int32)).mean(), (got_target.view(np.int32) ==
                                                                      want_target.view(np.int32)).mean()
    print(f"bitwise equal: pix {same[0]:.6f}, target {same[1]:.6f}")
    assert min(same) >= 0.999


@pytest.mark.parametrize("kind,S,T,P,V", [("h36m", 3, 20, 2, 4), ("cmu", 2, 33, 5, 5), ("h36m", 1, 7, 8, 16),
                                          ("cmu", 5, 64, 1, 2)])
def test_synth_motion_matches_the_twin(kind, S, T, P, V):
    rig = synth.make_rig(V, kind)
    pix, target, calib = inputs.synth_motion(S, T, P, rig, seed=4, start=11)
    want_pix, want_target = synth.synth_motion(4, 11, S, T, P, calib.cpu().numpy(), rig.room)
    _check_twin(pix, target, want_pix, want_target)
    # any split of the sequences gives the same bits
    a = inputs.synth_motion(1, T, P, rig, seed=4, start=11)
    b = inputs.synth_motion(S - 1, T, P, rig, seed=4, start=12)
    assert torch.equal(torch.cat([a[0], b[0]]), pix) and torch.equal(torch.cat([a[1], b[1]]), target)


def test_synth_motion_per_row_cameras_and_conf_ones():
    S, T, P, V = 3, 10, 3, 4
    rig = synth.make_rig(V, "h36m")
    cams = inputs.synth_cameras(S, V, "h36m", seed=2).repeat_interleave(T * P, 0)
    pix, target, calib = inputs.synth_motion(S, T, P, rig, seed=2, start=0, conf_mode="ones", cameras=cams)
    want_pix, want_target = synth.synth_motion(2, 0, S, T, P, cams.cpu().numpy(), rig.room, conf_mode="ones")
    _check_twin(pix, target, want_pix, want_target)
    assert calib.data_ptr() == cams.data_ptr() or torch.equal(calib, cams)
    # the 3D motion does not depend on the cameras
    _, t2, _ = inputs.synth_motion(S, T, P, rig, seed=2, start=0)
    assert torch.equal(t2, target)


def _rows(kind, V, P, S, T, seed=1, noise=(2.0, 0.1, 0.05)):
    """The device pipeline: (robustly triangulated person rows [S, T, P, J, 3], the rows' owners [S, T, P])."""
    rig = synth.make_rig(V, kind)
    pix, _, calib = inputs.synth_motion(S, T, P, rig, seed=seed, start=0)
    if noise is not None:
        inputs.add_detector_noise(pix, calib, seed, 0, *noise)
    scene, perm = inputs.synth_people(pix, P, seed, 0)
    members, labels, _ = inputs.associate_people(scene, calib)
    owner, _ = inputs.association_score(members, labels, perm)
    rows = inputs.gather_people(scene, members).view(S * T * P, V, J, 3)
    points, _ = inputs.triangulate_robust(rows, calib)
    return points.view(S, T, P, J, 3), owner.view(S, T, P)


@pytest.mark.parametrize("P", [2, 4, 8])
def test_tracker_matches_the_oracle_on_the_noisy_pipeline(P):
    S, T = 64, 60
    points, owner = _rows("cmu", 5, P, S, T, seed=P)
    ids, state = inputs.track_people(points, min_joints=3, max_dist=0.2, max_age=5, max_tracks=2 * P)
    pts = points.cpu().numpy()
    want, _ = oracle.track(pts, max_tracks=2 * P, min_joints=3, max_dist=0.2, max_age=5)
    got = ids.cpu().numpy()
    print(f"P={P}: {np.isnan(pts).any(-1).mean():.4f} of the joints NaN, {(got >= 0).mean():.4f} of the rows tracked, "
          f"{got.max() + 1} ids at most")
    np.testing.assert_array_equal(got, want)
    acc = inputs.tracking_score(ids, owner, P)
    np.testing.assert_array_equal(acc.cpu().numpy(), oracle.score(got, owner.cpu().numpy(), P))


def test_chunks_split_and_graph_capture():
    P, S, T = 4, 48, 50
    points, _ = _rows("h36m", 4, P, S, T, seed=7)
    mask = (torch.rand(S, T, P, J, device="cuda") > 0.1).float()
    kw = dict(min_joints=3, max_dist=0.15, max_age=3, max_tracks=6)
    whole, wstate = inputs.track_people(points, mask, **kw)
    # frames in chunks on one state
    state = inputs.track_state(S, 6, J)
    parts = [inputs.track_people(points[:, a:b], mask[:, a:b], state=state, **kw)[0] for a, b in ((0, 1), (1, 23), (23, T))]
    assert torch.equal(torch.cat(parts, 1), whole) and torch.equal(state, wstate)
    # sequences split over calls
    a, sa = inputs.track_people(points[:17], mask[:17], **kw)
    b, sb = inputs.track_people(points[17:], mask[17:], **kw)
    assert torch.equal(torch.cat([a, b]), whole) and torch.equal(torch.cat([sa, sb]), wstate)
    # CUDA-graph capture of tracking and scoring, replayed on a zeroed state
    L = _lib.lib()
    owner = torch.randint(-1, P, (S, T, P), dtype=torch.int32, device="cuda")
    g_state = inputs.track_state(S, 6, J)
    g_ids = torch.full_like(whole, 9)
    g_acc = torch.zeros(_lib.TRACK_ACC_LEN, dtype=torch.float64, device="cuda")
    pts, msk = points.contiguous(), mask.contiguous()
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()

    def chain(stream):
        _lib.check(L.mpl_track_people(pts.data_ptr(), msk.data_ptr(), S, T, P, J, 3, 0.15, 3, 6, g_state.data_ptr(),
                                      g_ids.data_ptr(), stream))
        _lib.check(L.mpl_tracking_score(g_ids.data_ptr(), owner.data_ptr(), S, T, P, P, g_acc.data_ptr(), stream))

    with torch.cuda.stream(s):
        chain(s.cuda_stream)                                           # warm up (sets the kernel's shared-memory limit)
        s.synchronize()
        with torch.cuda.graph(g, stream=s):
            chain(s.cuda_stream)
    g_state.zero_()
    g_ids.fill_(-5)
    g_acc.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(g_ids, whole) and torch.equal(g_state, wstate)
    assert torch.equal(g_acc, inputs.tracking_score(whole, owner, P))


def test_largest_shapes_match_the_oracle():
    # K = 64 rows, 128 tracks, 32 joints: the largest shared-memory footprint
    S, T, K, Jx = 2, 6, 64, 32
    rng = np.random.default_rng(3)
    base = rng.uniform(-5, 5, (S, 1, K, 1, 3)) + rng.normal(0, 0.1, (S, 1, K, Jx, 3))
    pts = (base + rng.normal(0, 0.02, (S, T, K, Jx, 3))).astype(np.float32)
    pts[rng.random(pts.shape[:4]) < 0.1] = np.nan
    pts[:, 2, ::3] = np.nan
    ids, _ = inputs.track_people(torch.from_numpy(pts).cuda(), min_joints=4, max_dist=0.3, max_age=1, max_tracks=128)
    want, _ = oracle.track(pts, max_tracks=128, min_joints=4, max_dist=0.3, max_age=1)
    np.testing.assert_array_equal(ids.cpu().numpy(), want)
    ids, _ = inputs.track_people(torch.from_numpy(pts).cuda(), min_joints=4, max_dist=0.3, max_age=1, max_tracks=40)
    want, _ = oracle.track(pts, max_tracks=40, min_joints=4, max_dist=0.3, max_age=1)
    np.testing.assert_array_equal(ids.cpu().numpy(), want)
    assert (want == -1).any()


@pytest.mark.parametrize("kind,V,P", [("cmu", 5, 4), ("h36m", 4, 2), ("h36m", 4, 8)])
def test_noiseless_sequences_are_tracked(kind, V, P):
    S, T = 64, 60
    points, owner = _rows(kind, V, P, S, T, seed=3, noise=None)
    ids, _ = inputs.track_people(points, max_tracks=2 * P)
    a = inputs.tracking_score(ids, owner, P).cpu().numpy()
    mota = 1 - (a[4] + a[5] + a[6]) / a[2]
    print(f"{kind} V={V} P={P}: MOTA {mota:.6f}, misses {int(a[4])}, FP {int(a[5])}, IDSW {int(a[6])}, frag {int(a[7])}, "
          f"MT {int(a[8])} / {S * P}, tracks {int(a[10])}")
    assert a[6] == 0 and mota >= 0.98


def test_evaluate_frames():
    kw = dict(arch="cmu0", views=5, depth=2, poses=4 * 16 * 64, micro_batch=4 * 16 * 32, precision="fp32", people=4,
              frames=16)
    line = evaluate.run(**kw)
    t = line["tracking"]
    print({k: t[k] for k in ("sequences", "objects", "matches", "id_switches", "mota", "tracks_per_person", "ms")})
    assert t["sequences"] == 64 and t["frames"] == 64 * 16 and t["objects"] == 64 * 16 * 4
    assert t["id_switches"] == 0 and t["mota"] >= 0.98 and t["ms"] > 0
    assert line["association"]["frames"] == 64 * 16
    noisy = evaluate.run(**kw, pixel_noise=2.0, outlier_rate=0.1, miss_rate=0.05, random_cameras=True)
    print(noisy["tracking"])
    assert 0.0 < noisy["tracking"]["mota"] <= 1.0
    with pytest.raises(ValueError):
        evaluate.run(**kw, calib_noise=(0.5, 20), calibrate_rig=1024)
    with pytest.raises(ValueError):
        evaluate.run(**dict(kw, micro_batch=63))
    with pytest.raises(ValueError):
        evaluate.run(**dict(kw, people=0))
