"""Multi-person association on the device: mpl_synth_people is bitwise its numpy twin; noiseless people are associated with
pair precision >= 0.999 and >= 99 % of associable people pure and complete, and a person row seen in every view
triangulates bitwise like the person-ordered row; on noisy detections with outliers members, labels and people are bitwise
tests/association_oracle.py's on every frame it does not flag as near; results do not depend on the frame split, CUDA-graph
capture or a repeated calibration stride; gather and score match numpy exactly; evaluate.run(people=...) reports the
association."""
import numpy as np
import pytest
import torch

from openmpl_b200 import _lib, evaluate, inputs, synth

import association_oracle as oracle

pytestmark = pytest.mark.gpu

J = 17


def _scene(kind, V, P, F, seed=1, start=0, noise=None, cameras=False):
    """(scene, perm, calib per frame or rig, pix [F P, V, J, 3]) of frames [start, start + F) on the device."""
    rig = synth.make_rig(V, kind)
    cams = inputs.synth_cameras(F, V, kind, seed=seed, start=start) if cameras else None
    pix, _, calib = inputs.synth_project(F * P, rig, seed=seed, start=start * P,
                                         cameras=None if cams is None else cams.repeat_interleave(P, 0))
    if noise is not None:
        inputs.add_detector_noise(pix, calib, seed, start * P, *noise)
    scene, perm = inputs.synth_people(pix, P, seed, start)
    return scene, perm, (calib if cams is None else cams), pix


def _np(*ts):
    return [t.cpu().numpy() for t in ts]


@pytest.mark.parametrize("P,V", [(1, 4), (3, 5), (8, 4), (16, 8), (8, 16), (64, 2)])
def test_synth_people_matches_the_twin(P, V):
    F = 97
    pix = torch.randn(F * P, V, J, 3, device="cuda")
    pix[0, 0, 0, 0] = float("nan")
    pix[-1, -1, -1, 2] = -0.0
    scene, perm = inputs.synth_people(pix, P, seed=3, start=1000)
    want_scene, want_perm = synth.synth_people(pix.cpu().numpy(), P, seed=3, start=1000)
    np.testing.assert_array_equal(perm.cpu().numpy(), want_perm)
    np.testing.assert_array_equal(scene.cpu().numpy().view(np.int32), want_scene.view(np.int32))
    assert (np.sort(want_perm, -1) == np.arange(P)).all()
    a = inputs.synth_people(pix[:40 * P], P, seed=3, start=1000)
    b = inputs.synth_people(pix[40 * P:], P, seed=3, start=1040)
    assert torch.equal(torch.cat([a[1], b[1]]), perm)
    assert torch.equal(torch.cat([a[0], b[0]]).view(torch.int32), scene.view(torch.int32))     # NaN != NaN: compare bits


@pytest.mark.parametrize("kind,V", [("h36m", 4), ("cmu", 5)])
@pytest.mark.parametrize("P", [2, 3, 4, 5, 6, 7, 8])
def test_noiseless_people_are_associated(kind, V, P):
    F = 400
    scene, perm, calib, pix = _scene(kind, V, P, F, seed=P)
    members, labels, people = inputs.associate_people(scene, calib)
    owner, acc = inputs.association_score(members, labels, perm)
    a = acc.cpu().numpy()
    precision, complete = a[6] / a[5], a[4] / a[1]
    print(f"{kind} V={V} P={P}: pair precision {precision:.6f} recall {a[6] / a[7]:.6f} complete {complete:.6f} "
          f"({int(a[4])} / {int(a[1])}), people past K {int((people - P).clamp(min=0).sum())}")
    assert a[0] == F and precision >= 0.999 and complete >= 0.99
    # a pure, complete row whose owner is active in every view is the owner's row: the same triangulation, bit for bit
    rows = inputs.gather_people(scene, members).view(F * P, V, J, 3)
    pts, used = inputs.triangulate(rows, calib)
    own = owner.long().clamp(min=0) + torch.arange(F, device="cuda")[:, None] * P
    ref, ref_used = inputs.triangulate(pix[own.view(-1)], calib)
    m, lab, o, pm = _np(members, labels, owner, perm)
    full = np.zeros((F, P), dtype=bool)
    for f in range(F):
        for k in range(P):
            if o[f, k] < 0 or (m[f, k] < 0).any():
                continue
            slots = [int(np.nonzero(pm[f, v] == o[f, k])[0][0]) for v in range(V)]
            full[f, k] = all(pm[f, v, m[f, k, v]] == o[f, k] for v in range(V)) and \
                all(lab[f, slots[v], v] != -2 for v in range(V))
    sel = torch.from_numpy(full.reshape(-1)).cuda()
    assert sel.float().mean() > 0.5
    assert torch.equal(pts[sel].view(torch.int32), ref[sel].view(torch.int32)) and torch.equal(used[sel], ref_used[sel])


CASES = [("h36m", 4, 4, 300, 0.1, 3), ("cmu", 5, 4, 300, 0.1, 3), ("cmu", 5, 6, 200, 0.2, 5), ("h36m", 8, 16, 40, 0.1, 3),
         ("h36m", 16, 8, 40, 0.1, 3), ("cmu", 2, 3, 300, 0.05, 1)]


@pytest.mark.parametrize("kind,V,P,F,max_dist,min_joints", CASES)
def test_noisy_detections_match_the_oracle(kind, V, P, F, max_dist, min_joints):
    scene, perm, calib, _ = _scene(kind, V, P, F, seed=V + P, start=11, noise=(2.0, 0.1, 0.05), cameras=True)
    members, labels, people = inputs.associate_people(scene, calib, min_joints=min_joints, max_dist=max_dist)
    m, lab, n = _np(members, labels, people)
    want_m, want_lab, want_n, near = oracle.associate(scene.cpu().numpy(), calib.cpu().numpy(), 0.0, min_joints, max_dist)
    ok = ~near
    print(f"{kind} V={V} P={P}: {ok.mean():.4f} of {F} frames unflagged, mean people {n.mean():.2f}")
    assert ok.mean() >= 0.99
    np.testing.assert_array_equal(m[ok], want_m[ok])
    np.testing.assert_array_equal(lab[ok], want_lab[ok])
    np.testing.assert_array_equal(n[ok], want_n[ok])
    # and the score of the device's association is the oracle's score of it
    owner, acc = inputs.association_score(members, labels, perm)
    want_owner, want_acc = oracle.score(m, lab, perm.cpu().numpy())
    np.testing.assert_array_equal(owner.cpu().numpy(), want_owner)
    np.testing.assert_array_equal(acc.cpu().numpy(), want_acc)


def test_split_graph_capture_and_stride():
    V, P, F = 5, 6, 500
    scene, _, calib, _ = _scene("cmu", V, P, F, seed=2, noise=(2.0, 0.1, 0.0), cameras=True)
    full = inputs.associate_people(scene, calib, max_people=4)
    for cut in (1, 123, 499):
        a = inputs.associate_people(scene[:cut], calib[:cut], max_people=4)
        b = inputs.associate_people(scene[cut:], calib[cut:], max_people=4)
        for x, y, z in zip(a, b, full):
            assert torch.equal(torch.cat([x, y]), z)
    # one block repeated under a stride is bitwise stride 0
    rig = calib[0].contiguous()
    ref = inputs.associate_people(scene, rig)
    rep = inputs.associate_people(scene, rig.expand(F, V, 18).contiguous())
    for x, y in zip(ref, rep):
        assert torch.equal(x, y)
    padded = torch.zeros(F, V * 18 + 7, dtype=torch.float64, device="cuda")
    padded[:, :V * 18] = rig.reshape(-1)
    out = [torch.full_like(t, 7) for t in ref]
    L = _lib.lib()
    _lib.check(L.mpl_associate_people_strided(scene.data_ptr(), padded.data_ptr(), V * 18 + 7, F, P, V, J, 0.0, 3, 0.1, P,
                                              out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(), None))
    torch.cuda.synchronize()
    for x, y in zip(ref, out):
        assert torch.equal(x, y)
    # CUDA-graph capture of the whole chain: associate, gather, score
    perm = torch.rand(F, V, P, device="cuda").argsort(-1).int()
    members, labels, people = (torch.full_like(t, 9) for t in full)
    rows = torch.empty(F, 4, V, J, 3, device="cuda")
    owner = torch.empty(F, 4, dtype=torch.int32, device="cuda")
    acc = torch.zeros(8, dtype=torch.float64, device="cuda")
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()

    def chain(stream):
        _lib.check(L.mpl_associate_people_strided(scene.data_ptr(), calib.data_ptr(), 18 * V, F, P, V, J, 0.0, 3, 0.1, 4,
                                                  members.data_ptr(), labels.data_ptr(), people.data_ptr(), stream))
        _lib.check(L.mpl_gather_people(scene.data_ptr(), members.data_ptr(), F, P, 4, V, J, rows.data_ptr(), stream))
        _lib.check(L.mpl_association_score(members.data_ptr(), labels.data_ptr(), perm.data_ptr(), F, P, 4, V,
                                           owner.data_ptr(), acc.data_ptr(), stream))

    with torch.cuda.stream(s):
        chain(s.cuda_stream)                                           # warm up (sets the kernel's shared-memory limit)
        s.synchronize()
        with torch.cuda.graph(g, stream=s):
            chain(s.cuda_stream)
    for t in (members, labels, people, rows, owner):
        t.fill_(-5)
    acc.zero_()
    g.replay()
    torch.cuda.synchronize()
    for x, y in zip((members, labels, people), full):
        assert torch.equal(x, y)
    assert torch.equal(rows, inputs.gather_people(scene, full[0]))
    o, a = inputs.association_score(full[0], full[1], perm)
    assert torch.equal(owner, o) and torch.equal(acc, a)


def test_gather_and_score_match_numpy():
    F, P, K, V = 300, 5, 7, 4
    scene = torch.randn(F, P, V, J, 3, device="cuda")
    scene[3, 1, 2, 4, 0] = float("nan")
    members = torch.randint(-1, P, (F, K, V), dtype=torch.int32, device="cuda")
    out = inputs.gather_people(scene, members).cpu().numpy()
    sc, m = _np(scene, members)
    want = np.where((m >= 0)[..., None, None], sc[np.arange(F)[:, None, None], np.maximum(m, 0), np.arange(V)], 0.0)
    np.testing.assert_array_equal(out.view(np.int32), want.astype(np.float32).view(np.int32))
    labels = torch.randint(-2, K, (F, P, V), dtype=torch.int32, device="cuda")
    perm = torch.rand(F, V, P, device="cuda").argsort(-1).int()
    acc = torch.full((8,), 0.5, dtype=torch.float64, device="cuda")
    owner, acc = inputs.association_score(members, labels, perm, acc)
    want_owner, want_acc = oracle.score(m, labels.cpu().numpy(), perm.cpu().numpy())
    np.testing.assert_array_equal(owner.cpu().numpy(), want_owner)
    np.testing.assert_array_equal(acc.cpu().numpy(), want_acc + 0.5)


def test_evaluate_people():
    kw = dict(arch="cmu0", views=5, depth=2, poses=16384, micro_batch=4096, precision="fp32", triangulate=True, people=4)
    line = evaluate.run(**kw)
    a = line["association"]
    print({k: a[k] for k in ("frames", "associable_people", "pair_precision", "pair_recall", "pure_fraction",
                              "complete_fraction", "dropped_past_k")})
    assert a["frames"] == 4096 and a["pair_precision"] >= 0.999 and a["complete_fraction"] >= 0.99
    assert a["scored_rows"] > 0.9 * 16384 and line["poses"] == a["scored_rows"]
    assert np.isfinite(line["mpjpe_cm"]["absolute"]) and np.isfinite(line["triangulation"]["mpjpe_cm"]["triangulated_joints"])
    noisy = evaluate.run(**kw, pixel_noise=2.0, outlier_rate=0.1, triangulate_robust=True, random_cameras=True,
                         lens_distortion=(-0.2, 0.1, 0.0, 0.0, 0.0), calib_noise=(0.1, 5.0), refine_triangulations=True,
                         triangulation_pmpjpe=True)
    b = noisy["association"]
    print({k: b[k] for k in ("pair_precision", "pair_recall", "pure_fraction", "complete_fraction")},
          noisy["triangulation_robust"]["mpjpe_cm"])
    assert 0.5 < b["pair_precision"] <= 1.0 and 0.5 < b["pair_recall"] <= 1.0
    assert np.isfinite(noisy["triangulation_robust"]["refined"]["procrustes_aligned"]["p_mpjpe_cm"])
