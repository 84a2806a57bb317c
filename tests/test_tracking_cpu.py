"""Tracking across frames without a GPU: the numpy twin of mpl_synth_motion, the numpy oracle of the tracker and the score
(tests/tracking_oracle.py) on hand-built sequences, the argument rules of the three entry points (checked before any CUDA
call) and of evaluate.py's --frames options."""
import ctypes
import math
import os
import re

import numpy as np
import pytest

from conftest import ROOT
from openmpl_b200 import _lib, evaluate, inputs, synth

import tracking_oracle as oracle

J = 17


def _rig(V, kind="h36m"):
    r = synth.make_rig(V, kind)
    return inputs.pack_calibration(r.R, r.t, r.f, r.c, r.image_size)


# ---- the motion twin ---------------------------------------------------------------------------------------------------------
def test_motion_prefix_and_split():
    room = synth.make_rig(4).room
    whole = synth.motion_joints(3, 10, 5, 40, 3, room)
    np.testing.assert_array_equal(synth.motion_joints(3, 10, 5, 17, 3, room), whole[:, :17])      # frames: a prefix
    np.testing.assert_array_equal(np.concatenate([synth.motion_joints(3, 10, 2, 40, 3, room),
                                                  synth.motion_joints(3, 12, 3, 40, 3, room)]), whole)
    assert not np.array_equal(whole[:, 0], whole[:, 1])                                          # it moves
    calib = _rig(4)
    pix, target = synth.synth_motion(3, 10, 5, 40, 3, calib, room)
    assert pix.shape == (5 * 40 * 3, 4, J, 3) and target.shape == (5 * 40 * 3, J, 3)
    np.testing.assert_array_equal(target, whole.reshape(-1, J, 3).astype(np.float32))
    a, _ = synth.synth_motion(3, 10, 2, 40, 3, calib, room)
    b, _ = synth.synth_motion(3, 12, 3, 40, 3, calib, room)
    np.testing.assert_array_equal(np.concatenate([a, b]), pix)


@pytest.mark.parametrize("kind", ["h36m", "cmu"])
def test_motion_stays_in_the_room_and_is_smooth(kind):
    room = synth.make_rig(4, kind).room
    fps = 30.0
    X = synth.motion_joints(1, 0, 50, 300, 4, room, fps)
    root = X[..., 0, :]
    assert (root[..., 0] >= room[0]).all() and (root[..., 0] <= room[1]).all()
    assert (root[..., 1] >= room[2]).all() and (root[..., 1] <= room[3]).all()
    assert (root[..., 2] >= 0.8).all() and (root[..., 2] <= 1.0).all()
    # |d root / dt| <= 2 pi f_max a_max per axis, |d theta / dt| <= 0.5 rad/s: per frame each joint moves at most
    # (2 pi 0.1 0.5 |(w_x, w_y)| + 0.5 |o_xy|) / fps
    w = np.hypot(room[1] - room[0], room[3] - room[2])
    o_xy = np.linalg.norm((X[:, :1, :, :, :2] - X[:, :1, :, :1, :2]), axis=-1)                  # heading turns o, not its norm
    step = np.linalg.norm(np.diff(X, axis=1), axis=-1)
    bound = (2 * math.pi * 0.1 * 0.5 * w + 0.5 * o_xy) / fps
    assert (step <= bound * (1 + 1e-9) + 1e-12).all()
    print(f"{kind}: largest joint step {step.max() * fps:.3f} m/s, bound {bound.max() * fps:.3f} m/s")
    # the body keeps its shape: joint-to-root distances are constant in time
    d = np.linalg.norm(X - X[..., :1, :], axis=-1)
    np.testing.assert_allclose(d, np.broadcast_to(d[:, :1], d.shape), rtol=0, atol=1e-12)


def test_motion_confidences_are_synth_projects():
    rig = synth.make_rig(4)
    calib = _rig(4)
    S, T, P, start = 3, 7, 2, 5
    pix, _ = synth.synth_motion(9, start, S, T, P, calib, rig.room)
    ref = synth.make_batch(S * T * P, rig, seed=9, start=start * T * P)["poses"][..., 2]
    both = (ref > 0) & (pix[..., 2] > 0)
    assert both.mean() > 0.5
    np.testing.assert_array_equal(pix[..., 2][both], ref[both])
    ones, _ = synth.synth_motion(9, start, S, T, P, calib, rig.room, conf_mode="ones")
    assert set(np.unique(ones[..., 2])) <= {0.0, 1.0}


# ---- the tracker oracle on hand-built sequences -----------------------------------------------------------------------------
def _person(x, y, J=5):
    """A small body of J joints around (x, y, 1)."""
    off = np.stack([np.linspace(-0.2, 0.2, J), np.linspace(0.1, -0.1, J), np.linspace(-0.5, 0.5, J)], -1)
    return (np.array([x, y, 1.0]) + off).astype(np.float32)


def _seq(frames):
    """frames: list of lists of (x, y) or None rows -> points [1, T, K, 5, 3] (None rows are NaN)."""
    K = max(len(f) for f in frames)
    out = np.full((1, len(frames), K, 5, 3), np.nan, dtype=np.float32)
    for t, f in enumerate(frames):
        for k, r in enumerate(f):
            if r is not None:
                out[0, t, k] = _person(*r)
    return out


def test_two_people_crossing_keep_their_ids():
    T = 21
    frames = [[(-1.0 + 0.1 * t, 0.0 + 0.01 * t), (1.0 - 0.1 * t, 0.05)] for t in range(T)]
    frames = [f if t % 2 else f[::-1] for t, f in enumerate(frames)]                    # rows swap order every frame
    ids, _ = oracle.track(_seq(frames), max_tracks=4, max_dist=0.2)
    a = np.where(np.arange(T) % 2 == 1, ids[0, :, 0], ids[0, :, 1])                      # person a's row is 0 on odd frames
    b = np.where(np.arange(T) % 2 == 1, ids[0, :, 1], ids[0, :, 0])
    assert (a == 1).all() and (b == 0).all()                                             # b is row 0 of frame 0: born first


def test_gaps_up_to_max_age_keep_the_id():
    steady = [(0.0, 0.0)]
    for gap, same in ((3, True), (4, False)):
        frames = [steady] * 3 + [[None]] * gap + [steady] * 2
        ids, _ = oracle.track(_seq(frames), max_tracks=2, max_age=3)
        assert (ids[0, :3, 0] == 0).all() and (ids[0, 3:3 + gap, 0] == -1).all()
        assert (ids[0, 3 + gap:, 0] == (0 if same else 1)).all(), gap


def test_capacity_refusal_and_min_joints():
    frames = [[(0.0, 0.0), (2.0, 0.0), (4.0, 0.0)]]
    ids, _ = oracle.track(_seq(frames), max_tracks=2)
    np.testing.assert_array_equal(ids[0, 0], [0, 1, -1])
    pts = _seq(frames)
    pts[0, 0, 1, 2:] = np.nan                                                             # 2 used joints: no detection
    ids, _ = oracle.track(pts, max_tracks=4, min_joints=3)
    np.testing.assert_array_equal(ids[0, 0], [0, -1, 1])
    ids, _ = oracle.track(pts, max_tracks=4, min_joints=2)
    np.testing.assert_array_equal(ids[0, 0], [0, 1, 2])


def test_nan_masked_and_partial_updates():
    p0 = _person(0.0, 0.0)
    pts = np.stack([p0, p0 + np.float32(0.05), p0 + np.float32(0.05)])[None, :, None]        # [1, 3, 1, 5, 3]
    pts[0, 1, 0, 0] = np.nan                                                              # joint 0 unseen in frame 1
    mask = np.ones((1, 3, 1, 5), dtype=np.float32)
    mask[0, 1, 0, 1] = 0.0                                                                # joint 1 masked in frame 1
    tr = oracle.Tracker(2, min_joints=3)
    for t in range(3):
        assert tr.step(pts[0, t], mask[0, t])[0] == 0
        tk = tr.tracks[0]
        if t == 1:                                                                        # joints 0 and 1 keep frame 0
            np.testing.assert_array_equal(tk.pos[:2], p0[:2])
            np.testing.assert_array_equal(tk.pos[2:], pts[0, 1, 0, 2:])
    # the cost is the median over the shared joints: one far joint does not break the match
    far = pts[0, 2, 0].copy()
    far[4] += 10.0
    assert oracle.cost(tr.tracks[0], far, np.ones(5, bool), 3) == 0.0


def test_tie_break_by_key():
    # two tracks at the same distance from one row: the smaller id (key = id K + k) wins
    tr = oracle.Tracker(4, min_joints=1, max_dist=1.0)
    tr.step(np.stack([_person(-0.1, 0.0), _person(0.1, 0.0)]))
    ids = tr.step(np.stack([_person(0.0, 0.0), np.full((5, 3), np.nan, np.float32)]))
    np.testing.assert_array_equal(ids, [0, -1])
    tr = oracle.Tracker(4, min_joints=1, max_dist=1.0)
    tr.step(np.stack([_person(0.1, 0.0), _person(-0.1, 0.0)]))
    np.testing.assert_array_equal(tr.step(np.stack([_person(0.0, 0.0), _person(5.0, 0.0)])), [0, 2])


def test_chunked_equals_whole():
    rng = np.random.default_rng(1)
    pts = rng.normal(0, 0.05, (3, 30, 4, 6, 3)).astype(np.float32) + np.arange(4, dtype=np.float32)[None, None, :, None, None]
    pts[rng.random(pts.shape[:4]) < 0.2] = np.nan
    pts[:, 10:14, 2] = np.nan
    whole, _ = oracle.track(pts, max_tracks=5, max_dist=0.3, max_age=2)
    a, trs = oracle.track(pts[:, :11], max_tracks=5, max_dist=0.3, max_age=2)
    b, _ = oracle.track(pts[:, 11:], trackers=trs)
    np.testing.assert_array_equal(np.concatenate([a, b], 1), whole)
    assert (whole >= 0).mean() > 0.5 and whole.max() >= 4


# ---- the score on hand-built cases --------------------------------------------------------------------------------------------
def test_score_counts():
    T, K, P = 10, 3, 2
    tid = np.full((1, T, K), -1, np.int32)
    own = np.full((1, T, K), -1, np.int32)
    # person 0: id 0 in frames 0-3, nothing in 4-5, id 0 in 6-7, id 2 in 8-9 (one fragmentation, one switch)
    for t in list(range(4)) + [6, 7]:
        tid[0, t, 0], own[0, t, 0] = 0, 0
    for t in (8, 9):
        tid[0, t, 0], own[0, t, 0] = 2, 0
    # person 1: matched in frame 0 only (mostly lost); a duplicate row of person 0 in frame 3 is a false positive
    tid[0, 0, 1], own[0, 0, 1] = 1, 1
    tid[0, 3, 2], own[0, 3, 2] = 1, 0
    # a row without an owner but with an id is a false positive too
    tid[0, 5, 1] = 3
    acc = oracle.score(tid, own, P)
    want = dict(seq=1, frames=T, objects=T * P, matches=9, misses=T * P - 9, fp=2, idsw=1, frag=1, mt=1, ml=1, tracks=4)
    np.testing.assert_array_equal(acc, list(want.values()))


# ---- argument rules -----------------------------------------------------------------------------------------------------------
def test_new_symbols_are_declared_and_exported():
    header = open(os.path.join(ROOT, "include", "mpl_b200.h")).read()
    assert "#define MPL_ABI_VERSION 11" in header and "#define MPL_TRACK_ACC_LEN 11" in header
    new = {"mpl_synth_motion", "mpl_track_state_bytes", "mpl_track_people", "mpl_tracking_score"}
    assert new <= set(re.findall(r"\b(mpl_[a-z0-9_]+)\s*\(", header)) and new <= set(_lib.EXPORTS)
    L = ctypes.CDLL(_lib.LIB_PATH)
    for name in new:
        assert hasattr(L, name), name
    assert _lib.TRACK_ACC_LEN == 11


def test_state_bytes():
    L = _lib.lib()
    assert L.mpl_track_state_bytes(8, 17) == 4 * (4 + 8 * (4 + 3 * 17))
    for m, j in ((0, 17), (129, 17), (8, 0), (8, 33), (-1, 5)):
        assert L.mpl_track_state_bytes(m, j) == 0, (m, j)
    assert L.mpl_track_state_bytes(128, 32) > 0 and L.mpl_track_state_bytes(1, 1) > 0


def test_entry_points_reject_bad_arguments_before_any_cuda_call():
    L = _lib.lib()
    buf = ctypes.create_string_buffer(64)                               # host memory: never dereferenced on rejected paths
    p = ctypes.cast(buf, ctypes.c_void_p)
    E, OK = _lib.MPL_ERR_INVALID_ARGUMENT, _lib.MPL_OK

    def motion(S=2, start=0, T=3, P=2, V=4, J=17, cs=0, fps=30.0, ptr=p):
        return L.mpl_synth_motion(1, start, S, T, P, V, J, ptr, cs, ptr, fps, 0, ptr, ptr, None)

    for kw in (dict(S=-1), dict(start=-1), dict(T=0), dict(P=0), dict(V=0), dict(V=17), dict(J=0), dict(fps=0.0),
               dict(fps=-1.0), dict(fps=float("inf")), dict(fps=float("nan")), dict(cs=1), dict(cs=71), dict(S=0, T=0),
               dict(ptr=None)):
        assert motion(**kw) == E, kw
        assert L.mpl_last_error().decode().startswith("mpl_synth_motion"), kw
    assert motion(S=0, ptr=None) == OK and motion(S=0, cs=72) == OK

    def track(S=2, T=3, K=4, J=17, mj=3, md=0.2, age=5, nt=8, pts=p, state=p, out=p):
        return L.mpl_track_people(pts, None, S, T, K, J, mj, md, age, nt, state, out, None)

    for kw in (dict(S=-1), dict(T=-1), dict(T=1 << 31), dict(K=0), dict(K=65), dict(J=0), dict(J=33, mj=3), dict(mj=0),
               dict(mj=18), dict(md=0.0), dict(md=-1.0), dict(md=float("inf")), dict(md=float("nan")), dict(age=-1),
               dict(nt=0), dict(nt=129), dict(S=0, K=0), dict(T=0, nt=0), dict(pts=None), dict(state=None), dict(out=None),
               dict(state=ctypes.c_void_p(p.value + 2))):
        assert track(**kw) == E, kw
        assert L.mpl_last_error().decode().startswith("mpl_track_people"), kw
    for kw in (dict(S=0), dict(T=0), dict(S=0, pts=None, state=None, out=None), dict(T=0, K=64, J=32, mj=32, nt=128)):
        assert track(**kw) == OK, kw

    def score(S=2, T=3, K=4, P=4, ptr=p, acc=p):
        return L.mpl_tracking_score(ptr, ptr, S, T, K, P, acc, None)

    for kw in (dict(S=-1), dict(T=-1), dict(T=1 << 31), dict(K=0), dict(P=0), dict(S=0, P=0), dict(ptr=None),
               dict(acc=None)):
        assert score(**kw) == E, kw
        assert L.mpl_last_error().decode().startswith("mpl_tracking_score"), kw
    assert score(S=0, ptr=None, acc=None) == OK and score(T=0, ptr=None, acc=None) == OK


def test_wrappers_reject_bad_shapes():
    import torch
    with pytest.raises(ValueError, match="points must be"):
        inputs.track_people(torch.zeros(2, 3, 4, 17))
    with pytest.raises(ValueError, match="joint_mask"):
        inputs.track_people(torch.zeros(2, 3, 4, 17, 3), joint_mask=torch.ones(2, 3, 4))
    with pytest.raises(ValueError, match="state must be"):
        inputs.track_people(torch.zeros(2, 3, 4, 17, 3), state=torch.zeros(2, 7, dtype=torch.uint8))
    with pytest.raises(ValueError, match="unsupported tracker shape"):
        inputs.track_state(2, 129, 17, device="cpu")
    with pytest.raises(ValueError, match="owner"):
        inputs.tracking_score(torch.zeros(2, 3, 4, dtype=torch.int32), torch.zeros(2, 3, 5, dtype=torch.int32), 4)
    with pytest.raises(ValueError, match="per row"):
        inputs.synth_motion(2, 3, 2, synth.make_rig(4), device="cpu", cameras=np.zeros((4, 18)))


def test_evaluation_refuses_invalid_frames_options():
    for kw in (dict(frames=8), dict(people=4, frames=1), dict(people=4, frames=8, micro_batch=31),
               dict(people=4, frames=8, calib_noise=(0.5, 20), calibrate_rig=1024),
               dict(people=4, frames=8, track_max_dist=0.0), dict(people=4, frames=8, track_max_age=-1),
               dict(people=4, frames=8, poses=31)):
        with pytest.raises(ValueError):
            evaluate.run(**kw)
    for args in (["--frames", "8"], ["--people", "4", "--frames", "1"], ["--people", "4", "--frames", "8", "--micro-batch", "31"],
                 ["--people", "4", "--frames", "8", "--track-max-dist", "0"],
                 ["--people", "4", "--frames", "8", "--track-max-age", "-1"]):
        with pytest.raises(SystemExit):
            evaluate.main(args)
