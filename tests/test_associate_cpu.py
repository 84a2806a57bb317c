"""Multi-person association without a GPU: the numpy oracle (tests/association_oracle.py) on hand-built scenes and costs,
the numpy twin of mpl_synth_people, the argument rules of the four entry points (checked before any CUDA call) and of
evaluate.py's --people options."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT
from openmpl_b200 import _lib, evaluate, inputs, synth

import association_oracle as oracle

INF = np.inf


def _rig(V, kind="h36m"):
    r = synth.make_rig(V, kind)
    return inputs.pack_calibration(r.R, r.t, r.f, r.c, r.image_size)


def _project(X, calib, conf=1.0):
    """X [J, 3] world points -> [V, J, 3] pixels (u, v, conf) through calib [V, 18]."""
    out = np.empty((len(calib), len(X), 3), dtype=np.float32)
    for v, c in enumerate(calib):
        y = (X - c[9:12]) @ c[:9].reshape(3, 3).T
        out[v, :, 0] = c[12] * y[:, 0] / y[:, 2] + c[14]
        out[v, :, 1] = c[13] * y[:, 1] / y[:, 2] + c[15]
        out[v, :, 2] = conf
    return out


def _costs(M, pairs):
    """A symmetric cost matrix with +inf off the given {(a, b): cost}."""
    c = np.full((M, M), INF)
    for (a, b), x in pairs.items():
        c[a, b] = c[b, a] = x
    return c


# ---- clustering rules on given costs (P slots, V views, detection m = s V + v) ------------------------------------------
def test_chain_is_not_merged_by_complete_linkage():
    # one slot, three views: 0-1 and 1-2 pass, 0-2 does not.  Single linkage would give one person of three.
    P, V = 1, 3
    cost = _costs(3, {(0, 1): 0.01, (1, 2): 0.02, (0, 2): 0.5})
    members, labels, people = oracle.cluster(cost, np.ones(3, bool), P, V, 0.1, K=2)
    assert people == 1
    np.testing.assert_array_equal(members, [[0, 0, -1], [-1, -1, -1]])
    np.testing.assert_array_equal(labels, [[0, 0, -1]])
    # once 0-2 passes too, the three are one person
    cost = _costs(3, {(0, 1): 0.01, (1, 2): 0.02, (0, 2): 0.05})
    members, labels, people = oracle.cluster(cost, np.ones(3, bool), P, V, 0.1, K=2)
    assert people == 1 and (members[0] == 0).all() and (labels == 0).all()


def test_clusters_sharing_a_view_are_not_merged():
    # two slots, two views: m = s V + v.  (0, v0) - (1, v1) cheapest, then (0, v0) - (0, v1): view 1 is taken
    P, V = 2, 2
    cost = _costs(4, {(0, 3): 0.01, (0, 1): 0.02, (2, 1): 0.03})
    members, labels, people = oracle.cluster(cost, np.ones(4, bool), P, V, 0.1, K=2)
    assert people == 2
    np.testing.assert_array_equal(members, [[0, 1], [1, 0]])          # person 0: slot 0 of view 0, slot 1 of view 1
    np.testing.assert_array_equal(labels, [[0, 1], [1, 0]])


def test_pair_order_is_cost_then_key():
    # equal costs: the smaller key m1 P V + m2 (m1 the lower view) wins
    P, V = 2, 2
    cost = _costs(4, {(0, 1): 0.05, (0, 3): 0.05})
    members, _, people = oracle.cluster(cost, np.ones(4, bool), P, V, 0.1, K=2)
    assert people == 1
    np.testing.assert_array_equal(members[0], [0, 0])                 # key 0 * 4 + 1 < 0 * 4 + 3


def test_ranking_ties_inactive_and_past_k():
    # three views, three slots: two people of two members and one of three; detection 8 (slot 2, view 2) inactive
    P, V = 3, 3
    active = np.ones(9, bool)
    active[8] = False
    cost = _costs(9, {(3, 4): 0.01, (0, 2): 0.02, (6, 7): 0.03, (6, 5): 0.04, (7, 5): 0.04})
    members, labels, people = oracle.cluster(cost, active, P, V, 0.1, K=2)
    assert people == 3
    # the three-member person first, then the two-member ones by their smallest member: {0, 2} before {3, 4}
    np.testing.assert_array_equal(members, [[2, 2, 1], [0, -1, 0]])
    np.testing.assert_array_equal(labels, [[1, -1, 1], [-1, -1, 0], [0, 0, -2]])


# ---- costs from geometry ------------------------------------------------------------------------------------------------
def _two_view_scene(J=6, seed=0):
    cal = _rig(2)
    rng = np.random.default_rng(seed)
    X = np.array([0.0, 0.25, 0.9]) + 0.25 * rng.standard_normal((J, 3))
    return cal, X, _project(X, cal)


def test_pair_cost_is_the_median_line_distance_and_ignores_an_outlier_joint():
    cal, X, pix = _two_view_scene()
    pix[1, 2, :2] = (50.0, 60.0)                                       # a confident false detection in view 1
    cost, active = oracle.pair_costs(pix[None], cal, 0.0, 3)            # P = 1: detections 0 (view 0) and 1 (view 1)
    assert active.all()
    # independent distances: closest points of the two rays by least squares
    d = []
    for j in range(6):
        rays = []
        for v in range(2):
            c = cal[v]
            q = np.array([(pix[v, j, 0] - c[14]) / c[12], (pix[v, j, 1] - c[15]) / c[13], 1.0])
            rays.append((c[9:12], c[:9].reshape(3, 3).T @ q))
        (c1, d1), (c2, d2) = rays
        ab = np.linalg.lstsq(np.stack([d1, -d2], 1), c2 - c1, rcond=None)[0]
        d.append(np.linalg.norm(c1 + ab[0] * d1 - c2 - ab[1] * d2))
    d = np.array(d)
    assert d[2] > 0.1 and np.delete(d, 2).max() < 1e-6
    assert abs(cost[0, 1] - np.median(d)) < 1e-9                       # even count: the mean of the two middle values
    assert cost[0, 1] < 1e-6 < np.mean(d) / 10
    members, labels, people, near = oracle.associate(pix[None, None], cal)
    assert people[0] == 1 and (members[0, 0] == 0).all() and not near[0]


def test_pair_sharing_fewer_than_min_joints_has_no_cost():
    cal, X, pix = _two_view_scene(J=5)
    pix[0, 3:, 2] = 0.0                                                # view 0 sees joints 0, 1, 2
    pix[1, [0, 4], 2] = 0.0                                            # view 1 sees joints 1, 2, 3
    cost, active = oracle.pair_costs(pix[None], cal, 0.0, 3)
    assert active.all() and cost[0, 1] == INF                          # both active, only joints 1 and 2 shared
    cost, _ = oracle.pair_costs(pix[None], cal, 0.0, 2)
    assert cost[0, 1] < 1e-6
    cost, active = oracle.pair_costs(pix[None], cal, 0.0, 4)
    assert not active.any()
    _, labels, people, _ = oracle.associate(pix[None, None], cal, min_joints=4)
    assert people[0] == 0 and (labels == -2).all()


def test_noiseless_people_are_found_and_score_perfectly():
    V, P = 4, 3
    cal = _rig(V)
    rng = np.random.default_rng(3)
    pix = np.concatenate([_project(np.array([x, y, 0.9]) + 0.25 * rng.standard_normal((17, 3)), cal)[None]
                          for x, y in ((-0.6, -1.0), (0.0, 0.5), (0.6, 1.6))])
    scene, perm = synth.synth_people(pix, P, seed=1, start=5)
    members, labels, people, near = oracle.associate(scene, cal)
    assert people[0] == P and not near[0]
    owner, acc = oracle.score(members, labels, perm)
    assert sorted(owner[0]) == [0, 1, 2]
    np.testing.assert_array_equal(acc, [1, P, P, P, P, P * 6, P * 6, P * 6])
    for k in range(P):
        for v in range(V):
            assert perm[0, v, members[0, k, v]] == owner[0, k]


def test_score_counts_impure_rows():
    # V = 3, P = 2; row 0 mixes person 0 (views 0, 1) and person 1 (view 2); row 1 holds person 1 in views 0 and 1
    perm = np.array([[[0, 1], [0, 1], [1, 0]]], dtype=np.int32)         # view 2: slot 0 holds person 1
    members = np.array([[[0, 0, 0], [1, 1, -1]]], dtype=np.int32)
    labels = np.array([[[0, 0, 0], [1, 1, -2]]], dtype=np.int32)        # detection (slot 1, view 2) inactive
    owner, acc = oracle.score(members, labels, perm)
    np.testing.assert_array_equal(owner, [[0, 1]])
    # active detections: person 0 in views 0 and 1 (its view-2 slot is inactive), person 1 in all three views.  Row 1 is pure
    # but misses person 1's view 2, so no row is complete
    np.testing.assert_array_equal(acc, [1, 2, 2, 1, 0, 3 + 1, 1 + 1, 1 + 3])


# ---- the scene generator's numpy twin -------------------------------------------------------------------------------------
def test_synth_people_twin_permutes_and_depends_on_the_global_frame_only():
    F, P, V, J = 30, 5, 3, 4
    pix = np.arange(F * P * V * J * 3, dtype=np.float32).reshape(F * P, V, J, 3)
    scene, perm = synth.synth_people(pix, P, seed=7, start=100)
    assert scene.shape == (F, P, V, J, 3) and perm.shape == (F, V, P) and perm.dtype == np.int32
    assert (np.sort(perm, -1) == np.arange(P)).all()
    for f in range(F):
        for v in range(V):
            for s in range(P):
                np.testing.assert_array_equal(scene[f, s, v], pix[f * P + perm[f, v, s], v])
    a = synth.people_permutations(7, 100, 11, P, V)
    b = synth.people_permutations(7, 111, F - 11, P, V)
    np.testing.assert_array_equal(np.concatenate([a, b]), perm)
    assert (perm != np.arange(P)).any()                                 # not the identity
    U = synth._uniforms(7, 100, F, V * P, key1=4).reshape(F, V, P)
    assert (np.diff(np.take_along_axis(U, perm, -1), axis=-1) >= 0).all()


# ---- argument rules --------------------------------------------------------------------------------------------------------
def test_new_symbols_are_declared_and_exported():
    header = open(os.path.join(ROOT, "include", "mpl_b200.h")).read()
    assert "#define MPL_ABI_VERSION 11" in header
    new = {"mpl_synth_people", "mpl_associate_people", "mpl_associate_people_strided", "mpl_gather_people",
           "mpl_association_score"}
    assert new <= set(re.findall(r"\b(mpl_[a-z0-9_]+)\s*\(", header)) and new <= set(_lib.EXPORTS)
    L = ctypes.CDLL(_lib.LIB_PATH)
    for name in new:
        assert hasattr(L, name), name
    assert _lib.lib().mpl_abi_version() == 11


def test_entry_points_reject_bad_arguments_before_any_cuda_call():
    L = _lib.lib()
    buf = ctypes.create_string_buffer(64)                               # host memory: never dereferenced on rejected paths
    p = ctypes.cast(buf, ctypes.c_void_p)
    E, OK = _lib.MPL_ERR_INVALID_ARGUMENT, _lib.MPL_OK

    def assoc(F=2, P=4, V=4, J=17, min_joints=3, max_dist=0.1, K=4, cs=0, scene=p, calib=p, out=p):
        yield L.mpl_associate_people_strided(scene, calib, cs, F, P, V, J, 0.0, min_joints, max_dist, K, out, out, out, None)
        if cs == 0:
            yield L.mpl_associate_people(scene, calib, F, P, V, J, 0.0, min_joints, max_dist, K, out, out, out, None)

    bad = [dict(F=-1), dict(V=1), dict(V=17), dict(P=0), dict(P=33, V=4), dict(J=0), dict(J=33, min_joints=3),
           dict(min_joints=0), dict(min_joints=18), dict(max_dist=0.0), dict(max_dist=-1.0), dict(max_dist=float("inf")),
           dict(max_dist=float("nan")), dict(K=0), dict(cs=1), dict(cs=-72), dict(cs=71), dict(F=0, V=17),
           dict(F=0, K=0), dict(scene=None), dict(calib=None), dict(out=None)]
    for kw in bad:
        for status in assoc(**kw):
            assert status == E, kw
            assert L.mpl_last_error().decode().startswith("mpl_associate_people_strided"), kw
    for kw in (dict(F=0), dict(F=0, scene=None, calib=None, out=None), dict(F=0, P=32, V=4, J=32, min_joints=32, cs=72),
               dict(F=0, P=64, V=2, K=1000)):
        for status in assoc(**kw):
            assert status == OK, kw

    def synth_call(F=2, start=0, P=4, V=4, J=17, pix=p, scene=ctypes.c_void_p(p.value + 16), perm=p):
        return L.mpl_synth_people(1, start, F, P, V, J, pix, scene, perm, None)

    for kw in (dict(F=-1), dict(start=-1), dict(V=0), dict(V=17), dict(P=0), dict(P=33), dict(J=0), dict(F=0, P=0),
               dict(pix=None), dict(scene=None), dict(perm=None), dict(scene=p)):
        assert synth_call(**kw) == E, kw
        assert L.mpl_last_error().decode().startswith("mpl_synth_people"), kw
    assert synth_call(F=0, pix=None, scene=None, perm=None) == OK
    assert synth_call(F=0, P=128, V=1) == OK

    def gather(F=2, P=4, K=4, V=4, J=17, scene=p, members=p, out=p):
        return L.mpl_gather_people(scene, members, F, P, K, V, J, out, None)

    for kw in (dict(F=-1), dict(P=0), dict(K=0), dict(V=0), dict(V=17), dict(J=0), dict(F=0, K=0), dict(scene=None),
               dict(members=None), dict(out=None)):
        assert gather(**kw) == E, kw
        assert L.mpl_last_error().decode().startswith("mpl_gather_people"), kw
    assert gather(F=0, scene=None, members=None, out=None) == OK

    def score(F=2, P=4, K=4, V=4, ptr=p, acc=p):
        return L.mpl_association_score(ptr, ptr, ptr, F, P, K, V, ptr, acc, None)

    for kw in (dict(F=-1), dict(P=0), dict(P=33), dict(K=0), dict(V=0), dict(V=17), dict(F=0, K=0), dict(ptr=None),
               dict(acc=None)):
        assert score(**kw) == E, kw
        assert L.mpl_last_error().decode().startswith("mpl_association_score"), kw
    assert score(F=0, ptr=None, acc=None) == OK


def test_wrappers_reject_bad_shapes():
    import torch
    with pytest.raises(ValueError, match=r"\[F P, V, J, 3\]"):
        inputs.synth_people(torch.zeros(10, 4, 17, 3), 4, 0, 0)
    with pytest.raises(ValueError, match="scene must be"):
        inputs.associate_people(torch.zeros(2, 4, 4, 17), _rig(4))
    with pytest.raises(ValueError, match="per-pose calibration"):
        inputs.associate_people(torch.zeros(2, 3, 4, 17, 3), np.zeros((3, 4, 18)))
    with pytest.raises(ValueError, match="members must be"):
        inputs.gather_people(torch.zeros(2, 3, 4, 17, 3), torch.zeros(2, 3, 4, dtype=torch.int64))
    i32 = dict(dtype=torch.int32)
    with pytest.raises(ValueError, match="perm"):
        inputs.association_score(torch.zeros(2, 3, 4, **i32), torch.zeros(2, 3, 4, **i32), torch.zeros(2, 3, 4, **i32))


def test_evaluation_refuses_invalid_people_options():
    for kw in (dict(people=1), dict(people=4, calib_noise=(0.5, 20), calibrate_rig=1024), dict(people=4, assoc_max_dist=0.0),
               dict(people=4, assoc_max_dist=float("nan")), dict(people=4, assoc_min_joints=0),
               dict(people=4, assoc_min_joints=18), dict(people=4, micro_batch=3), dict(people=40, views=4)):
        with pytest.raises(ValueError):
            evaluate.run(**kw)
    for args in (["--people", "1"], ["--people", "4", "--calib-noise", "0.5,20", "--calibrate-rig", "1024"],
                 ["--people", "4", "--assoc-max-dist", "0"], ["--people", "4", "--assoc-min-joints", "0"],
                 ["--people", "4", "--micro-batch", "2"], ["--people", "40"]):
        with pytest.raises(SystemExit):
            evaluate.main(args)
