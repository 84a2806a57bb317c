"""Grouped MPJPE and masked / grouped P-MPJPE on the device (ABI 7): both match the numpy oracle over group orders, masks,
conf3d, room un-scaling and Procrustes modes, reduce to the ungrouped entry points where they should (bitwise for one
pose), ignore whatever lies under a masked joint, replay from a CUDA graph, do not depend on the batch split, and the
evaluation reports the P-MPJPE of its triangulations."""
import os

import numpy as np
import pytest
import torch

import masked_pmpjpe_oracle as mpo
from conftest import GOLDEN_DIR
from openmpl_b200 import _lib, evaluate, inputs, metric, synth
from oracle import mpl_oracle

pytestmark = pytest.mark.gpu

ROOM = {"room_x_scale": 1.7, "room_center": [0.5, -0.25, 1.0]}
MODES = [(True, "best"), (False, "best"), (True, False), (True, True), (False, True)]


def _poses(B, J, seed, noise=0.05):
    rng = np.random.default_rng(seed)
    gt = (rng.normal(0, 0.3, size=(B, J, 3)) + rng.uniform(-2, 2, size=(B, 1, 3))).astype(np.float32)
    pred = (gt + rng.normal(0, noise, size=(B, J, 3))).astype(np.float32)
    return pred, gt


def _groups(B, G, order, seed):
    rng = np.random.default_rng(seed)
    g = rng.integers(0, G, B)
    if order == "sorted":
        return np.sort(g)
    if order == "unlabelled":                            # -1 and values >= G are dropped
        g[rng.random(B) < 0.1] = -1
        g[rng.random(B) < 0.05] = G + 3
    return g


def _cuda(*xs):
    return [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in xs]


def _grouped_mpjpe(pred, gt, group, G, conf=None, room=None):
    acc = metric.MpjpeAccumulator(pred.shape[1], num_groups=G)
    acc.update(*_cuda(pred, gt), None if conf is None else _cuda(conf)[0], room=room, group=_cuda(group)[0])
    return acc


GROUPED_CASES = [(1, "sorted", 1, 1), (1, "sorted", 17, 4097), (15, "sorted", 17, 4097), (15, "shuffled", 40, 4097),
                 (15, "unlabelled", 1, 4097), (4096, "shuffled", 17, 4097), (4096, "unlabelled", 40, 4097),
                 (15, "shuffled", 17, 1), (4096, "sorted", 40, 1)]


def _check_grouped_mpjpe(G, order, J, B, conf_on, room, seed):
    pred, gt = _poses(B, J, seed)
    group = _groups(B, G, order, seed + 1)
    conf = (np.random.default_rng(seed + 2).random((B, J)) > 0.2).astype(np.float32) if conf_on else None
    got = _grouped_mpjpe(pred, gt, group, G, conf, room).acc.cpu().numpy()
    p, g = mpl_oracle.room_unscale(pred, gt, room) if room is not None else (pred, gt)
    want = mpo.grouped_metric_sums(p, g, group, G, conf)
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-300)


@pytest.mark.parametrize("G,order,J,B", GROUPED_CASES)
@pytest.mark.parametrize("conf_on", [False, True])
@pytest.mark.parametrize("room", [None, ROOM], ids=["noroom", "room"])
def test_grouped_mpjpe_matches_the_oracle(G, order, J, B, conf_on, room):
    _check_grouped_mpjpe(G, order, J, B, conf_on, room, seed=G + J + B)


@pytest.mark.parametrize("G,order", [(15, "sorted"), (15, "shuffled"), (4096, "unlabelled")])
def test_grouped_mpjpe_matches_the_oracle_at_a_million_poses(G, order):
    """Shared block sums (G = 15) and global atomics (G = 4096) over a batch well past the L2."""
    _check_grouped_mpjpe(G, order, 17, 1 << 20, True, None, seed=G)


@pytest.mark.parametrize("J", [1, 17, 40])
@pytest.mark.parametrize("conf_on", [False, True])
@pytest.mark.parametrize("room", [None, ROOM], ids=["noroom", "room"])
def test_one_group_is_the_ungrouped_entry_point(J, conf_on, room):
    for B in (1, 4097, 1 << 20) if J == 17 else (1, 4097):
        pred, gt = _poses(B, J, B + J)
        conf = (np.random.default_rng(B).random((B, J)) > 0.2).astype(np.float32) if conf_on else None
        plain = metric.MpjpeAccumulator(J)
        plain.update(*_cuda(pred, gt), None if conf is None else _cuda(conf)[0], room=room)
        grouped = _grouped_mpjpe(pred, gt, np.zeros(B, np.int32), 1, conf, room)
        unlabelled = torch.zeros(1, 11 * J + 1, dtype=torch.float64, device="cuda")
        c = None if conf is None else _cuda(np.repeat(conf[:, :, None], 3, axis=2))[0]
        p, g = _cuda(pred, gt)
        _lib.check(_lib.lib().mpl_mpjpe_accumulate_grouped(p.data_ptr(), g.data_ptr(), None if c is None else c.data_ptr(),
                                                           None, 1, B, J, 100.0, None if room is None else
                                                           (_lib.c_float * 6)(*([1.7] * 3 + ROOM["room_center"])),
                                                           unlabelled.data_ptr(), torch.cuda.current_stream().cuda_stream))
        a, b, n = plain.acc.cpu().numpy(), grouped.acc.cpu().numpy()[0], unlabelled.cpu().numpy()[0]
        if B == 1:
            assert a.tobytes() == b.tobytes() == n.tobytes()
        else:
            np.testing.assert_allclose(b, a, rtol=1e-12, atol=1e-300)
            np.testing.assert_allclose(n, a, rtol=1e-12, atol=1e-300)


def _masked_inputs(B, J, seed, off=0.2):
    pred, gt = _poses(B, J, seed)
    rng = np.random.default_rng(seed + 1)
    mask = (rng.random((B, J)) > off).astype(np.float32)
    if B > 8:
        mask[3, 2:] = 0                                  # two used joints: skipped
        pred[5, :, 2] = 0.25                             # a planar prediction: one singular value vanishes
        gt[6] = 0.5                                      # coincident targets (exact sums): skipped
    pred[mask == 0] = np.nan                             # poison under the mask
    gt[(mask == 0) & (rng.random((B, J)) > 0.5)] = np.inf
    return pred, gt, mask


def _masked(pred, gt, mask, group=None, G=None, scaling=True, reflection="best", unit=True):
    acc = metric.PmpjpeAccumulator(pred.shape[1], output_in_meter=unit, scaling=scaling, reflection=reflection, masked=True,
                                   num_groups=G)
    acc.update(*_cuda(pred, gt), mask=None if mask is None else _cuda(mask)[0],
               group=None if group is None else _cuda(group)[0])
    return acc


@pytest.mark.parametrize("scaling,reflection", MODES)
@pytest.mark.parametrize("J", [1, 17, 40])
@pytest.mark.parametrize("B", [1, 4097])
@pytest.mark.parametrize("G", [None, 15])
def test_masked_pmpjpe_matches_the_oracle(scaling, reflection, J, B, G):
    pred, gt, mask = _masked_inputs(B, J, seed=B + J)
    group = None if G is None else _groups(B, G, "unlabelled", B)
    got = _masked(pred, gt, mask, group, G, scaling, reflection).acc.cpu().numpy().reshape(-1, 2 * J + 4)
    want = mpo.masked_pmpjpe_sums(pred, gt, mask, group, G or 1, scaling=scaling, reflection=reflection)
    np.testing.assert_array_equal(got[:, J:2 * J], want[:, J:2 * J])          # counts are exact
    np.testing.assert_array_equal(got[:, 2 * J + 2:], want[:, 2 * J + 2:])
    np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-8)
    if J >= 17 and B > 1:
        assert want[:, 2 * J + 2].sum() > 0 and want[:, 2 * J + 3].sum() > 0


@pytest.mark.parametrize("scaling,reflection", MODES)
def test_all_ones_mask_is_bitwise_the_unmasked_kernel_per_pose(scaling, reflection):
    g = np.load(os.path.join(GOLDEN_DIR, "procrustes.npz"))
    cases = [(g["B"], g["A"], False)] + [(*_poses(64, 17, 9), True)]
    for pred, gt, unit in cases:
        J = pred.shape[1]
        for b in range(len(pred)):
            plain = metric.PmpjpeAccumulator(J, output_in_meter=unit, scaling=scaling, reflection=reflection)
            plain.update(*_cuda(pred[b:b + 1], gt[b:b + 1]))
            m = _masked(pred[b:b + 1], gt[b:b + 1], np.ones((1, J), np.float32), scaling=scaling, reflection=reflection,
                        unit=unit)
            a, c = plain.acc.cpu().numpy(), m.acc.cpu().numpy()
            assert a[:J].tobytes() == c[:J].tobytes() and a[J:J + 2].tobytes() == c[2 * J:2 * J + 2].tobytes(), b
            assert c[J:2 * J].tolist() == [1.0] * J and c[2 * J + 2:].tolist() == [1.0, 0.0]


def test_masked_sums_at_a_million_poses():
    """All-ones mask: the unmasked kernel's sums in the masked layout (up to summation order); 20 % of joints off: the same
    sums for any batch split."""
    B, J = 1 << 20, 17
    pred, gt = _poses(B, J, 3)
    plain = metric.PmpjpeAccumulator(J)
    plain.update(*_cuda(pred, gt))
    a = plain.acc.cpu().numpy()
    want = np.concatenate([a[:J], np.full(J, B), a[J:J + 2], [B, 0]])
    np.testing.assert_allclose(_masked(pred, gt, np.ones((B, J), np.float32)).acc.cpu().numpy(), want, rtol=1e-12)
    np.testing.assert_allclose(_masked(pred, gt, None).acc.cpu().numpy(), want, rtol=1e-12)
    pred, gt, mask = _masked_inputs(B, J, 4)
    whole = _masked(pred, gt, mask).acc.cpu().numpy()
    k = 300001
    parts = metric.PmpjpeAccumulator(J, masked=True)
    for s in (slice(0, k), slice(k, B)):
        parts.update(*_cuda(pred[s], gt[s]), mask=_cuda(mask[s])[0])
    np.testing.assert_allclose(parts.acc.cpu().numpy(), whole, rtol=1e-12)
    assert whole[2 * J + 3] > 0


@pytest.mark.parametrize("B", [32, 4097])
def test_values_under_masked_joints_change_nothing(B):
    """Bitwise within one warp's poses (one atomic per address); to the summation order beyond."""
    J, G = 17, 4
    pred, gt, mask = _masked_inputs(B, J, 11)
    group = _groups(B, G, "unlabelled", 12)
    base = _masked(pred, gt, mask, group, G).acc.cpu().numpy()
    rng = np.random.default_rng(13)
    for fill in (0.0, 1e30, -np.inf, None):
        p, g = pred.copy(), gt.copy()
        off = mask == 0
        p[off] = rng.normal(size=p[off].shape) if fill is None else fill
        g[off] = rng.normal(size=g[off].shape) if fill is None else fill
        got = _masked(p, g, mask, group, G).acc.cpu().numpy()
        if B == 32:
            assert got.tobytes() == base.tobytes()
        else:
            np.testing.assert_allclose(got, base, rtol=1e-13)
    m3 = np.repeat(mask[:, :, None], 3, axis=2)
    m3[:, :, 1] *= 1 + rng.random((B, J)).astype(np.float32)                   # any positive value counts as used
    np.testing.assert_allclose(_masked(pred, gt, m3, group, G).acc.cpu().numpy(), base, rtol=1e-13)


@pytest.mark.parametrize("G,J", [(15, 17), (15, 40), (4096, 17)])
def test_both_entry_points_replay_from_a_cuda_graph_and_ignore_the_batch_split(G, J):
    B = 20000
    pred, gt, mask = _masked_inputs(B, J, G + J)
    gt_m = np.nan_to_num(gt, posinf=0.0)
    pred_m = np.nan_to_num(pred)
    group = _groups(B, G, "unlabelled", 3)
    conf = (mask > 0).astype(np.float32)
    p, g, pm, gm, m, c, grp = _cuda(pred, gt, pred_m, gt_m, mask, conf, group.astype(np.int32))
    ma = metric.MpjpeAccumulator(J, num_groups=G)
    pa = metric.PmpjpeAccumulator(J, num_groups=G)
    ma.update(pm, gm, c, group=grp)
    pa.update(p, g, mask=m, group=grp)
    eager = [ma.acc.clone(), pa.acc.clone()]
    ma.acc.zero_()
    pa.acc.zero_()
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            ma.update(pm, gm, c, group=grp)
            pa.update(p, g, mask=m, group=grp)
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(2):
        graph.replay()
    torch.cuda.synchronize()
    for a, e in zip((ma.acc, pa.acc), eager):
        np.testing.assert_allclose(a.cpu().numpy(), 2 * e.cpu().numpy(), rtol=1e-12, atol=1e-300)
    # split at a point that is not a multiple of any tile or warp
    ma2 = metric.MpjpeAccumulator(J, num_groups=G)
    pa2 = metric.PmpjpeAccumulator(J, num_groups=G)
    for sl in (slice(0, 7777), slice(7777, B)):
        ma2.update(pm[sl], gm[sl], c[sl], group=grp[sl])
        pa2.update(p[sl], g[sl], mask=m[sl], group=grp[sl])
    np.testing.assert_allclose(ma2.acc.cpu().numpy(), eager[0].cpu().numpy(), rtol=1e-12, atol=1e-300)
    np.testing.assert_allclose(pa2.acc.cpu().numpy(), eager[1].cpu().numpy(), rtol=1e-12, atol=1e-300)


def test_evaluation_reports_the_pmpjpe_of_the_triangulations():
    kw = dict(arch="cmu0", views=4, poses=2000, precision="fp32", pixel_noise=2, outlier_rate=0.1, triangulate=True,
              triangulate_robust=True)
    line = evaluate.run(**kw, triangulation_pmpjpe=True, refine_triangulations=True)
    pix, target, calib = inputs.synth_project(2000, synth.make_rig(4, "cmu"), seed=1, start=0)
    inputs.add_detector_noise(pix, calib, 1, 0, 2.0, 0.1, 0.0)
    lin, used = inputs.triangulate(pix, calib)
    rob, inl = inputs.triangulate_robust(pix, calib, inlier_px=10.0)
    tgt = target.cpu().numpy()
    for entry, pts, mask in (("triangulation", lin, used >= 2), ("triangulation_robust", rob, inl != 0)):
        pa = line[entry]["procrustes_aligned"]
        assert set(pa) == {"p_mpjpe_cm", "aligned_poses", "skipped_poses"}
        assert pa["aligned_poses"] + pa["skipped_poses"] == 2000 and np.isfinite(pa["p_mpjpe_cm"])
        want = metric.finalize_pmpjpe_masked(mpo.masked_pmpjpe_sums(pts.cpu().numpy(), tgt, mask.cpu().numpy())[0], 17)
        assert abs(pa["p_mpjpe_cm"] - want["p_mpjpe"]) <= 1e-7 * want["p_mpjpe"]
        assert (pa["aligned_poses"], pa["skipped_poses"]) == (want["aligned"], want["skipped"])
        assert set(line[entry]["refined"]["procrustes_aligned"]) == set(pa)
    plain = evaluate.run(**kw)
    assert set(plain) == {"metric", "value", "unit", "n_gpus", "ms_total", "poses", "dtype", "data", "config", "mpjpe_cm",
                          "tflops", "triangulation", "triangulation_robust"}
    for entry in ("triangulation", "triangulation_robust"):
        assert set(plain[entry]) == {"mpjpe_cm", "under_determined_joints", "method", "note"}
    with pytest.raises(ValueError, match="triangulation_pmpjpe"):
        evaluate.run(arch="cmu0", views=4, poses=100, triangulation_pmpjpe=True)
