"""CPU checks of the grouped / masked metric sums (ABI 7): the numpy oracle agrees with the reference-pinned sums where
they overlap, ignores whatever lies under a masked joint, skips the poses it must skip, and its group blocks add up to the
ungrouped sums.  The two C entry points reject every bad argument before any CUDA call, the wrappers reject bad group and
mask shapes, and a grouped accumulator all-reduces every block over two gloo ranks."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

import masked_pmpjpe_oracle as mpo
from openmpl_b200 import _lib, metric
from oracle import mpl_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _poses(B, J=17, seed=0, noise=0.03):
    rng = np.random.default_rng(seed)
    gt = rng.standard_normal((B, J, 3)).astype(np.float32)
    pred = (gt @ np.linalg.qr(rng.standard_normal((3, 3)))[0] * 1.1 + noise * rng.standard_normal((B, J, 3)) + 0.2)
    return pred.astype(np.float32), gt


def rank_batch(rank):
    """The batch of one rank of the two-rank test: groups with -1 entries, a random mask."""
    pred, gt = _poses(23 + 6 * rank, seed=10 + rank)
    rng = np.random.default_rng(50 + rank)
    return pred, gt, rng.integers(-1, 5, len(pred)), (rng.random(gt.shape[:2]) > 0.2).astype(np.float32)


@pytest.mark.parametrize("scaling", [True, False])
@pytest.mark.parametrize("reflection", ["best", False, True])
def test_every_joint_used_is_the_unmasked_sums(scaling, reflection):
    pred, gt = _poses(40)
    want = mpo.pmpjpe_sums_in_masked_layout(pred, gt, scaling=scaling, reflection=reflection)
    for mask in (None, np.ones(gt.shape[:2], np.float32)):
        got = mpo.masked_pmpjpe_sums(pred, gt, mask, scaling=scaling, reflection=reflection)[0]
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-12)
    r = metric.finalize_pmpjpe_masked(want, 17)
    assert abs(r["p_mpjpe"] - metric.finalize_pmpjpe(mpl_oracle.pmpjpe_sums(pred, gt, scaling=scaling, reflection=reflection),
                                                     17)["p_mpjpe"]) < 1e-12


def test_values_under_masked_joints_change_nothing():
    pred, gt = _poses(30, seed=1)
    mask = (np.random.default_rng(2).random(gt.shape[:2]) > 0.3).astype(np.float32)
    want = mpo.masked_pmpjpe_sums(pred, gt, mask)
    for fill in (np.nan, np.inf, -np.inf, 1e6):
        p, g = pred.copy(), gt.copy()
        p[mask == 0] = fill
        g[mask == 0, 1] = -fill
        np.testing.assert_array_equal(mpo.masked_pmpjpe_sums(p, g, mask), want)
    # a non-finite coordinate disables its joint even where the mask is 1
    p = pred.copy()
    p[mask == 0] = np.nan
    np.testing.assert_array_equal(mpo.masked_pmpjpe_sums(p, gt, None), want)


def test_too_few_joints_or_coincident_points_are_skipped():
    pred, gt = _poses(4, seed=3)
    mask = np.ones(gt.shape[:2], np.float32)
    mask[0, 2:] = 0                                      # two used joints
    gt[1] = gt[1, :1]                                    # every target joint at one point
    pred[2] = 5.0                                        # every predicted joint at one point
    acc = mpo.masked_pmpjpe_sums(pred, gt, mask)[0]
    J = 17
    assert acc[2 * J + 2] == 1 and acc[2 * J + 3] == 3
    np.testing.assert_array_equal(acc[J:2 * J], np.ones(J))
    mask[3, 3:] = 0                                      # exactly three used joints: aligned
    acc = mpo.masked_pmpjpe_sums(pred, gt, mask)[0]
    assert acc[2 * J + 2] == 1 and acc[J:J + 3].tolist() == [1, 1, 1] and acc[J + 3] == 0


def test_group_blocks_add_up_and_out_of_range_groups_are_ignored():
    pred, gt = _poses(50, seed=4)
    rng = np.random.default_rng(5)
    group = rng.integers(-2, 7, 50)                      # -2, -1, 5, 6 fall outside [0, 5)
    conf = (rng.random(gt.shape[:2]) > 0.2).astype(np.float32)
    keep = (group >= 0) & (group < 5)
    m = mpo.grouped_metric_sums(pred, gt, group, 5, conf)
    np.testing.assert_allclose(m.sum(0), mpl_oracle.metric_sums(pred[keep], gt[keep], conf[keep]), rtol=1e-12)
    assert m[:, -1].tolist() == [float((group == g).sum()) for g in range(5)]
    p = mpo.masked_pmpjpe_sums(pred, gt, conf, group, 5)
    np.testing.assert_allclose(p.sum(0), mpo.masked_pmpjpe_sums(pred[keep], gt[keep], conf[keep])[0], rtol=1e-12)
    np.testing.assert_array_equal(mpo.grouped_metric_sums(pred, gt, None, 1), mpl_oracle.metric_sums(pred, gt)[None])


def _call_grouped(**kw):
    a = dict(pred=8, gt=8, conf=None, group=8, G=2, B=4, J=17, unit=100.0, room=None, acc=8)
    a.update(kw)
    return _lib.lib().mpl_mpjpe_accumulate_grouped(a["pred"], a["gt"], a["conf"], a["group"], a["G"], a["B"], a["J"],
                                                   a["unit"], a["room"], a["acc"], None)


def _call_masked(**kw):
    a = dict(pred=8, gt=8, mask=None, group=8, G=2, B=4, J=17, unit=100.0, scaling=1, reflection=-1, acc=8)
    a.update(kw)
    return _lib.lib().mpl_pmpjpe_accumulate_masked(a["pred"], a["gt"], a["mask"], a["group"], a["G"], a["B"], a["J"],
                                                   a["unit"], a["scaling"], a["reflection"], a["acc"], None)


BAD = [dict(G=0), dict(G=-1), dict(G=65537), dict(group=None), dict(pred=None), dict(gt=None), dict(acc=None), dict(B=-1),
       dict(J=0), dict(J=-3), dict(B=0, acc=None)]


@pytest.mark.parametrize("bad", BAD, ids=[",".join(f"{k}={v}" for k, v in b.items()) for b in BAD])
def test_entry_points_reject_bad_arguments_before_any_cuda_call(bad):
    # with pointers that are not device memory: an accepted call would reach CUDA and fail differently (or fault)
    assert _call_grouped(**bad) == _lib.MPL_ERR_INVALID_ARGUMENT
    assert b"mpl_mpjpe_accumulate_grouped" in _lib.lib().mpl_last_error()
    assert _call_masked(**bad) == _lib.MPL_ERR_INVALID_ARGUMENT
    assert b"mpl_pmpjpe_accumulate_masked" in _lib.lib().mpl_last_error()


@pytest.mark.parametrize("reflection", [-2, 2])
def test_masked_entry_point_rejects_a_bad_reflection(reflection):
    assert _call_masked(reflection=reflection) == _lib.MPL_ERR_INVALID_ARGUMENT


def test_batch_zero_and_one_group_without_labels_are_accepted_without_cuda():
    assert _call_grouped(B=0) == _lib.MPL_OK and _call_masked(B=0) == _lib.MPL_OK
    assert _call_grouped(B=0, group=None, G=1) == _lib.MPL_OK and _call_masked(B=0, group=None, G=1) == _lib.MPL_OK


def test_wrappers_reject_bad_group_and_mask_shapes():
    pred = torch.zeros(4, 17, 3)
    for bad in (65537, 0):
        with pytest.raises(ValueError, match="num_groups"):
            metric.MpjpeAccumulator(17, device="cpu", num_groups=bad)
    acc = metric.MpjpeAccumulator(17, device="cpu", num_groups=3)
    for g in (None, torch.zeros(3, dtype=torch.int64), torch.zeros(4, 1, dtype=torch.int64), torch.zeros(4)):
        with pytest.raises(ValueError, match="group"):
            acc.update(pred, pred, group=g)
    with pytest.raises(ValueError, match="group"):
        metric.MpjpeAccumulator(17, device="cpu").update(pred, pred, group=torch.zeros(4, dtype=torch.int64))
    pacc = metric.PmpjpeAccumulator(17, device="cpu", masked=True)
    for m in (torch.ones(4, 16), torch.ones(3, 17), torch.ones(4, 17, 2), torch.ones(4), torch.ones(4, 17, 3, 1)):
        with pytest.raises(ValueError, match="mask"):
            pacc.update(pred, pred, mask=m)
    with pytest.raises(ValueError, match="mask"):
        metric.PmpjpeAccumulator(17, device="cpu").update(pred, pred, mask=torch.ones(4, 17))
    with pytest.raises(ValueError, match="group"):
        metric.PmpjpeAccumulator(17, device="cpu", num_groups=2).update(pred, pred, group=torch.zeros(5, dtype=torch.int32))
    assert pacc.acc.shape == (38,) and metric.PmpjpeAccumulator(17, device="cpu", num_groups=2).acc.shape == (2, 38)


def test_mask_with_three_values_per_joint_needs_all_three():
    m = torch.ones(2, 17, 3)
    m[0, 4, 1] = 0
    got = metric._mask_arg(m, 2, 17, "cpu")
    assert got.dtype == torch.float32 and got.shape == (2, 17)
    assert float(got[0, 4]) == 0 and float(got.sum()) == 33


def test_grouped_results_give_per_group_dicts_and_the_unweighted_mean():
    pred, gt = _poses(60, seed=6)
    group = np.random.default_rng(7).integers(0, 3, 60)
    group[group == 1] = 2                               # group 1 stays empty
    acc = metric.MpjpeAccumulator(17, device="cpu", num_groups=3)
    acc.acc += torch.from_numpy(mpo.grouped_metric_sums(pred, gt, group, 3))
    res = acc.result(names=["a", "b", "c"])
    whole = metric.finalize(mpl_oracle.metric_sums(pred, gt), 17)
    assert res["n"] == 60 and abs(res["mpjpe_abs"] - whole["mpjpe_abs"]) < 1e-12
    assert [g["group"] for g in res["groups"]] == ["a", "b", "c"] and res["groups"][1]["n"] == 0
    for k in ("mpjpe_abs", "mpjpe_rel"):
        want = np.mean([mpl_oracle.evaluate(pred[group == g], gt[group == g], relative=k == "mpjpe_rel")["mpjpe"] for g in (0, 2)])
        assert abs(res["group_mean"][k] - want) < 1e-10
    pacc = metric.PmpjpeAccumulator(17, device="cpu", num_groups=3)
    pacc.acc += torch.from_numpy(mpo.masked_pmpjpe_sums(pred, gt, None, group, 3))
    pres = pacc.result()
    assert pres["aligned"] == 60 and pres["skipped"] == 0 and pres["groups"][1]["n"] == 0
    want = np.mean([metric.finalize_pmpjpe(mpl_oracle.pmpjpe_sums(pred[group == g], gt[group == g]), 17)["p_mpjpe"]
                    for g in (0, 2)])
    assert abs(pres["group_mean"]["p_mpjpe"] - want) < 1e-10


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_two_rank_all_reduce_reduces_every_group_block(tmp_path):
    G = 5
    out = tmp_path / "grouped.json"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "grouped_dist_worker.py"), str(out), str(G)]
    r = subprocess.run(cmd, cwd=ROOT, env=dict(os.environ, OMP_NUM_THREADS="2"), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    d = json.load(open(out))
    batches = [rank_batch(k) for k in range(2)]
    pred, gt, group, mask = (np.concatenate([b[i] for b in batches]) for i in range(4))
    np.testing.assert_allclose(d["mpjpe"], mpo.grouped_metric_sums(pred, gt, group, G), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(d["pmpjpe"], mpo.masked_pmpjpe_sums(pred, gt, mask, group, G), rtol=1e-12, atol=1e-12)
    assert all(np.asarray(d["mpjpe"])[:, -1] > 0)
