"""K6 host side: MPJPE accumulators on the device + their reduction over ranks.

Mirrors `evaluate()` of the reference (`MPL/lib/core/function_mpl.py:670-687`) and `calc_mpjpe` /
`calc_distance_per_dim` (`MPL/lib/core/evaluate.py:91-125`): unit rule (x100 when OUTPUT_IN_METER), root-relative
variant, `joints_3d_conf <= 0` masking with NaN semantics.  Predictions never leave the GPU: each batch adds into
`11 J + 1` fp64 running sums (layout in include/mpl_b200.h) and ranks are combined with ONE all-reduce at the end.
`PmpjpeAccumulator` does the same for the Procrustes-aligned error (`MPL/lib/utils/pose_utils.py:61-143`).

With `num_groups=G` both keep one block of sums per group (`[G, L]`), and `update(..., group=...)` says which block each
pose adds into (e.g. the H36M action): `result()` then adds a finalised dict per group and their unweighted mean, the
"average" row of a per-action table.  `PmpjpeAccumulator(masked=True)` aligns each pose on the joints its mask marks.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib


def acc_len(J: int) -> int:
    return 11 * J + 1


def pmetric_masked_len(J: int) -> int:
    return 2 * J + 4


MAX_GROUPS = 65536


def _check_num_groups(num_groups):
    if num_groups is not None and not 1 <= int(num_groups) <= MAX_GROUPS:
        raise ValueError(f"num_groups must be in [1, {MAX_GROUPS}], got {num_groups}")


def _group_arg(group, num_groups, B, device):
    """group -> a contiguous int32 [B] tensor on the device (None without num_groups); required iff num_groups is set."""
    if num_groups is None:
        if group is not None:
            raise ValueError("group given to an accumulator built without num_groups")
        return None
    if group is None:
        raise ValueError("an accumulator built with num_groups needs group=[B] in every update")
    group = torch.as_tensor(group)
    if group.dim() != 1 or group.shape[0] != B:
        raise ValueError(f"group must have shape [{B}], got {tuple(group.shape)}")
    if group.dtype.is_floating_point or group.dtype == torch.bool:
        raise ValueError(f"group must be an integer tensor, got {group.dtype}")
    return group.to(device, torch.int32).contiguous()


def _group_results(blocks: np.ndarray, finalize_one, names, keys) -> tuple[list, dict]:
    """Per-group finalised dicts (labelled by `names`) and the unweighted mean of `keys` over groups with n > 0."""
    if names is not None and len(names) != len(blocks):
        raise ValueError(f"names has {len(names)} entries for {len(blocks)} groups")
    groups = []
    for g, blk in enumerate(blocks):
        r = finalize_one(blk)
        r["group"] = names[g] if names is not None else g
        groups.append(r)
    filled = [r for r in groups if r["n"] > 0]
    mean = {k: float(np.mean([r[k] for r in filled])) if filled else float("nan") for k in keys}
    mean["groups"] = len(filled)
    return groups, mean


class MpjpeAccumulator:
    def __init__(self, num_joints: int = 17, output_in_meter: bool = True, device=None, num_groups: int | None = None):
        _check_num_groups(num_groups)
        self.J = num_joints
        self.unit = 100.0 if output_in_meter else 1.0
        self.num_groups = None if num_groups is None else int(num_groups)
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        shape = (acc_len(num_joints),) if num_groups is None else (self.num_groups, acc_len(num_joints))
        self.acc = torch.zeros(shape, dtype=torch.float64, device=self.device)

    def update(self, pred: torch.Tensor, gt: torch.Tensor, conf3d: torch.Tensor | None = None, room: dict | None = None,
               group: torch.Tensor | None = None):
        """pred, gt: [B, J, 3] fp32 on the device; conf3d: None, [B, J], [B, J, 1] or [B, J, 3] (the dataset's
        `joints_3d_conf`, `function_mpl.py:489-490,682-684`).  room: the `meta` entries of a room-normalised dataset --
        {'room_x_scale', 'room_center'} when 'room_scaled_equal', else {'room_x_scale', 'room_y_scale'} -- for the
        un-scaling `validate()` applies before it stores predictions and targets (`function_mpl.py:476-488`).
        group: [B] integers (any device), required iff the accumulator has num_groups: the block each pose adds into; a
        value outside [0, num_groups) drops the pose."""
        B = pred.shape[0]
        group = _group_arg(group, self.num_groups, B, self.device)
        affine = None
        if room is not None:
            if "room_center" in room:                     # 'room_scaled_equal': v * s + centre on every axis
                s = float(room["room_x_scale"])
                c = [float(x) for x in room["room_center"]]
                vals = [s, s, s] + c
            else:                                         # x and y scaled separately, z untouched
                vals = [float(room["room_x_scale"]), float(room["room_y_scale"]), 1.0, 0.0, 0.0, 0.0]
            import ctypes
            affine = (ctypes.c_float * 6)(*vals)
        pred = pred.to(self.device, torch.float32).contiguous()
        gt = gt.to(self.device, torch.float32).contiguous()
        if conf3d is not None:
            c = conf3d.to(self.device, torch.float32)
            if c.dim() == 2:
                c = c[:, :, None]
            conf3d = c.expand(B, self.J, 3).contiguous()
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            conf_ptr = conf3d.data_ptr() if conf3d is not None else None
            if group is None:
                _lib.check(_lib.lib().mpl_mpjpe_accumulate(pred.data_ptr(), gt.data_ptr(), conf_ptr, B, self.J, self.unit,
                                                           affine, self.acc.data_ptr(), stream))
            else:
                _lib.check(_lib.lib().mpl_mpjpe_accumulate_grouped(pred.data_ptr(), gt.data_ptr(), conf_ptr, group.data_ptr(),
                                                                   self.num_groups, B, self.J, self.unit, affine,
                                                                   self.acc.data_ptr(), stream))

    def all_reduce(self):
        """Sum the accumulators over all ranks (NCCL over NVLink on the GPU box; one call of `11 J + 1` doubles, or of the
        whole [G, 11 J + 1] tensor when grouped)."""
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(self.acc, op=dist.ReduceOp.SUM)
        return self

    def result(self, names=None) -> dict:
        """The finalised sums.  Grouped: the top-level keys come from the sum over groups; "groups" holds one dict per
        group (its "group" is names[g] if given, else g) and "group_mean" the unweighted mean over groups with n > 0 of
        mpjpe_abs and mpjpe_rel."""
        acc = self.acc.detach().cpu().numpy()
        if self.num_groups is None:
            return finalize(acc, self.J)
        out = finalize(acc.sum(axis=0), self.J)
        out["groups"], out["group_mean"] = _group_results(acc, lambda a: finalize(a, self.J), names, ("mpjpe_abs", "mpjpe_rel"))
        return out


def _mask_arg(mask, B, J, device):
    """mask [B, J], [B, J, 1] or [B, J, 3] -> contiguous fp32 [B, J] on the device, > 0 where the joint is used.  Three
    values per joint: used iff all three are > 0 (MPJPE's per-coordinate rule)."""
    mask = torch.as_tensor(mask)
    if mask.dim() not in (2, 3) or tuple(mask.shape[:2]) != (B, J) or (mask.dim() == 3 and mask.shape[2] not in (1, 3)):
        raise ValueError(f"mask must be [{B}, {J}], [{B}, {J}, 1] or [{B}, {J}, 3], got {tuple(mask.shape)}")
    mask = mask.to(device)
    if mask.dim() == 3:
        mask = (mask > 0).all(dim=2)
    return mask.to(torch.float32).contiguous()


class PmpjpeAccumulator:
    """Procrustes-aligned MPJPE (P-MPJPE): every prediction is first aligned to its ground truth with
    `PoseUtils.procrustes` of the reference (`MPL/lib/utils/pose_utils.py:61-143`; similarity transform, reflection
    'best' by default), then scored like `calc_mpjpe`.  `J + 3` fp64 running sums on the device, one all-reduce.

    With masked=True or num_groups set it keeps the `2 J + 4` sums of `mpl_pmpjpe_accumulate_masked` per group instead:
    each pose is aligned on its used joints only (mask > 0 and finite), and poses with fewer than 3 of them, or with
    coincident points, are counted as skipped."""

    REFLECTION = {"best": -1, False: 0, True: 1}

    def __init__(self, num_joints: int = 17, output_in_meter: bool = True, scaling: bool = True, reflection="best",
                 device=None, num_groups: int | None = None, masked: bool = False):
        _check_num_groups(num_groups)
        self.J = num_joints
        self.unit = 100.0 if output_in_meter else 1.0
        self.scaling = bool(scaling)
        self.reflection = self.REFLECTION[reflection]
        self.num_groups = None if num_groups is None else int(num_groups)
        self.masked = bool(masked) or num_groups is not None
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        if not self.masked:
            shape = (num_joints + 3,)
        elif num_groups is None:
            shape = (pmetric_masked_len(num_joints),)
        else:
            shape = (self.num_groups, pmetric_masked_len(num_joints))
        self.acc = torch.zeros(shape, dtype=torch.float64, device=self.device)

    def update(self, pred: torch.Tensor, gt: torch.Tensor, mask: torch.Tensor | None = None, group: torch.Tensor | None = None):
        """pred, gt: [B, J, 3] fp32 on the device.  mask (masked accumulators only): None, [B, J], [B, J, 1] or [B, J, 3],
        e.g. the dataset's `joints_3d_conf`; group: [B] integers, required iff the accumulator has num_groups."""
        B = pred.shape[0]
        if mask is not None and not self.masked:
            raise ValueError("mask given to an accumulator built without masked=True or num_groups")
        group = _group_arg(group, self.num_groups, B, self.device)
        mask = _mask_arg(mask, B, self.J, self.device) if mask is not None else None
        pred = pred.to(self.device, torch.float32).contiguous()
        gt = gt.to(self.device, torch.float32).contiguous()
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device).cuda_stream
            if not self.masked:
                _lib.check(_lib.lib().mpl_pmpjpe_accumulate(pred.data_ptr(), gt.data_ptr(), B, self.J, self.unit,
                                                            int(self.scaling), self.reflection, self.acc.data_ptr(), stream))
            else:
                _lib.check(_lib.lib().mpl_pmpjpe_accumulate_masked(
                    pred.data_ptr(), gt.data_ptr(), None if mask is None else mask.data_ptr(),
                    None if group is None else group.data_ptr(), self.num_groups or 1, B, self.J, self.unit,
                    int(self.scaling), self.reflection, self.acc.data_ptr(), stream))

    def all_reduce(self):
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(self.acc, op=dist.ReduceOp.SUM)
        return self

    def result(self, names=None) -> dict:
        """Unmasked: finalize_pmpjpe.  Masked: finalize_pmpjpe_masked of the sum over groups, and when grouped "groups"
        (one dict per group, labelled by names) and "group_mean" (the unweighted mean of p_mpjpe over groups with n > 0)."""
        acc = self.acc.detach().cpu().numpy()
        if not self.masked:
            return finalize_pmpjpe(acc, self.J)
        if self.num_groups is None:
            return finalize_pmpjpe_masked(acc, self.J)
        out = finalize_pmpjpe_masked(acc.sum(axis=0), self.J)
        out["groups"], out["group_mean"] = _group_results(acc, lambda a: finalize_pmpjpe_masked(a, self.J), names, ("p_mpjpe",))
        return out


def finalize_pmpjpe_masked(acc: np.ndarray, J: int) -> dict:
    """`2 J + 4` masked sums -> pjpe_aligned[j] = sum_j / count_j, p_mpjpe = their mean over joints with count_j > 0 (with
    every joint used: finalize_pmpjpe's value), mean d and scale over the aligned poses, and the pose counts.  n is the
    number of aligned poses."""
    acc = np.asarray(acc, dtype=np.float64)
    cnt = acc[J:2 * J]
    na = acc[2 * J + 2]
    with np.errstate(invalid="ignore", divide="ignore"):
        pj = acc[0:J] / cnt
        out = {"n": int(round(na)), "aligned": int(round(na)), "skipped": int(round(acc[2 * J + 3])), "pjpe_aligned": pj,
               "joint_count": cnt.copy(), "residual": float(acc[2 * J] / na), "scale": float(acc[2 * J + 1] / na)}
    seen = cnt > 0
    out["p_mpjpe"] = float(pj[seen].mean()) if seen.any() else float("nan")
    return out


def finalize_pmpjpe(acc: np.ndarray, J: int) -> dict:
    """Running sums -> per-joint P-MPJPE, its mean, mean normalised residual d and mean scale."""
    acc = np.asarray(acc, dtype=np.float64)
    n = acc[J + 2]
    with np.errstate(invalid="ignore", divide="ignore"):
        out = {"n": int(round(n)), "pjpe_aligned": acc[0:J] / n, "residual": float(acc[J] / n), "scale": float(acc[J + 1] / n)}
    out["p_mpjpe"] = float(out["pjpe_aligned"].mean())
    return out


def finalize(acc: np.ndarray, J: int) -> dict:
    """Running sums -> the quantities `evaluate()` logs: per-joint MPJPE, its mean, per-dim distances."""
    acc = np.asarray(acc, dtype=np.float64)
    n = acc[11 * J]
    cnt = acc[8 * J:11 * J].reshape(J, 3)
    with np.errstate(invalid="ignore", divide="ignore"):
        out = {
            "n": int(round(n)),
            "pjpe_abs": acc[0:J] / n,
            "pjpe_rel": acc[J:2 * J] / n,
            "dist_abs": acc[2 * J:5 * J].reshape(J, 3) / cnt,      # nanmean over unmasked entries
            "dist_rel": acc[5 * J:8 * J].reshape(J, 3) / cnt,
        }
    out["mpjpe_abs"] = float(out["pjpe_abs"].mean())
    out["mpjpe_rel"] = float(out["pjpe_rel"].mean())
    return out
