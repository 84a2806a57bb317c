"""numpy fp64 restatement of the grouped metric sums of include/mpl_b200.h (ABI 7): mpl_mpjpe_accumulate_grouped as
`mpl_oracle.metric_sums` per group subset, and mpl_pmpjpe_accumulate_masked on top of the reference-pinned
`mpl_oracle.procrustes` applied to each pose's used joints."""
import numpy as np

from oracle import mpl_oracle


def used_joints(pred, gt, mask=None):
    """[B, J] bool: (mask is None or mask > 0) and the six coordinates finite."""
    pred = np.asarray(pred, dtype=np.float64)
    gt = np.asarray(gt, dtype=np.float64)
    use = np.isfinite(pred).all(-1) & np.isfinite(gt).all(-1)
    if mask is not None:
        use &= np.asarray(mask) > 0
    return use


def grouped_metric_sums(pred, gt, group, num_groups, conf_3d=None, output_in_meter=True):
    """[G, 11 J + 1]: block g is metric_sums over the poses with group == g; other groups add nothing."""
    pred = np.asarray(pred, dtype=np.float32)
    B, J, _ = pred.shape
    group = np.zeros(B, np.int64) if group is None else np.asarray(group)
    out = np.zeros((num_groups, 11 * J + 1))
    for g in range(num_groups):
        sel = group == g
        if sel.any():
            c = None if conf_3d is None else np.asarray(conf_3d)[sel]
            out[g] = mpl_oracle.metric_sums(pred[sel], np.asarray(gt)[sel], c, output_in_meter)
    return out


def masked_pmpjpe_sums(pred, gt, mask=None, group=None, num_groups=1, output_in_meter=True, scaling=True, reflection="best"):
    """[G, 2 J + 4] in the layout of MPL_PMETRIC_MASKED_ACC_LEN: per aligned pose, procrustes(gt[used], pred[used])."""
    pred = np.array(pred, dtype=np.float64)
    gt = np.array(gt, dtype=np.float64)
    B, J, _ = pred.shape
    use = used_joints(pred, gt, mask)
    if output_in_meter:
        pred, gt = pred * 100, gt * 100
    group = np.zeros(B, np.int64) if group is None else np.asarray(group)
    acc = np.zeros((num_groups, 2 * J + 4))
    for b in range(B):
        g = int(group[b])
        if not 0 <= g < num_groups:
            continue
        u = use[b]
        A, Bp = gt[b][u], pred[b][u]
        if u.sum() < 3 or ((A - A.mean(0)) ** 2).sum() <= 0 or ((Bp - Bp.mean(0)) ** 2).sum() <= 0:
            acc[g, 2 * J + 3] += 1
            continue
        d, Z, tf = mpl_oracle.procrustes(A, Bp, scaling, reflection)
        acc[g, np.flatnonzero(u)] += np.sqrt(((Z - A) ** 2).sum(-1))
        acc[g, J + np.flatnonzero(u)] += 1
        acc[g, 2 * J] += d
        acc[g, 2 * J + 1] += tf["scale"] if scaling else 1.0
        acc[g, 2 * J + 2] += 1
    return acc


def pmpjpe_sums_in_masked_layout(pred, gt, **kw):
    """mpl_oracle.pmpjpe_sums (every joint used) restated in the masked layout."""
    s = mpl_oracle.pmpjpe_sums(pred, gt, **kw)
    J = len(s) - 3
    return np.concatenate([s[:J], np.full(J, s[J + 2]), s[J:J + 2], [s[J + 2], 0.0]])
