"""N2: batched input builder — raw detector output + calibrations -> the model's (poses, rays, centers).

Replaces the per-sample numpy of `JointsDataset_MPL.__getitem__`
(`MPL/lib/dataset/joints_dataset_mpl.py:615-648,701-715,762-772,817-820,872-904`) with one streaming kernel.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import _lib


def pack_calibration(R, t, f, c, image_size) -> np.ndarray:
    """[..., V, 18] float64 rows: R (9, row-major world->cam), t (3), fx, fy, cx, cy, w, h.

    R [..., V, 3, 3], t [..., V, 3], f and c [..., V, 2]; leading batch dimensions give one calibration per pose (a
    [B, V, 18] result is what the calibration-taking entry points accept per pose).  image_size (w, h), or any array that
    broadcasts to [..., V, 2].
    """
    R, t, f, c = (np.asarray(a, dtype=np.float64) for a in (R, t, f, c))
    lead = R.shape[:-2]
    wh = np.broadcast_to(np.asarray(image_size, dtype=np.float64), lead + (2,))
    return np.concatenate([R.reshape(lead + (9,)), t.reshape(lead + (3,)), f.reshape(lead + (2,)), c.reshape(lead + (2,)), wh],
                          axis=-1)


def build_inputs(pix: torch.Tensor, calib) -> tuple:
    """pix [B, V, J, 3] fp32 (u, v, conf) pixels on the device; calib [V, 18], or [B, V, 18] with one calibration per pose
    -> poses, rays [B,V,J,3], centers [B,V,1,3]."""
    B, V, J, _ = pix.shape
    device = pix.device
    pix = pix.to(torch.float32).contiguous()
    calib, stride = _calib_arg(calib, B, V, device)
    poses = torch.empty((B, V, J, 3), dtype=torch.float32, device=device)
    rays = torch.empty_like(poses)
    centers = torch.empty((B, V, 1, 3), dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device).cuda_stream
        _lib.check(_lib.lib().mpl_build_inputs_strided(pix.data_ptr(), calib.data_ptr(), stride, B, V, J, poses.data_ptr(),
                                                       rays.data_ptr(), centers.data_ptr(), stream))
    return poses, rays, centers


def triangulate(pix: torch.Tensor, calib, min_conf: float = 0.0) -> tuple:
    """Linear multi-view triangulation of raw detections (`mpl_triangulate`; the baseline of
    `MPL/lib/multiviews/triangulate.py:59-115`), enqueued on the current stream.

    pix [B, V, J, 3] fp32 (u, v, conf) pixels on the device; calib [V, 18] or [B, V, 18] (numpy or tensor) as for
    `build_inputs`.  A view is used for a joint iff conf > min_conf and the pixel lies strictly inside the image.  Returns
    (points [B, J, 3] fp32 world units, NaN where fewer than 2 views are used; views_used [B, J] int32).
    """
    B, V, J, _ = pix.shape
    device = pix.device
    pix = pix.to(torch.float32).contiguous()
    calib, stride = _calib_arg(calib, B, V, device)
    points = torch.empty((B, J, 3), dtype=torch.float32, device=device)
    views_used = torch.empty((B, J), dtype=torch.int32, device=device)
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device).cuda_stream
        _lib.check(_lib.lib().mpl_triangulate_strided(pix.data_ptr(), calib.data_ptr(), stride, B, V, J, float(min_conf),
                                                      points.data_ptr(), views_used.data_ptr(), stream))
    return points, views_used


def triangulate_robust(pix: torch.Tensor, calib, min_conf: float = 0.0, inlier_px: float = 10.0) -> tuple:
    """Outlier-robust triangulation of raw detections (`mpl_triangulate_robust`), enqueued on the current stream.

    calib [V, 18] or [B, V, 18]; candidate views as in `triangulate`.  Every candidate pair gives a two-view DLT hypothesis scored by the MSAC cost
    sum_c min(e_c^2, inlier_px^2) over the candidates' pixel reprojection errors; the cheapest one's inliers (e_c < inlier_px)
    are refitted by a DLT with rows weighted by conf.  Returns (points [B, J, 3] fp32 world units, NaN where fewer than two
    candidates or inliers; inliers [B, J] int32 bitmask of the inlier views, bit v for view v, 0 where the point is NaN).
    """
    B, V, J, _ = pix.shape
    device = pix.device
    pix = pix.to(torch.float32).contiguous()
    calib, stride = _calib_arg(calib, B, V, device)
    points = torch.empty((B, J, 3), dtype=torch.float32, device=device)
    inliers = torch.empty((B, J), dtype=torch.int32, device=device)
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device).cuda_stream
        _lib.check(_lib.lib().mpl_triangulate_robust_strided(pix.data_ptr(), calib.data_ptr(), stride, B, V, J, float(min_conf),
                                                             float(inlier_px), points.data_ptr(), inliers.data_ptr(), stream))
    return points, inliers


def refine_triangulation(pix: torch.Tensor, calib, init: torch.Tensor, view_mask: torch.Tensor | None = None,
                         min_conf: float = 0.0, max_iters: int = 20) -> tuple:
    """Levenberg-Marquardt refinement of triangulated points on the confidence-weighted reprojection error
    (`mpl_triangulate_refine`), enqueued on the current stream.

    pix [B, V, J, 3] fp32 (u, v, conf) pixels on the device; calib [V, 18] or [B, V, 18] as for `build_inputs`; init
    [B, J, 3] starting points, e.g. the points of `triangulate` or `triangulate_robust`.  Per (pose, joint), the views used
    are the candidates of `triangulate` (conf > min_conf, strictly inside the image) whose bit is set in view_mask [B, J]
    int32 (None: every candidate).  Pass `triangulate_robust`'s inliers as view_mask to refine over them; do NOT pass the
    views_used count of `triangulate`, which is a number of views, not a bitmask.  Minimises
    sum_v conf_v^2 |pi(P_v X) - x_v|^2 in fp64 (the maximum-likelihood point when the pixel noise has std sigma / conf)
    with at most max_iters (1 to 100) iterations.  Returns (points [B, J, 3] fp32; reproj_px [B, J] fp32, the conf-weighted
    RMS pixel error at the refined point).  Where init is not finite, fewer than two views are used or init lies behind a
    used camera, points is init unchanged and reproj_px is NaN.
    """
    B, V, J, _ = pix.shape
    device = pix.device
    if tuple(init.shape) != (B, J, 3):
        raise ValueError(f"init must be [B, J, 3] = [{B}, {J}, 3], got {list(init.shape)}")
    if view_mask is not None and (tuple(view_mask.shape) != (B, J) or view_mask.dtype != torch.int32):
        raise ValueError(f"view_mask must be a [B, J] = [{B}, {J}] int32 bitmask, got {list(view_mask.shape)} "
                         f"{view_mask.dtype}")
    pix = pix.to(torch.float32).contiguous()
    init = init.to(device=device, dtype=torch.float32).contiguous()
    mask = None if view_mask is None else view_mask.to(device).contiguous()
    calib, stride = _calib_arg(calib, B, V, device)
    points = torch.empty((B, J, 3), dtype=torch.float32, device=device)
    reproj_px = torch.empty((B, J), dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device).cuda_stream
        _lib.check(_lib.lib().mpl_triangulate_refine_strided(
            pix.data_ptr(), calib.data_ptr(), stride, B, V, J, float(min_conf),
            None if mask is None else mask.data_ptr(), init.data_ptr(), int(max_iters), points.data_ptr(),
            reproj_px.data_ptr(), stream))
    return points, reproj_px


def add_detector_noise(pix: torch.Tensor, calib, seed: int, start: int, sigma_px: float, p_outlier: float,
                       p_miss: float) -> torch.Tensor:
    """Detector-error model (`mpl_synth_detector_noise`) applied IN PLACE to raw pixels of poses [start, start + B),
    enqueued on the current stream; returns `pix`.

    pix [B, V, J, 3] contiguous fp32 (u, v, conf) on the device, as `synth_project` returns it; calib [V, 18] or
    [B, V, 18] (only w, h are read).  Per entry with conf > 0: a miss (conf = 0) with probability p_miss, a confident false detection anywhere in
    the image with probability p_outlier, otherwise Gaussian pixel noise of std sigma_px / conf.  The draws depend only on
    (seed, global pose index), under a key separate from `synth_project`'s; `synth.detector_noise` is the numpy twin.
    """
    if pix.dtype != torch.float32 or not pix.is_contiguous() or pix.dim() != 4 or pix.shape[-1] != 3:
        raise ValueError("add_detector_noise works in place on a contiguous float32 [B, V, J, 3] tensor")
    B, V, J, _ = pix.shape
    calib, stride = _calib_arg(calib, B, V, pix.device)
    with torch.cuda.device(pix.device):
        stream = torch.cuda.current_stream(pix.device).cuda_stream
        _lib.check(_lib.lib().mpl_synth_detector_noise_strided(int(seed), int(start), B, V, J, calib.data_ptr(), stride,
                                                               float(sigma_px), float(p_outlier), float(p_miss), pix.data_ptr(),
                                                               stream))
    return pix


def distort_pixels(pix: torch.Tensor, calib, dist) -> torch.Tensor:
    """Lens distortion (`mpl_distort_pixels`) applied IN PLACE to ideal pinhole pixels, enqueued on the current stream;
    returns `pix`.

    pix [B, V, J, 3] contiguous fp32 (u, v, conf) on the device, e.g. as `synth_project` returns it (before
    `add_detector_noise`, which models errors in detector pixels); calib [V, 18] or [B, V, 18]; dist (k1, k2, p1, p2, k3)
    per view, [V, 5] or [B, V, 5] (numpy or tensor; OpenCV's distCoeffs order).  Each entry with conf != 0 moves to where
    OpenCV's 5-coefficient model images it; an entry past a fold of the model (see include/mpl_b200.h) gets conf = 0.
    Zero coefficients leave pix bitwise unchanged.  `synth.distort_pixels` is the numpy twin.
    """
    if pix.dtype != torch.float32 or not pix.is_contiguous() or pix.dim() != 4 or pix.shape[-1] != 3:
        raise ValueError("distort_pixels works in place on a contiguous float32 [B, V, J, 3] tensor")
    B, V, J, _ = pix.shape
    calib, cstride = _calib_arg(calib, B, V, pix.device)
    dist, dstride = _dist_arg(dist, B, V, pix.device)
    with torch.cuda.device(pix.device):
        stream = torch.cuda.current_stream(pix.device).cuda_stream
        _lib.check(_lib.lib().mpl_distort_pixels_strided(pix.data_ptr(), pix.data_ptr(), calib.data_ptr(), cstride,
                                                         dist.data_ptr(), dstride, B, V, J, stream))
    return pix


def undistort_pixels(pix: torch.Tensor, calib, dist, margin=None) -> tuple:
    """Undistortion of detected pixels for the triangulations (`mpl_undistort_pixels`), enqueued on the current stream.

    pix [B, V, J, 3] fp32 (u, v, conf) raw detections on the device; calib [V, 18] or [B, V, 18]; dist [V, 5] or [B, V, 5]
    as for `distort_pixels`.  margin: (margin_x, margin_y) pixels, or one number for both; None = half the image on each
    side, (max w / 2, max h / 2) over the calibration's views (read from calib: a device tensor costs one synchronisation;
    pass the margin to avoid it).  Returns (pix_u, calib_u): pix_u [B, V, J, 3] the pinhole pixels of the same rays shifted
    by the margin, calib_u the calibration of calib's shape with cx + margin_x, cy + margin_y, w + 2 margin_x,
    h + 2 margin_y, to pass with pix_u to `triangulate`, `triangulate_robust` and `refine_triangulation`.  Entries whose raw
    pixel is not strictly inside the original image get conf 0 (the candidate sets stay those of the raw pixels), and so
    do entries the Newton inversion fails on (with NaN pixels).  An undistorted pixel further than the margin outside
    the image fails the triangulations' candidate test and is dropped.
    """
    if pix.dim() != 4 or pix.shape[-1] != 3:
        raise ValueError(f"undistort_pixels takes a [B, V, J, 3] tensor, got {list(pix.shape)}")
    B, V, J, _ = pix.shape
    device = pix.device
    pix = pix.to(torch.float32).contiguous()
    calib, cstride = _calib_arg(calib, B, V, device)
    dist, dstride = _dist_arg(dist, B, V, device)
    if margin is None:
        wh = calib[..., 16:18].reshape(-1, 2).amax(0).cpu() if calib.numel() else torch.zeros(2, dtype=torch.float64)
        mx, my = float(wh[0]) / 2.0, float(wh[1]) / 2.0
    elif np.ndim(margin) == 0:
        mx = my = float(margin)
    else:
        mx, my = (float(m) for m in margin)
    if not (np.isfinite(mx) and np.isfinite(my) and mx >= 0 and my >= 0):
        raise ValueError(f"margin must be finite and >= 0, got ({mx}, {my})")
    out = torch.empty_like(pix)
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device).cuda_stream
        _lib.check(_lib.lib().mpl_undistort_pixels_strided(pix.data_ptr(), out.data_ptr(), calib.data_ptr(), cstride,
                                                           dist.data_ptr(), dstride, mx, my, B, V, J, stream))
    calib_u = calib.clone()
    calib_u[..., 14] += mx
    calib_u[..., 15] += my
    calib_u[..., 16] += 2.0 * mx
    calib_u[..., 17] += 2.0 * my
    return out, calib_u


def calibration_noise(calib, seed: int, start: int, sigma_rot: float, sigma_pos: float, device=None) -> torch.Tensor:
    """Calibration errors (`mpl_synth_calib_noise`), enqueued on the current stream; returns a new fp64 tensor.

    calib [V, 18] (a fixed rig, perturbed as pose `start`) or [B, V, 18] (one calibration per pose, poses [start, start + B)),
    numpy or tensor.  Per (pose, view): R' = Exp(sigma_rot n) R (radians, a rotation in the camera frame) and
    t' = t + sigma_pos m (world units), n and m standard normal 3-vectors drawn under a Philox key of their own; the
    intrinsics are copied.  The draws depend only on (seed, global pose index); `synth.calibration_noise` is the numpy twin.
    """
    if device is None:
        device = calib.device if isinstance(calib, torch.Tensor) else torch.device("cuda", torch.cuda.current_device())
    c = calib.to(device=device, dtype=torch.float64) if isinstance(calib, torch.Tensor) else \
        torch.as_tensor(np.asarray(calib, dtype=np.float64)).to(device)
    c = c.contiguous()
    if c.dim() not in (2, 3) or c.shape[-1] != 18:
        raise ValueError(f"calib must be [V, 18] or [B, V, 18], got {list(c.shape)}")
    V = c.shape[-2]
    B = 1 if c.dim() == 2 else c.shape[0]
    out = torch.empty_like(c)
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device).cuda_stream
        _lib.check(_lib.lib().mpl_synth_calib_noise(int(seed), int(start), B, V, c.data_ptr(), 0 if c.dim() == 2 else 18 * V,
                                                    float(sigma_rot), float(sigma_pos), out.data_ptr(), stream))
    return out


def calibrate_rig(pix: torch.Tensor, calib, init: torch.Tensor, view_mask: torch.Tensor | None = None,
                  sigma_px: float = 1.0, sigma_rot: float = math.radians(1.0), sigma_pos: float = 0.05,
                  min_conf: float = 0.0, max_iters: int = 30) -> tuple:
    """Bundle adjustment of a rig's extrinsics from its detections (`mpl_calibrate_rig`), enqueued on the current stream.

    pix [B, V, J, 3] fp32 (u, v, conf) pixels of B poses seen by one rig calib [V, 18]; init [B, J, 3] starting points, e.g.
    `triangulate(pix, calib)[0]`; view_mask [B, J] int32 bitmask or None (every candidate view, as in
    `refine_triangulation`).  Levenberg-Marquardt on sum conf^2 / sigma_px^2 |reprojection error|^2 plus the Gaussian prior
    |omega_v|^2 / sigma_rot^2 + |c_v - c0_v|^2 / sigma_pos^2 on each camera's rotation (radians) and centre (world units),
    the distribution `calibration_noise` draws from.  Returns (calib_refined [V, 18] fp64 with the intrinsics of calib;
    points [B, J, 3] fp32, the refined joints where they took part and init elsewhere; report [8] fp64 = items,
    observations, cost at the start and at the end, conf-weighted RMS pixel error at the start and at the end, iterations,
    accepted steps), all on the device.
    """
    B, V, J, _ = pix.shape
    device = pix.device
    if tuple(init.shape) != (B, J, 3):
        raise ValueError(f"init must be [B, J, 3] = [{B}, {J}, 3], got {list(init.shape)}")
    if view_mask is not None and (tuple(view_mask.shape) != (B, J) or view_mask.dtype != torch.int32):
        raise ValueError(f"view_mask must be a [B, J] = [{B}, {J}] int32 bitmask, got {list(view_mask.shape)} "
                         f"{view_mask.dtype}")
    pix = pix.to(torch.float32).contiguous()
    init = init.to(device=device, dtype=torch.float32).contiguous()
    mask = None if view_mask is None else view_mask.to(device).contiguous()
    calib, stride = _calib_arg(calib, B, V, device)
    if stride != 0 or tuple(calib.shape) != (V, 18):
        raise ValueError(f"calibrate_rig takes one rig calib [V, 18] = [{V}, 18], got {list(calib.shape)}")
    L = _lib.lib()
    nbytes = L.mpl_calibrate_rig_workspace_bytes(B, V, J)
    if nbytes == 0:
        raise ValueError(f"calibrate_rig: unsupported shape B={B} V={V} J={J} (2 <= V <= 16, B >= 1, J >= 1)")
    ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
    calib_out = torch.empty_like(calib)
    points = torch.empty((B, J, 3), dtype=torch.float32, device=device)
    report = torch.empty(8, dtype=torch.float64, device=device)
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device).cuda_stream
        _lib.check(L.mpl_calibrate_rig(pix.data_ptr(), calib.data_ptr(), B, V, J, float(min_conf),
                                       None if mask is None else mask.data_ptr(), init.data_ptr(), float(sigma_px),
                                       float(sigma_rot), float(sigma_pos), int(max_iters), calib_out.data_ptr(),
                                       points.data_ptr(), report.data_ptr(), ws.data_ptr(), nbytes, stream))
    return calib_out, points, report


def synth_people(pix: torch.Tensor, people: int, seed: int, start: int) -> tuple:
    """Multi-person scenes out of person-ordered pixels (`mpl_synth_people`), enqueued on the current stream.

    pix [F P, V, J, 3] fp32 on the device holds person p of frame f in row f P + p, e.g. `synth_project` of poses
    [start P, (start + F) P) with lens and detector noise.  Each view's P detections are put into its P slots in a random
    order drawn per (seed, global frame index start + f) under a Philox key of their own.  Returns (scene [F, P, V, J, 3],
    scene[f, s, v] = pix[f P + perm[f, v, s], v] bit for bit; perm [F, V, P] int32, the person in each slot).
    `synth.synth_people` is the numpy twin.
    """
    if pix.dim() != 4 or pix.shape[-1] != 3 or pix.shape[0] % people:
        raise ValueError(f"pix must be [F P, V, J, 3] with P = {people}, got {list(pix.shape)}")
    B, V, J, _ = pix.shape
    F = B // people
    pix = pix.to(torch.float32).contiguous()
    scene = torch.empty((F, people, V, J, 3), dtype=torch.float32, device=pix.device)
    perm = torch.empty((F, V, people), dtype=torch.int32, device=pix.device)
    with torch.cuda.device(pix.device):
        stream = torch.cuda.current_stream(pix.device).cuda_stream
        _lib.check(_lib.lib().mpl_synth_people(int(seed), int(start), F, int(people), V, J, pix.data_ptr(), scene.data_ptr(),
                                               perm.data_ptr(), stream))
    return scene, perm


def associate_people(scene: torch.Tensor, calib, min_conf: float = 0.0, min_joints: int = 3, max_dist: float = 0.1,
                     max_people: int | None = None) -> tuple:
    """Cross-view association of the detections of multi-person scenes (`mpl_associate_people`), enqueued on the current
    stream.

    scene [F, P, V, J, 3] fp32 (u, v, conf) pinhole pixels (undistort first when the cameras have a lens); calib [V, 18] or
    [F, V, 18] (one calibration per frame).  A detection is active with at least min_joints candidate joints (conf >
    min_conf, strictly inside the image); the cost of two active detections of different views is the median, over their
    shared candidate joints, of the distance between their rays (world units); pairs with cost <= max_dist are merged
    greedily, cheapest first, into clusters with at most one detection per view whose member pairs all pass the threshold.
    Clusters of >= 2 detections are people, ranked by size, then by their first detection.  Returns (members [F, K, V]
    int32 slots or -1, K = max_people (default P); labels [F, P, V] int32: the detection's person rank if < K, -1 when
    active but in no such person, -2 when inactive; people [F] int32, the number of people, which may exceed K).
    """
    if scene.dim() != 5 or scene.shape[-1] != 3:
        raise ValueError(f"scene must be [F, P, V, J, 3], got {list(scene.shape)}")
    F, P, V, J, _ = scene.shape
    K = P if max_people is None else int(max_people)
    device = scene.device
    scene = scene.to(torch.float32).contiguous()
    calib, stride = _calib_arg(calib, F, V, device)
    members = torch.empty((F, K, V), dtype=torch.int32, device=device)
    labels = torch.empty((F, P, V), dtype=torch.int32, device=device)
    people = torch.empty((F,), dtype=torch.int32, device=device)
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device).cuda_stream
        _lib.check(_lib.lib().mpl_associate_people_strided(
            scene.data_ptr(), calib.data_ptr(), stride, F, P, V, J, float(min_conf), int(min_joints), float(max_dist), K,
            members.data_ptr(), labels.data_ptr(), people.data_ptr(), stream))
    return members, labels, people


def gather_people(scene: torch.Tensor, members: torch.Tensor) -> torch.Tensor:
    """The detections of each associated person (`mpl_gather_people`), enqueued on the current stream: out [F, K, V, J, 3],
    out[f, k, v] = scene[f, members[f, k, v], v] bit for bit, zeros where the member is -1.  `out.view(F * K, V, J, 3)` is a
    batch of people for `build_inputs`, the model and the triangulations."""
    if scene.dim() != 5 or scene.shape[-1] != 3:
        raise ValueError(f"scene must be [F, P, V, J, 3], got {list(scene.shape)}")
    F, P, V, J, _ = scene.shape
    if members.dim() != 3 or members.shape[0] != F or members.shape[2] != V or members.dtype != torch.int32:
        raise ValueError(f"members must be an int32 [F, K, V] = [{F}, K, {V}] tensor, got {list(members.shape)} {members.dtype}")
    K = members.shape[1]
    scene = scene.to(torch.float32).contiguous()
    members = members.to(scene.device).contiguous()
    out = torch.empty((F, K, V, J, 3), dtype=torch.float32, device=scene.device)
    with torch.cuda.device(scene.device):
        stream = torch.cuda.current_stream(scene.device).cuda_stream
        _lib.check(_lib.lib().mpl_gather_people(scene.data_ptr(), members.data_ptr(), F, P, K, V, J, out.data_ptr(), stream))
    return out


def association_score(members: torch.Tensor, labels: torch.Tensor, perm: torch.Tensor, acc: torch.Tensor | None = None) -> tuple:
    """Scores an association against the true slots (`mpl_association_score`), enqueued on the current stream.

    members [F, K, V] and labels [F, P, V] of `associate_people`, perm [F, V, P] of `synth_people`.  Returns (owner [F, K]
    int32: the true person with the most members in each row, ties to the smaller index, -1 for an empty row; acc [8] fp64,
    the running sums of include/mpl_b200.h added into `acc` when given: frames, associable people, non-empty rows, pure
    rows, complete rows, predicted linked pairs, correct linked pairs, true pairs)."""
    if members.dim() != 3 or labels.dim() != 3 or perm.dim() != 3:
        raise ValueError("members [F, K, V], labels [F, P, V] and perm [F, V, P] must be 3-dimensional")
    F, K, V = members.shape
    P = labels.shape[1]
    if tuple(labels.shape) != (F, P, V) or tuple(perm.shape) != (F, V, P):
        raise ValueError(f"labels must be [F, P, V] and perm [F, V, P] for members {list(members.shape)}, got "
                         f"{list(labels.shape)} and {list(perm.shape)}")
    for name, t in (("members", members), ("labels", labels), ("perm", perm)):
        if t.dtype != torch.int32:
            raise ValueError(f"{name} must be int32, got {t.dtype}")
    device = members.device
    if acc is None:
        acc = torch.zeros(_lib.ASSOC_ACC_LEN, dtype=torch.float64, device=device)
    elif acc.dtype != torch.float64 or tuple(acc.shape) != (_lib.ASSOC_ACC_LEN,) or not acc.is_contiguous():
        raise ValueError(f"acc must be a contiguous float64 [{_lib.ASSOC_ACC_LEN}] tensor")
    members, labels, perm = (t.to(device).contiguous() for t in (members, labels, perm))
    owner = torch.empty((F, K), dtype=torch.int32, device=device)
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device).cuda_stream
        _lib.check(_lib.lib().mpl_association_score(members.data_ptr(), labels.data_ptr(), perm.data_ptr(), F, P, K, V,
                                                    owner.data_ptr(), acc.data_ptr(), stream))
    return owner, acc


def synth_motion(sequences: int, frames: int, people: int, rig, seed: int = 0, start: int = 0, fps: float = 30.0,
                 conf_mode: str = "uniform", device=None, cameras=None) -> tuple:
    """Sequences of people that move, generated and projected ON THE DEVICE (`mpl_synth_motion`).

    Row ((start + s) T + t) P + p is person p in frame t of global sequence start + s: a body of synth_project's shape
    walking a closed-form path in the rig's room and turning slowly (include/mpl_b200.h states the model), so person p of a
    sequence depends only on (seed, sequence, p, t).  Returns (pix [S T P, V, 17, 3] raw pixels (u, v, conf), target
    [S T P, 17, 3] metres, calib) as `synth_project` does: the rig's [V, 18] calibration, or `cameras`, a [S T P, V, 18]
    calibration per row.  Viewed as [F P, ...] with F = S T frames, pass frame (start + s) T + t to `synth_people` and row
    index r to `add_detector_noise`.  `synth.synth_motion` is the numpy twin.
    """
    from .synth import NUM_JOINTS
    device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    V, J = rig.num_views, NUM_JOINTS
    rows = sequences * frames * people
    if cameras is None:
        calib = torch.as_tensor(pack_calibration(rig.R, rig.t, rig.f, rig.c, rig.image_size)).to(device)
        stride = 0
    else:
        calib, stride = _calib_arg(cameras, rows, V, device)
        if stride == 0:
            raise ValueError("cameras must be a [S T P, V, 18] calibration per row")
    if conf_mode not in ("uniform", "ones"):
        raise ValueError(conf_mode)
    room = torch.as_tensor(np.asarray(rig.room, dtype=np.float64)).to(device)
    pix = torch.empty((rows, V, J, 3), dtype=torch.float32, device=device)
    target = torch.empty((rows, J, 3), dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device).cuda_stream
        _lib.check(_lib.lib().mpl_synth_motion(int(seed), int(start), int(sequences), int(frames), int(people), V, J,
                                               calib.data_ptr(), stride, room.data_ptr(), float(fps),
                                               int(conf_mode == "ones"), pix.data_ptr(), target.data_ptr(), stream))
    return pix, target, calib


def track_state(sequences: int, max_tracks: int, num_joints: int, device=None) -> torch.Tensor:
    """A zeroed tracker state for `track_people`: [S, mpl_track_state_bytes(max_tracks, J)] uint8, fresh sequences."""
    nbytes = _lib.lib().mpl_track_state_bytes(int(max_tracks), int(num_joints))
    if nbytes == 0:
        raise ValueError(f"unsupported tracker shape max_tracks={max_tracks} J={num_joints} (1 <= max_tracks <= 128, "
                         f"1 <= J <= 32)")
    device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    return torch.zeros((sequences, nbytes), dtype=torch.uint8, device=device)


def track_people(points: torch.Tensor, joint_mask: torch.Tensor | None = None, state: torch.Tensor | None = None,
                 min_joints: int = 3, max_dist: float = 0.2, max_age: int = 5, max_tracks: int | None = None) -> tuple:
    """Online tracking of person rows across frames (`mpl_track_people`), enqueued on the current stream.

    points [S, T, K, J, 3] fp32 on the device: per frame of S independent sequences, K rows of 3D joints (e.g. the robust
    triangulation of `gather_people` rows); NaN joints are not used.  joint_mask [S, T, K, J] (> 0: use the joint) or None.
    state: the [S, nbytes] uint8 tensor of `track_state` for the same max_tracks (default 2 K), updated in place, so frames
    can be fed in chunks; None: a fresh one.  A row with at least min_joints used joints is a detection; each frame, (track, row) pairs
    whose median joint distance is at most max_dist (world units) are matched greedily, cheapest first; unmatched tracks die
    after max_age missed frames, and unmatched detections start new tracks with the sequence's next id.  Returns (track_id
    [S, T, K] int32, -1 for rows without a track; state).
    """
    if points.dim() != 5 or points.shape[-1] != 3:
        raise ValueError(f"points must be [S, T, K, J, 3], got {list(points.shape)}")
    S, T, K, J, _ = points.shape
    device = points.device
    points = points.to(torch.float32).contiguous()
    mask = None
    if joint_mask is not None:
        if tuple(joint_mask.shape) != (S, T, K, J):
            raise ValueError(f"joint_mask must be [S, T, K, J] = [{S}, {T}, {K}, {J}], got {list(joint_mask.shape)}")
        mask = joint_mask.to(device=device, dtype=torch.float32).contiguous()
    max_tracks = 2 * K if max_tracks is None else int(max_tracks)
    if state is None:
        state = track_state(S, max_tracks, J, device)
    nbytes = _lib.lib().mpl_track_state_bytes(max_tracks, J)
    if state.dim() != 2 or tuple(state.shape) != (S, nbytes) or state.dtype != torch.uint8 or not state.is_contiguous() or \
            nbytes == 0:
        raise ValueError(f"state must be a contiguous uint8 [S, mpl_track_state_bytes(max_tracks, J)] tensor for S={S}, "
                         f"max_tracks={max_tracks}, J={J}, got {list(state.shape)} {state.dtype}")
    track_id = torch.empty((S, T, K), dtype=torch.int32, device=device)
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device).cuda_stream
        _lib.check(_lib.lib().mpl_track_people(points.data_ptr(), None if mask is None else mask.data_ptr(), S, T, K, J,
                                               int(min_joints), float(max_dist), int(max_age), max_tracks,
                                               state.data_ptr(), track_id.data_ptr(), stream))
    return track_id, state


def tracking_score(track_id: torch.Tensor, owner: torch.Tensor, people: int, acc: torch.Tensor | None = None) -> torch.Tensor:
    """CLEAR-MOT style counts of a tracking against the rows' true persons (`mpl_tracking_score`), enqueued on the current
    stream.  track_id [S, T, K] of `track_people` (whole sequences from a fresh state), owner [S, T, K] int32 (the true
    person of each row, -1 for none, e.g. `association_score`'s owner), people P per frame.  Returns acc [11] fp64, the
    running sums of include/mpl_b200.h added into `acc` when given: sequences, frames, objects, matches, misses, false
    positives, ID switches, fragmentations, mostly tracked, mostly lost, tracks."""
    if track_id.dim() != 3 or tuple(owner.shape) != tuple(track_id.shape):
        raise ValueError(f"track_id and owner must both be [S, T, K], got {list(track_id.shape)} and {list(owner.shape)}")
    if track_id.dtype != torch.int32 or owner.dtype != torch.int32:
        raise ValueError("track_id and owner must be int32")
    S, T, K = track_id.shape
    device = track_id.device
    if acc is None:
        acc = torch.zeros(_lib.TRACK_ACC_LEN, dtype=torch.float64, device=device)
    elif acc.dtype != torch.float64 or tuple(acc.shape) != (_lib.TRACK_ACC_LEN,) or not acc.is_contiguous():
        raise ValueError(f"acc must be a contiguous float64 [{_lib.TRACK_ACC_LEN}] tensor")
    track_id, owner = (t.to(device).contiguous() for t in (track_id, owner))
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device).cuda_stream
        _lib.check(_lib.lib().mpl_tracking_score(track_id.data_ptr(), owner.data_ptr(), S, T, K, int(people), acc.data_ptr(),
                                                 stream))
    return acc


def _dist_arg(dist, B: int, V: int, device) -> tuple:
    """(contiguous fp64 device tensor, dist_stride): [V, 5] -> stride 0 (one lens set for the batch); [B, V, 5] -> 5 V."""
    if isinstance(dist, torch.Tensor):
        dist = dist.to(device=device, dtype=torch.float64).contiguous()
    else:
        dist = torch.as_tensor(np.asarray(dist, dtype=np.float64)).to(device).contiguous()
    if dist.dim() == 2 and tuple(dist.shape) == (V, 5):
        return dist, 0
    if dist.dim() == 3 and dist.shape[0] == B and tuple(dist.shape[1:]) == (V, 5):
        return dist, 5 * V
    raise ValueError(f"dist must be [V, 5] = [{V}, 5] or [B, V, 5] = [{B}, {V}, 5], got {list(dist.shape)}")


def _calib_arg(calib, B: int, V: int, device) -> tuple:
    """(contiguous fp64 device tensor, calib_stride): [V, 18] -> stride 0 (one rig for the batch); [B, V, 18] -> 18 V."""
    if isinstance(calib, torch.Tensor):
        calib = calib.to(device=device, dtype=torch.float64).contiguous()
    else:
        calib = torch.as_tensor(np.asarray(calib, dtype=np.float64)).to(device).contiguous()
    if calib.dim() != 3:
        return calib, 0
    if calib.shape[0] != B or tuple(calib.shape[1:]) != (V, 18):
        raise ValueError(f"a per-pose calibration must be [B, V, 18] = [{B}, {V}, 18], got {list(calib.shape)}")
    return calib, 18 * V


def synth_project(batch: int, rig, seed: int = 0, start: int = 0, conf_mode: str = "uniform", device=None,
                  cameras=None) -> tuple:
    """N3: MHP-style synthetic poses generated and projected ON THE DEVICE (`mpl_synth_project`).

    Pose i depends only on (seed, start + i) — the same Philox stream as `synth.make_batch` — so ranks / micro-batches
    can shard the global index range freely.  Returns (pix [B,V,17,3] raw pixels (u, v, conf), target [B,17,3] metres,
    calib [V,18] fp64 on the device); `build_inputs(pix, calib)` turns the pixels into the model's inputs.  With
    `cameras`, a [B, V, 18] calibration per pose (e.g. from `synth_cameras`), the poses are projected through those
    instead of the rig's, and `calib` is that tensor; the 3D poses (placed in the rig's room) do not change.
    """
    from .synth import NUM_JOINTS
    device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    V, J = rig.num_views, NUM_JOINTS
    if cameras is None:
        calib = torch.as_tensor(pack_calibration(rig.R, rig.t, rig.f, rig.c, rig.image_size)).to(device)
        stride = 0
    else:
        calib, stride = _calib_arg(cameras, batch, V, device)
        if stride == 0:
            raise ValueError("cameras must be a [B, V, 18] calibration per pose")
    room = torch.as_tensor(np.asarray(rig.room, dtype=np.float64)).to(device)
    pix = torch.empty((batch, V, J, 3), dtype=torch.float32, device=device)
    target = torch.empty((batch, J, 3), dtype=torch.float32, device=device)
    if conf_mode not in ("uniform", "ones"):
        raise ValueError(conf_mode)
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device).cuda_stream
        _lib.check(_lib.lib().mpl_synth_project_strided(int(seed), int(start), int(batch), V, J, calib.data_ptr(), stride,
                                                        room.data_ptr(), int(conf_mode == "ones"), pix.data_ptr(),
                                                        target.data_ptr(), stream))
    return pix, target, calib


def synth_cameras(batch: int, num_views: int, kind: str = "h36m", seed: int = 0, start: int = 0, device=None) -> torch.Tensor:
    """Random camera setups generated ON THE DEVICE (`mpl_synth_cameras`): [B, V, 18] fp64 calibrations of poses
    [start, start + batch) around the room of rig `kind` ("h36m" or "cmu": its focal length, image size and room).  Pose
    i's cameras depend only on (seed, start + i), under a Philox key separate from the poses' and the detector noise's;
    `synth.random_cameras` is the numpy twin.  Feed them to `synth_project(..., cameras=...)` and every calibration-taking
    entry point of this module.
    """
    from .synth import rig_kind
    f0, (w, h), room = rig_kind(kind)
    device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    room = torch.as_tensor(np.asarray(room, dtype=np.float64)).to(device)
    calib = torch.empty((batch, num_views, 18), dtype=torch.float64, device=device)
    with torch.cuda.device(device):
        stream = torch.cuda.current_stream(device).cuda_stream
        _lib.check(_lib.lib().mpl_synth_cameras(int(seed), int(start), int(batch), int(num_views), float(f0), float(w),
                                                float(h), room.data_ptr(), calib.data_ptr(), stream))
    return calib
