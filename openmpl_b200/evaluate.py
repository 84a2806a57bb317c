"""Large-batch evaluation loop on synthetic MHP-style data — the device-resident counterpart of the reference's
`validate()` (`MPL/lib/core/function_mpl.py:293-649`) for BASELINE.json configs 3-5.

    python -m openmpl_b200.evaluate --arch hm0 --views 4 --poses 10000000               # config 5 on one GPU
    torchrun --nproc-per-node 8 -m openmpl_b200.evaluate --arch cmu0 --views 5 ...      # config 3: ranks shard the poses
    python -m openmpl_b200.evaluate --arch kptok --views 8 --depth 12 --poses 262144    # config 4: view sweep
    python -m openmpl_b200.evaluate --arch hm0 --views 4 --triangulate                   # + the triangulation baseline
    python -m openmpl_b200.evaluate --arch hm0 --views 4 --pixel-noise 2 --outlier-rate 0.1 --triangulate \
        --triangulate-robust                                                            # noisy detections, both baselines
    python -m openmpl_b200.evaluate --arch hm0 --views 4 --random-cameras --triangulate  # a random camera setup per pose
    python -m openmpl_b200.evaluate --arch hm0 --views 4 --pixel-noise 2 --triangulate --triangulate-robust \
        --refine-triangulations                                                         # + nonlinear refinement of both
    python -m openmpl_b200.evaluate --arch hm0 --views 4 --pixel-noise 2 --triangulate --triangulate-robust \
        --triangulation-pmpjpe                                                          # + P-MPJPE of both baselines
    python -m openmpl_b200.evaluate --arch hm0 --views 4 --lens-distortion=-0.207,0.248,-0.0009,-0.0016,-0.0031 \
        --triangulate --triangulate-robust --refine-triangulations                      # cameras with a lens
    python -m openmpl_b200.evaluate --arch hm0 --views 4 --pixel-noise 1 --calib-noise 0.5,20 --triangulate \
        --calibrate-rig 16384                                                           # a miscalibrated rig, recalibrated
    python -m openmpl_b200.evaluate --arch cmu0 --views 5 --people 4 --pixel-noise 2 --outlier-rate 0.1 --triangulate \
        --triangulate-robust                                                            # 4 people per frame, associated
    python -m openmpl_b200.evaluate --arch cmu0 --views 5 --people 4 --frames 64 --pixel-noise 2 --outlier-rate 0.1 \
        --triangulate-robust                                                            # sequences of 64 frames, tracked

Per micro-batch, entirely on the device: `mpl_synth_project` (3D poses from the counter-based generator keyed by the
GLOBAL pose index, projected through the V calibrations) -> `mpl_build_inputs` (clip, confidence zeroing, screen
normalisation, rays) -> `mpl_forward` -> `mpl_mpjpe_accumulate` + `mpl_pmpjpe_accumulate` (fp64 running sums).  Predictions never leave the GPU;
ranks own contiguous slices of the index range, and one all-reduce of the 11 J + 1 (and J + 3 Procrustes) sums at the end
gives the MPJPE the reference's `evaluate()` would log (`function_mpl.py:670-687`) and the P-MPJPE of
`pose_utils.py:61-143`.  Prints one JSON line from rank 0.

With `--triangulate`, each micro-batch's pixels are also triangulated (`mpl_triangulate`, the linear baseline of
`MPL/lib/multiviews/triangulate.py:59-115`) and scored by a third MPJPE accumulator that masks joints seen by fewer than two
views; the line gains a "triangulation" entry.  Without the flag nothing of this runs.

`--pixel-noise PX`, `--outlier-rate P` and `--miss-rate P` corrupt each micro-batch's pixels right after they are generated
(`mpl_synth_detector_noise`: Gaussian noise of std PX / conf, confident false detections, misses; keyed by the global pose
index like the poses), so the lifter and the triangulations all see the same detections; the line's "data" entry records
the three values.  `--triangulate-robust` adds a "triangulation_robust" entry for `mpl_triangulate_robust` (pair RANSAC
with the MSAC cost at `--inlier-px`, then a confidence-weighted refit), masked where it finds fewer than two inliers.

`--random-cameras` gives every pose its own camera setup: each micro-batch first generates [B, V, 18] calibrations
(`mpl_synth_cameras`, random positions, heights, look-at points and focal lengths around the room of the rig kind, keyed
by the global pose index), then projects, corrupts, builds inputs and triangulates through them.  The line's "data" entry
records the camera model.  Without the flag the one rig of `--rig` serves every pose.

`--refine-triangulations` (with `--triangulate` and / or `--triangulate-robust`) refines each triangulation's points by
Levenberg-Marquardt on the conf^2-weighted reprojection error (`mpl_triangulate_refine`): the linear points over their
candidate views, the robust points over their inliers.  Each triangulation entry gains a "refined" sub-entry, scored by its
own accumulator under the parent entry's mask.  Without the flag nothing of this runs.

`--triangulation-pmpjpe` (with `--triangulate` and / or `--triangulate-robust`) also scores each triangulation entry, and
each "refined" sub-entry, by a masked P-MPJPE accumulator (`mpl_pmpjpe_accumulate_masked`) under that entry's own mask:
every pose is Procrustes-aligned on its triangulated joints only.  The entry gains "procrustes_aligned".  Without the flag
nothing of this runs.

`--lens-distortion K1,K2,P1,P2,K3` gives every view a lens of OpenCV's 5-coefficient model (`mpl_distort_pixels`): each
micro-batch's projected pixels are distorted before the detector noise (which models errors in detector pixels), the
lifter's inputs are built from the distorted pixels as the reference builds them from a real detector's, and every
triangulation and refinement runs on `mpl_undistort_pixels` output (margin half the image on each side) with the shifted
calibration it comes with.  It composes with `--random-cameras` (one lens, per-pose calibrations).  The line's "data"
entry records the coefficients.  Without the flag nothing of this runs.

`--calib-noise ROT_DEG,POS_MM` gives every consumer of the calibration a perturbed one (`mpl_synth_calib_noise`: each
camera rotated by a Gaussian rotation vector of std ROT_DEG degrees per axis in its own frame, its centre moved by a
Gaussian of std POS_MM mm per axis): the lifter's inputs, the undistortion, the triangulations and the refinement all use
it, while the synthetic pixels are still projected through the true cameras.  The rig is perturbed once (pose 0 of the
noise stream); with `--random-cameras` every pose's cameras are perturbed under its global index.  The line's "data" entry
records the two values.  `--calib-noise 0,0` gives the metrics of a run without the flag.

`--calibrate-rig N` (with `--calib-noise`, both values > 0; not with `--random-cameras`; N <= `--micro-batch`) recalibrates
the perturbed rig before the evaluation: every rank generates the N poses at global indices [poses, poses + N), disjoint
from the evaluated ones, through the same data path (true projection, lens, detector noise, undistortion), triangulates
them linearly under the perturbed rig and bundle-adjusts the rig's extrinsics and the joints (`mpl_calibrate_rig`, every
candidate view, sigma_px = `--pixel-noise` or 1 px when it is 0, the prior of `--calib-noise`).  The refined rotations and
centres then replace the perturbed ones for the whole evaluation (the intrinsics stay).  Every rank computes the same
bits, so no collective is needed.  The line gains a "rig_calibration" entry: poses, items, observations, iterations,
accepted steps, RMS pixel error before and after, per-view rotation (degrees) and centre (mm) errors of the perturbed and
of the calibrated rig against the true one, and its own time `ms`, outside `ms_total`.

`--people P` (P >= 2; not with `--calibrate-rig`) evaluates multi-person frames whose grouping is not given: `--poses`
counts persons, frame f holds the persons of global indices [f P, (f + 1) P), and each micro-batch is micro_batch // P
frames.  Per micro-batch: the persons are generated and projected with the lens and detector noise as above, put into
random detection slots per view (`mpl_synth_people`), associated across views (`mpl_associate_people`: rays of the
candidate joints, median line distance per cross-view pair at most `--assoc-max-dist` world units over at least
`--assoc-min-joints` shared joints, greedy complete linkage), on the undistorted scene with the shifted calibration when
there is a lens, and gathered into K = P person rows (`mpl_gather_people`, once from the raw scene for the lifter and once
from the undistorted one for the triangulations).  Every metric of the line scores the person rows against the target of
their owner, the true person with the most members in the row; rows without an owner add nothing.  `--random-cameras`
draws the cameras per frame (keyed by the global frame index) and `--calib-noise` applies as above.  The line gains an
"association" entry (`mpl_association_score`): the counts, pair precision and recall, the pure and complete fractions, the
people dropped past K and the parameters.  Without the flag nothing of this runs.

`--frames T` (with `--people P`, T >= 2) evaluates sequences of T frames of P people that move (`mpl_synth_motion`, FPS
frames per second): `--poses` counts person-frames, sequence i holds the frames [i T, (i + 1) T), ranks shard whole
sequences and a micro-batch holds micro_batch // (T P) of them (micro_batch >= T P).  The persons are generated by the
motion model instead of `mpl_synth_project`; the lens, detector noise, slots, association, gathering and every metric run as
with `--people` alone.  The person rows are then triangulated robustly (`mpl_triangulate_robust` at `--inlier-px`) and
tracked from a fresh state per sequence (`mpl_track_people`: `--track-max-dist`, `--track-max-age`, min_joints of
`--assoc-min-joints`, max_tracks = 2 P), and scored against the rows' owners (`mpl_tracking_score`).  `--random-cameras`
draws the cameras per sequence (keyed by the global sequence index), the same for all its frames.  The line gains a
"tracking" entry: the counts, MOTA = 1 - (misses + false positives + ID switches) / objects, the mostly tracked / lost
fractions, tracks per person, the parameters and the time of the tracking calls.  Without the flag nothing of this runs.
"""
from __future__ import annotations

import argparse
import json
import sys

import numpy as np
import torch

from . import dist as mdist, inputs, metric, spec, synth
from .models.multiview_mpl_b200 import MultiView_MPL

ARCHS = {
    # constructor flag sets of the shipped YAMLs / ablations (SURVEY.md Appendix A)
    "hm0": dict(spec.HM0_FLAGS), "cmu0": dict(spec.HM0_FLAGS), "chosen": dict(spec.CHOSEN_FLAGS),
    "kptok": dict(pose_3d_emb_learnable=True, confidence_input_as_third=True, FPT_blocks_view_keypoint_tokens=True),
}
DEFAULT_DEPTH = {"hm0": 12, "chosen": 12, "kptok": 12, "cmu0": 2}
DEFAULT_RIG = {"hm0": "h36m", "chosen": "h36m", "kptok": "h36m", "cmu0": "cmu"}
REFINE_MAX_ITERS = 20
FPS = 30.0                                             # frame rate of the --frames sequences
CALIBRATE_MAX_ITERS = 30


def run(arch="hm0", views=4, depth=None, poses=1 << 20, micro_batch=65536, precision="bf16", rig=None, seed=1,
        weight_seed=0, warmup=1, triangulate=False, pixel_noise=0.0, outlier_rate=0.0, miss_rate=0.0,
        triangulate_robust=False, inlier_px=10.0, random_cameras=False, refine_triangulations=False,
        triangulation_pmpjpe=False, lens_distortion=None, calib_noise=None, calibrate_rig=0, people=0,
        assoc_max_dist=0.1, assoc_min_joints=3, frames=0, track_max_dist=0.2, track_max_age=5):
    if frames:
        if not people:
            raise ValueError("frames needs people")
        if frames < 2:
            raise ValueError(f"frames must be >= 2, got {frames}")
        if micro_batch < frames * people:
            raise ValueError(f"micro_batch must hold at least one sequence of {frames} x {people} person-frames, got "
                             f"{micro_batch}")
        if poses < frames * people:
            raise ValueError(f"poses must hold at least one sequence of {frames} x {people} person-frames, got {poses}")
        if not (np.isfinite(track_max_dist) and track_max_dist > 0):
            raise ValueError(f"track_max_dist must be finite and > 0, got {track_max_dist}")
        if track_max_age < 0:
            raise ValueError(f"track_max_age must be >= 0, got {track_max_age}")
    if people:
        if people < 2:
            raise ValueError(f"people must be >= 2, got {people}")
        if people * views > 128:
            raise ValueError(f"people * views must be <= 128 (the detections of one frame), got {people} * {views}")
        if calibrate_rig:
            raise ValueError("calibrate_rig calibrates from single-person poses: not with people")
        if not (np.isfinite(assoc_max_dist) and assoc_max_dist > 0):
            raise ValueError(f"assoc_max_dist must be finite and > 0, got {assoc_max_dist}")
        if not 1 <= assoc_min_joints <= 17:
            raise ValueError(f"assoc_min_joints must be in [1, 17], got {assoc_min_joints}")
        if micro_batch < people:
            raise ValueError(f"micro_batch must hold at least one frame of {people} people, got {micro_batch}")
    if calib_noise is not None:
        calib_noise = tuple(float(x) for x in calib_noise)
        if len(calib_noise) != 2 or not all(np.isfinite(calib_noise)) or min(calib_noise) < 0:
            raise ValueError(f"calib_noise must be two finite numbers >= 0 (degrees, mm), got {calib_noise}")
    if calibrate_rig:
        if calib_noise is None or min(calib_noise) <= 0:
            raise ValueError("calibrate_rig needs calib_noise with both values > 0")
        if random_cameras:
            raise ValueError("calibrate_rig calibrates one fixed rig: not with random_cameras")
        if not 1 <= calibrate_rig <= micro_batch:
            raise ValueError(f"calibrate_rig must be in [1, micro_batch = {micro_batch}], got {calibrate_rig}")
    if lens_distortion is not None:
        lens_distortion = tuple(float(k) for k in lens_distortion)
        if len(lens_distortion) != 5 or not all(np.isfinite(lens_distortion)):
            raise ValueError(f"lens_distortion must be 5 finite numbers (k1, k2, p1, p2, k3), got {lens_distortion}")
    if refine_triangulations and not (triangulate or triangulate_robust):
        raise ValueError("refine_triangulations needs triangulate or triangulate_robust")
    if triangulation_pmpjpe and not (triangulate or triangulate_robust):
        raise ValueError("triangulation_pmpjpe needs triangulate or triangulate_robust")
    rank, world, local = mdist.init_from_env("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    depth = DEFAULT_DEPTH[arch] if depth is None else depth
    kw = dict(num_joints=17, embed_dim_ratio=32, num_heads=8, depth=depth, num_views=views, drop_path_rate=0.1, **ARCHS[arch])
    cfg = spec.make_config(**kw)
    model = MultiView_MPL(**kw, precision=precision)
    weights = synth.named_weights(spec.param_spec(cfg), seed=weight_seed)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in weights.items()})
    model = model.to(dev).eval()
    mdist.broadcast_state(model)                       # replicas bit-identical (they already are: same seed)
    rig_kind = rig or DEFAULT_RIG[arch]
    the_rig = synth.make_rig(views, rig_kind)
    if frames:                                         # sequences of frames of `people` persons: the range counts sequences
        sequences = poses // (frames * people)
        poses = sequences * frames * people
        micro_batch //= frames * people
        start, stop = mdist.shard_range(sequences, rank, world)
    elif people:                                       # frames of `people` persons: the index range counts frames
        nframes = poses // people
        poses = nframes * people
        micro_batch //= people
        start, stop = mdist.shard_range(nframes, rank, world)
    else:
        start, stop = mdist.shard_range(poses, rank, world)
    # with people, a person row adds into group 0 and a row without an owner into none (-1)
    grouped = dict(num_groups=1) if people else {}
    acc = metric.MpjpeAccumulator(cfg.J, output_in_meter=True, device=dev, **grouped)
    pacc = metric.PmpjpeAccumulator(cfg.J, output_in_meter=True, device=dev, **grouped)
    tacc = metric.MpjpeAccumulator(cfg.J, output_in_meter=True, device=dev, **grouped) if triangulate else None
    racc = metric.MpjpeAccumulator(cfg.J, output_in_meter=True, device=dev, **grouped) if triangulate_robust else None
    tfacc = (metric.MpjpeAccumulator(cfg.J, output_in_meter=True, device=dev, **grouped)
             if triangulate and refine_triangulations else None)
    rfacc = (metric.MpjpeAccumulator(cfg.J, output_in_meter=True, device=dev, **grouped)
             if triangulate_robust and refine_triangulations else None)
    # masked P-MPJPE of each triangulation entry, keyed like the accumulators above
    tp = {name: metric.PmpjpeAccumulator(cfg.J, output_in_meter=True, device=dev, masked=True, **grouped)
          for name, a in (("t", tacc), ("r", racc), ("tf", tfacc), ("rf", rfacc)) if triangulation_pmpjpe and a is not None}
    noisy = pixel_noise != 0 or outlier_rate != 0 or miss_rate != 0
    if lens_distortion is not None:
        lens = torch.tensor([lens_distortion] * views, dtype=torch.float64, device=dev)
        margin = (the_rig.image_size[0] / 2.0, the_rig.image_size[1] / 2.0)   # known here: no read-back of calib
    rig_calib = torch.as_tensor(inputs.pack_calibration(the_rig.R, the_rig.t, the_rig.f, the_rig.c, the_rig.image_size)).to(dev)
    if calib_noise is not None:
        sig_rot, sig_pos = np.radians(calib_noise[0]), calib_noise[1] / 1000.0
        used_rig = inputs.calibration_noise(rig_calib, seed, 0, sig_rot, sig_pos)     # the rig as pose 0 of the noise stream
    else:
        used_rig = rig_calib

    def synth_pixels(s0, n, cams, seqs=None):
        """Pixels of poses [s0, s0 + n) through the true cameras, with the lens and the detector noise; with seqs =
        (first sequence, sequences), the rows of those sequences of people that move."""
        if seqs is None:
            pix, target, calib = inputs.synth_project(n, the_rig, seed=seed, start=s0, device=dev, cameras=cams)
        else:
            pix, target, calib = inputs.synth_motion(seqs[1], frames, people, the_rig, seed=seed, start=seqs[0], fps=FPS,
                                                     device=dev, cameras=cams)
        if lens_distortion is not None:
            inputs.distort_pixels(pix, calib, lens)
        if noisy:
            inputs.add_detector_noise(pix, calib, seed, s0, pixel_noise, outlier_rate, miss_rate)
        return pix, target

    rig_report = None
    if calibrate_rig:
        ce0, ce1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ce0.record()
        pix, _ = synth_pixels(poses, calibrate_rig, None)
        cal = used_rig
        if lens_distortion is not None:
            pix, cal = inputs.undistort_pixels(pix, cal, lens, margin=margin)
        points, _ = inputs.triangulate(pix, cal)
        sigma_px = pixel_noise if pixel_noise > 0 else 1.0
        refined, _, rep = inputs.calibrate_rig(pix, cal, points, sigma_px=sigma_px, sigma_rot=sig_rot, sigma_pos=sig_pos,
                                               max_iters=CALIBRATE_MAX_ITERS)
        noisy_rig = used_rig
        used_rig = used_rig.clone()
        used_rig[:, :12] = refined[:, :12]                  # extrinsics only: the unshifted intrinsics stay
        ce1.record()
        torch.cuda.synchronize()
        cals = {"noisy": noisy_rig.cpu().numpy(), "calibrated": used_rig.cpu().numpy()}
        true_rig = rig_calib.cpu().numpy()
        rig_report = dict(ms=ce0.elapsed_time(ce1), report=rep.cpu().numpy(), sigma_px=sigma_px,
                          errors={k: rig_errors(c, true_rig) for k, c in cals.items()},
                          aligned={k: rig_errors(c, true_rig, align=True) for k, c in cals.items()} if views >= 3 else None)

    assoc_acc = torch.zeros(8, dtype=torch.float64, device=dev) if people else None
    dropped = torch.zeros(1, dtype=torch.float64, device=dev) if people else None
    track_acc = torch.zeros(11, dtype=torch.float64, device=dev) if frames else None
    track_events = []                                  # (start, end) events around each micro-batch's tracking calls

    def person_rows(f0, nf, seqs=None):
        """The person rows of frames [f0, f0 + nf): (pixels and calibration for the lifter, the same for the triangulations,
        the owners' targets, the group of each row: 0 with an owner, -1 without).  With seqs = (first sequence, sequences),
        the frames of those sequences, whose rows are also tracked and scored."""
        P = people
        u0, nu, per = (f0, nf, 1) if seqs is None else (seqs[0], seqs[1], frames)     # cameras per frame or per sequence
        cams = inputs.synth_cameras(nu, views, rig_kind, seed=seed, start=u0, device=dev) if random_cameras else None
        if cams is None:
            calib = used_rig
        elif calib_noise is not None:
            calib = inputs.calibration_noise(cams, seed, u0, sig_rot, sig_pos)
        else:
            calib = cams
        if cams is not None and per > 1:
            cams, calib = cams.repeat_interleave(per, 0), calib.repeat_interleave(per, 0)
        pix, target = synth_pixels(f0 * P, nf * P, None if cams is None else cams.repeat_interleave(P, 0), seqs)
        scene, perm = inputs.synth_people(pix, P, seed, f0)
        rows_calib = calib if calib.dim() == 2 else calib.repeat_interleave(P, 0)   # frame f's cameras for its slots and rows
        scene_t, tri_calib = scene, rows_calib
        if lens_distortion is not None:
            u, tri_calib = inputs.undistort_pixels(scene.view(nf * P, views, cfg.J, 3), rows_calib, lens, margin=margin)
            scene_t = u.view(scene.shape)
        members, labels, npeople = inputs.associate_people(
            scene_t, tri_calib if tri_calib.dim() == 2 else tri_calib[::P], min_joints=assoc_min_joints,
            max_dist=assoc_max_dist, max_people=P)
        owner, _ = inputs.association_score(members, labels, perm, assoc_acc)
        dropped.add_((npeople - P).clamp(min=0).sum().to(torch.float64))
        rows = inputs.gather_people(scene, members).view(nf * P, views, cfg.J, 3)
        rows_t = rows if scene_t is scene else inputs.gather_people(scene_t, members).view(nf * P, views, cfg.J, 3)
        idx = owner.clamp(min=0).long()[:, :, None, None].expand(nf, P, cfg.J, 3)
        target = target.view(nf, P, cfg.J, 3).gather(1, idx).view(nf * P, cfg.J, 3)
        group = torch.where(owner >= 0, 0, -1).to(torch.int32).view(-1)
        if seqs is not None:
            points, _ = inputs.triangulate_robust(rows_t, tri_calib, inlier_px=inlier_px)
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
            ids, _ = inputs.track_people(points.view(seqs[1], frames, P, cfg.J, 3), min_joints=assoc_min_joints,
                                         max_dist=track_max_dist, max_age=track_max_age, max_tracks=2 * P)
            inputs.tracking_score(ids, owner.view(seqs[1], frames, P), P, track_acc)
            ev[1].record()
            track_events.append(ev)
        return rows, rows_calib, (rows_t, tri_calib), target, group

    def step(s0, n):
        g, tri = {}, None
        if frames:
            pix, calib, tri, target, group = person_rows(s0 * frames, n * frames, (s0, n))
            g = {"group": group}
        elif people:
            pix, calib, tri, target, group = person_rows(s0, n)
            g = {"group": group}
        else:
            cams = inputs.synth_cameras(n, views, rig_kind, seed=seed, start=s0, device=dev) if random_cameras else None
            pix, target = synth_pixels(s0, n, cams)
            if cams is None:
                calib = used_rig
            elif calib_noise is not None:
                calib = inputs.calibration_noise(cams, seed, s0, sig_rot, sig_pos)
            else:
                calib = cams
        p, r, c = inputs.build_inputs(pix, calib)
        with torch.no_grad():
            out = model(p, rays=r, centers=c)
        out = out[0] if isinstance(out, tuple) else out
        acc.update(out, target, **g)
        pacc.update(out, target, **g)
        def score(key, a, points, mask):
            a.update(points, target, mask, **g)
            if key in tp:
                tp[key].update(points, target, mask, **g)

        if tri is not None:
            pix, calib = tri
        elif lens_distortion is not None and (tacc is not None or racc is not None):
            pix, calib = inputs.undistort_pixels(pix, calib, lens, margin=margin)
        if tacc is not None:
            points, used = inputs.triangulate(pix, calib)
            score("t", tacc, points, used >= 2)
            if tfacc is not None:
                score("tf", tfacc, inputs.refine_triangulation(pix, calib, points, max_iters=REFINE_MAX_ITERS)[0], used >= 2)
        if racc is not None:
            points, inl = inputs.triangulate_robust(pix, calib, inlier_px=inlier_px)
            score("r", racc, points, inl != 0)         # popcount >= 2: a non-zero inlier mask has at least two bits
            if rfacc is not None:
                score("rf", rfacc, inputs.refine_triangulation(pix, calib, points, view_mask=inl,
                                                                 max_iters=REFINE_MAX_ITERS)[0], inl != 0)

    for _ in range(warmup):                            # allocate the workspace, pack the weights
        step(start, min(micro_batch, max(stop - start, 1)))
    acc.acc.zero_()
    pacc.acc.zero_()
    for a in (tacc, racc, tfacc, rfacc, *tp.values()):
        if a is not None:
            a.acc.zero_()
    if people:
        assoc_acc.zero_()
        dropped.zero_()
    if frames:
        track_acc.zero_()
        track_events.clear()
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s0 in range(start, stop, micro_batch):
        step(s0, min(micro_batch, stop - s0))
    acc.all_reduce()                                   # the only collectives of the whole job:
    pacc.all_reduce()                                  # 11 J + 1 and J + 3 doubles
    for a in (tacc, racc, tfacc, rfacc, *tp.values()):
        if a is not None:
            a.all_reduce()
    if people and world > 1:
        torch.distributed.all_reduce(assoc_acc)
        torch.distributed.all_reduce(dropped)
        if frames:
            torch.distributed.all_reduce(track_acc)
    e1.record()
    torch.cuda.synchronize()
    ms = mdist.max_over_ranks(e0.elapsed_time(e1), dev)
    res, pres = acc.result(), pacc.result()
    line = None
    if rank == 0:
        line = {
            "metric": "poses/sec end-to-end synthetic evaluation (generate + project + build inputs + forward + MPJPE)",
            "value": poses / (ms / 1000.0), "unit": "poses/s", "n_gpus": world, "ms_total": ms, "poses": res["n"],
            "dtype": precision, "data": "synthetic (device generator keyed by global pose index)",
            "config": {"workload": f"{arch} V={views} depth={depth} D={cfg.fpt_dim} tokens={cfg.fpt_tokens}",
                       "micro_batch": micro_batch, "rig": rig or DEFAULT_RIG[arch], "flops_per_pose": spec.flops_per_pose(cfg)},
            "mpjpe_cm": {"absolute": res["mpjpe_abs"], "root_relative": res["mpjpe_rel"], "procrustes_aligned": pres["p_mpjpe"],
                         "note": "random-init weights: exercises the metric path, not a trained accuracy"},
            "tflops": poses / (ms / 1000.0) * spec.flops_per_pose(cfg) / 1e12 / world,
        }
        if noisy:
            line["data"] = {"source": line["data"], "pixel_noise_px": pixel_noise, "outlier_rate": outlier_rate,
                            "miss_rate": miss_rate,
                            "noise_model": "Gaussian of std pixel_noise_px / conf; outliers uniform in the image with conf "
                                           "0.3-1; misses set conf 0"}
        if random_cameras:
            if not isinstance(line["data"], dict):
                line["data"] = {"source": line["data"]}
            line["data"]["cameras"] = {
                "model": "random per sequence (mpl_synth_cameras, keyed by global sequence index)" if frames else
                         "random per pose (mpl_synth_cameras, keyed by global pose index)", "rig_kind": rig_kind,
                "azimuth": "2 pi (v + 0.8 (U0 - 0.5)) / V + 0.3", "distance_m": "4.5 (0.75 + 0.5 U1)",
                "height_m": "0.9 + 1.2 U2", "look_at": "room centre at 0.9 m + 0.5 (U3 - 0.5, U4 - 0.5, 0)",
                "focal_px": "f0 (0.8 + 0.4 U5), f0 of the rig kind"}
        if lens_distortion is not None:
            if not isinstance(line["data"], dict):
                line["data"] = {"source": line["data"]}
            line["data"]["lens_distortion"] = {
                "model": "OpenCV 5-coefficient Brown-Conrady on normalised camera coordinates, every view",
                "coefficients": dict(zip(("k1", "k2", "p1", "p2", "k3"), lens_distortion)),
                "pipeline": "projected pixels distorted before the detector noise; lifter inputs built from the distorted "
                            "pixels; triangulations on the undistorted pixels (margin half the image on each side)"}
        if calib_noise is not None:
            if not isinstance(line["data"], dict):
                line["data"] = {"source": line["data"]}
            line["data"]["calibration_noise"] = {
                "rotation_deg": calib_noise[0], "position_mm": calib_noise[1],
                "model": "per camera R' = Exp(w) R with w ~ N(0, rotation_deg^2 I) (camera frame), centre + N(0, "
                         "position_mm^2 I); the pixels are projected through the true cameras, every other step uses the "
                         "perturbed ones" + ("" if random_cameras else "; one perturbation of the rig (pose 0)")}
        if rig_report is not None:
            rp = rig_report["report"]
            line["rig_calibration"] = {
                "poses": calibrate_rig, "global_indices": [poses, poses + calibrate_rig], "items": int(rp[0]),
                "observations": int(rp[1]), "iterations": int(rp[6]), "accepted_steps": int(rp[7]),
                "rms_px": {"before": float(rp[4]), "after": float(rp[5])}, "sigma_px": rig_report["sigma_px"],
                "rotation_error_deg": {k: e[0] for k, e in rig_report["errors"].items()},
                "centre_error_mm": {k: e[1] for k, e in rig_report["errors"].items()},
                "method": f"Levenberg-Marquardt bundle adjustment of the extrinsics and the joints, Gaussian prior of "
                          f"--calib-noise, at most {CALIBRATE_MAX_ITERS} iterations, from the linear triangulation",
                "ms": rig_report["ms"], "note": "ms is not part of ms_total"}
            if rig_report["aligned"] is not None:
                line["rig_calibration"]["after_similarity_alignment"] = {
                    "rotation_error_deg": {k: e[0] for k, e in rig_report["aligned"].items()},
                    "centre_error_mm": {k: e[1] for k, e in rig_report["aligned"].items()},
                    "note": "each rig mapped into the true frame by the similarity fitting its centres to the true ones: "
                            "the images do not observe the world frame, so the bundle adjustment leaves that similarity "
                            "where the prior puts it"}
        if people:
            line["association"] = association_summary(assoc_acc.cpu().numpy(), float(dropped.item()), res["n"], people,
                                                      assoc_max_dist, assoc_min_joints)
        if frames:
            line["tracking"] = tracking_summary(track_acc.cpu().numpy(), sum(a.elapsed_time(b) for a, b in track_events),
                                                people, frames, track_max_dist, track_max_age, assoc_min_joints, inlier_px)
        # .reshape(-1): the sums of the one group with people
        if tacc is not None:
            line["triangulation"] = triangulation_summary(tacc.acc.detach().cpu().numpy().reshape(-1), cfg.J)
        if racc is not None:
            line["triangulation_robust"] = triangulation_summary(
                racc.acc.detach().cpu().numpy().reshape(-1), cfg.J,
                method=f"pair RANSAC, MSAC cost at {inlier_px:g} px, conf-weighted DLT refit over the inliers")
        for entry, a, views in (("triangulation", tfacc, "the candidate views"), ("triangulation_robust", rfacc, "the inliers")):
            if a is not None:
                line[entry]["refined"] = triangulation_summary(
                    a.acc.detach().cpu().numpy().reshape(-1), cfg.J,
                    method=f"Levenberg-Marquardt on the reprojection error over {views}, weights conf^2, "
                           f"at most {REFINE_MAX_ITERS} iterations")
        for key, entry, sub in (("t", "triangulation", None), ("r", "triangulation_robust", None),
                                ("tf", "triangulation", "refined"), ("rf", "triangulation_robust", "refined")):
            if key in tp:
                r = tp[key].result()
                target_entry = line[entry] if sub is None else line[entry][sub]
                target_entry["procrustes_aligned"] = {"p_mpjpe_cm": r["p_mpjpe"], "aligned_poses": r["aligned"],
                                                      "skipped_poses": r["skipped"]}
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    return line


def rig_errors(calib, true_calib, align=False):
    """Per view: rotation error (degrees, the angle of R R_true^T) and centre error (mm) of calib [V, 18] against true_calib.

    align: first map calib into the true rig's frame by the similarity that best fits its centres onto the true ones
    (Umeyama; needs V >= 3).  Images do not observe the world frame, so a bundle adjustment leaves the rig's 7-DoF
    similarity where its prior puts it; the aligned errors measure what it can observe."""
    if align:
        src, dst = true_calib[:, 9:12], calib[:, 9:12]              # dst ~ s Q src + t
        ms, md = src.mean(0), dst.mean(0)
        U, S, Vt = np.linalg.svd((dst - md).T @ (src - ms))
        D = np.diag([1.0, 1.0, np.sign(np.linalg.det(U @ Vt))])
        Q = U @ D @ Vt
        s = np.trace(np.diag(S) @ D) / ((src - ms) ** 2).sum()
        calib = calib.copy()
        calib[:, 9:12] = (dst - (md - s * Q @ ms)) @ Q / s
        calib[:, :9] = (calib[:, :9].reshape(-1, 3, 3) @ Q).reshape(-1, 9)
    R, Rt = calib[:, :9].reshape(-1, 3, 3), true_calib[:, :9].reshape(-1, 3, 3)
    fro = np.linalg.norm((R - Rt).reshape(len(R), 9), axis=1)        # |R - R_true|_F = 2 sqrt(2) sin(angle / 2)
    ang = np.degrees(2.0 * np.arcsin(np.minimum(fro / (2.0 * np.sqrt(2.0)), 1.0)))
    pos = 1000.0 * np.linalg.norm(calib[:, 9:12] - true_calib[:, 9:12], axis=1)
    return [float(a) for a in ang], [float(p) for p in pos]


def association_summary(acc, dropped, scored_rows, people, max_dist, min_joints):
    """The association entry of the JSON line from the 8 sums of mpl_association_score."""
    def ratio(a, b):
        return float(a / b) if b > 0 else float("nan")

    names = ("frames", "associable_people", "rows", "pure_rows", "complete_rows", "predicted_pairs", "correct_pairs",
             "true_pairs")
    out = {k: int(round(float(v))) for k, v in zip(names, acc)}
    out.update(pair_precision=ratio(acc[6], acc[5]), pair_recall=ratio(acc[6], acc[7]), pure_fraction=ratio(acc[3], acc[2]),
               complete_fraction=ratio(acc[4], acc[1]), dropped_past_k=int(round(dropped)), scored_rows=scored_rows,
               parameters={"people_per_frame": people, "K": people, "max_dist_m": max_dist, "min_joints": min_joints,
                           "min_conf": 0.0},
               method="median line distance of the candidate joints' rays per cross-view pair, greedy complete linkage",
               note="pure_fraction: pure rows over rows; complete_fraction: complete rows over associable people; rows "
                    "without an owner add nothing to the metrics")
    return out


def tracking_summary(acc, ms, people, frames, max_dist, max_age, min_joints, inlier_px):
    """The tracking entry of the JSON line from the 11 sums of mpl_tracking_score."""
    def ratio(a, b):
        return float(a / b) if b > 0 else float("nan")

    names = ("sequences", "frames", "objects", "matches", "misses", "false_positives", "id_switches", "fragmentations",
             "mostly_tracked", "mostly_lost", "tracks")
    out = {k: int(round(float(v))) for k, v in zip(names, acc)}
    persons = acc[0] * people
    out.update(mota=1.0 - ratio(acc[4] + acc[5] + acc[6], acc[2]), mostly_tracked_fraction=ratio(acc[8], persons),
               mostly_lost_fraction=ratio(acc[9], persons), tracks_per_person=ratio(acc[10], persons),
               parameters={"frames_per_sequence": frames, "fps": FPS, "people": people, "max_dist_m": max_dist,
                           "max_age_frames": max_age, "min_joints": min_joints, "max_tracks": 2 * people},
               motion="per person: root on a sinusoid in x and y inside the room (0.03-0.1 Hz), fixed height, heading "
                      "turning at most 0.5 rad/s, fixed body (mpl_synth_motion)",
               method=f"robust triangulation of the person rows (inlier {inlier_px:g} px), then greedy matching of the "
                      f"median joint distance to each track's last observed joints, from a fresh state per sequence",
               ms=ms, note="ms: device time of mpl_track_people and mpl_tracking_score (with the state's zeroing); ms_total "
                           "includes it and the triangulation for the tracker")
    return out


def triangulation_summary(acc, J, method="linear DLT, pixel-space rows, views with conf > 0 inside the image"):
    """The triangulation entry of the JSON line from the MPJPE sums of triangulated points masked by views_used >= 2.

    absolute / root_relative: the reference's masking convention (a masked joint adds zero error but counts as a pose).
    triangulated_joints: per joint, the error sum over its triangulated instances divided by their number (the x-count
    of the sums), averaged over the joints triangulated at least once.  dist_rel (NaN once a root is under-determined) is
    not reported; P-MPJPE over the triangulated joints is added by run(triangulation_pmpjpe=True).  For the robust triangulation the mask is "at least two
    inliers", so under_determined_joints counts the joints it rejected as well as those seen by fewer than two views.
    """
    res = metric.finalize(acc, J)
    cnt = np.asarray(acc[8 * J:11 * J:3], dtype=np.float64)
    seen = cnt > 0
    per_joint = np.asarray(acc[0:J], dtype=np.float64)[seen] / cnt[seen]
    return {"mpjpe_cm": {"absolute": res["mpjpe_abs"], "root_relative": res["mpjpe_rel"],
                         "triangulated_joints": float(per_joint.mean()) if seen.any() else float("nan")},
            "under_determined_joints": int(round(res["n"] * J - float(cnt.sum()))),
            "method": method,
            "note": "ms_total includes the triangulation and its accumulator"}


def main(argv=None):
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--arch", default="hm0", choices=sorted(ARCHS))
    p.add_argument("--views", type=int, default=4)
    p.add_argument("--depth", type=int, default=None)
    p.add_argument("--poses", type=int, default=1 << 20, help="global number of poses (sharded over ranks)")
    p.add_argument("--micro-batch", type=int, default=65536)
    p.add_argument("--precision", default="bf16", choices=["bf16", "tf32", "fp32"])
    p.add_argument("--rig", default=None, choices=[None, "h36m", "cmu"])
    p.add_argument("--seed", type=int, default=1)
    p.add_argument("--triangulate", action="store_true", help="also score the linear triangulation of the same pixels")
    p.add_argument("--triangulate-robust", action="store_true",
                   help="also score the robust (pair RANSAC + conf-weighted refit) triangulation of the same pixels")
    p.add_argument("--inlier-px", type=float, default=10.0, help="inlier threshold of --triangulate-robust, pixels")
    p.add_argument("--pixel-noise", type=float, default=0.0, metavar="PX",
                   help="detector noise: Gaussian pixel error of std PX / conf")
    p.add_argument("--outlier-rate", type=float, default=0.0, metavar="P",
                   help="detector noise: share of confident false detections")
    p.add_argument("--miss-rate", type=float, default=0.0, metavar="P", help="detector noise: share of missed detections")
    p.add_argument("--random-cameras", action="store_true",
                   help="a random camera setup per pose (around the room of --rig) instead of one ring for all poses")
    p.add_argument("--refine-triangulations", action="store_true",
                   help="also score each triangulation refined by Levenberg-Marquardt on the conf^2-weighted reprojection "
                        "error (needs --triangulate or --triangulate-robust)")
    p.add_argument("--triangulation-pmpjpe", action="store_true",
                   help="also score each triangulation by P-MPJPE, aligned on its triangulated joints only (needs "
                        "--triangulate or --triangulate-robust)")
    p.add_argument("--lens-distortion", default=None, metavar="K1,K2,P1,P2,K3",
                   help="a lens of OpenCV's 5-coefficient model on every view: distorted detections for the lifter, "
                        "undistorted ones for the triangulations")
    p.add_argument("--calib-noise", default=None, metavar="ROT_DEG,POS_MM",
                   help="perturb the calibration every step but the projection uses: Gaussian rotation of std ROT_DEG "
                        "degrees per axis and centre error of std POS_MM mm per axis, per camera")
    p.add_argument("--calibrate-rig", type=int, default=0, metavar="N",
                   help="recalibrate the perturbed rig's extrinsics by bundle adjustment on N extra poses before the "
                        "evaluation (needs --calib-noise with both values > 0, not --random-cameras, N <= --micro-batch)")
    p.add_argument("--people", type=int, default=0, metavar="P",
                   help="P >= 2 people per frame in random detection slots, associated across views before every metric "
                        "(not with --calibrate-rig)")
    p.add_argument("--assoc-max-dist", type=float, default=0.1, metavar="M",
                   help="association: largest median ray distance of a linked pair, world units (m)")
    p.add_argument("--assoc-min-joints", type=int, default=3, metavar="N",
                   help="association: candidate joints a detection needs, and joints a pair must share")
    p.add_argument("--frames", type=int, default=0, metavar="T",
                   help="sequences of T >= 2 frames of people that move, tracked across frames (needs --people; "
                        "--micro-batch >= T P)")
    p.add_argument("--track-max-dist", type=float, default=0.2, metavar="M",
                   help="tracking: largest median joint distance of a track and a row it matches, world units (m)")
    p.add_argument("--track-max-age", type=int, default=5, metavar="N",
                   help="tracking: missed frames after which a track is dropped")
    a = p.parse_args(argv)
    if a.frames:
        if not a.people:
            p.error("--frames needs --people")
        if a.frames < 2:
            p.error("--frames needs T >= 2")
        if a.micro_batch < a.frames * a.people:
            p.error("--micro-batch must hold at least one sequence of --frames x --people person-frames")
        if not (np.isfinite(a.track_max_dist) and a.track_max_dist > 0):
            p.error("--track-max-dist needs a finite value > 0")
        if a.track_max_age < 0:
            p.error("--track-max-age needs N >= 0")
    if a.people:
        if a.people < 2:
            p.error("--people needs P >= 2")
        if a.people * a.views > 128:
            p.error("--people P needs P * --views <= 128")
        if a.calibrate_rig:
            p.error("--calibrate-rig cannot be used with --people")
        if not (np.isfinite(a.assoc_max_dist) and a.assoc_max_dist > 0):
            p.error("--assoc-max-dist needs a finite value > 0")
        if not 1 <= a.assoc_min_joints <= 17:
            p.error("--assoc-min-joints needs 1 <= N <= 17")
        if a.micro_batch < a.people:
            p.error("--micro-batch must hold at least one frame of --people persons")
    cnoise = None
    if a.calib_noise is not None:
        try:
            cnoise = tuple(float(x) for x in a.calib_noise.split(","))
        except ValueError:
            cnoise = ()
        if len(cnoise) != 2 or not all(np.isfinite(cnoise)) or min(cnoise) < 0:
            p.error("--calib-noise needs two comma-separated finite numbers >= 0: ROT_DEG,POS_MM")
    if a.calibrate_rig:
        if cnoise is None or min(cnoise) <= 0:
            p.error("--calibrate-rig needs --calib-noise with both values > 0")
        if a.random_cameras:
            p.error("--calibrate-rig calibrates one fixed rig: it cannot be used with --random-cameras")
        if not 1 <= a.calibrate_rig <= a.micro_batch:
            p.error("--calibrate-rig N needs 1 <= N <= --micro-batch")
    lens = None
    if a.lens_distortion is not None:
        try:
            lens = tuple(float(k) for k in a.lens_distortion.split(","))
        except ValueError:
            lens = ()
        if len(lens) != 5 or not all(np.isfinite(lens)):
            p.error("--lens-distortion needs five comma-separated finite numbers K1,K2,P1,P2,K3")
    if a.refine_triangulations and not (a.triangulate or a.triangulate_robust):
        p.error("--refine-triangulations needs --triangulate or --triangulate-robust")
    if a.triangulation_pmpjpe and not (a.triangulate or a.triangulate_robust):
        p.error("--triangulation-pmpjpe needs --triangulate or --triangulate-robust")
    run(a.arch, a.views, a.depth, a.poses, a.micro_batch, a.precision, a.rig, a.seed, triangulate=a.triangulate,
        pixel_noise=a.pixel_noise, outlier_rate=a.outlier_rate, miss_rate=a.miss_rate,
        triangulate_robust=a.triangulate_robust, inlier_px=a.inlier_px, random_cameras=a.random_cameras,
        refine_triangulations=a.refine_triangulations, triangulation_pmpjpe=a.triangulation_pmpjpe, lens_distortion=lens,
        calib_noise=cnoise, calibrate_rig=a.calibrate_rig, people=a.people, assoc_max_dist=a.assoc_max_dist,
        assoc_min_joints=a.assoc_min_joints, frames=a.frames, track_max_dist=a.track_max_dist,
        track_max_age=a.track_max_age)


if __name__ == "__main__":
    sys.exit(main())
