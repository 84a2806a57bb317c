"""Synthetic multi-view inputs for the MPL lifter forward (SURVEY.md §8d).

Produces exactly the tensors the reference dataset hands to the model
(`MPL/lib/dataset/joints_dataset_mpl.py:443-811`), from synthetic 3D poses and
synthetic ring-camera calibrations:

* 3D pose: root uniform in the YAML room, other joints root + N(0, 0.25 m)
* projection `x_cam = R X + T_ext`, `u = K x_cam / z`   (`MPL/lib/utils/calib.py:42-77`)
* clip to the image and zero the confidence of clipped joints (`joints_dataset_mpl.py:701-715`)
* screen normalisation `(u / w) * 2 - [1, h / w]`          (`joints_dataset_mpl.py:817-820`)
* intrinsics normalised the same way                      (`joints_dataset_mpl.py:615-623`)
* rays `R^T [(x-cx)/fx, (y-cy)/fy, 1] + t`, centers `t^T` (`joints_dataset_mpl.py:638-648,872-898`)

The generator is counter based: pose `i` of seed `s` is the same whatever the
batch size or the rank that asks for it (Philox counter = i * blocks-per-pose),
so sharding over ranks yields identical data to a single-GPU run.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np

NUM_JOINTS = 17


@dataclass(frozen=True)
class Rig:
    """V ring cameras looking at the room centre (all angles in radians, lengths in metres)."""
    R: np.ndarray          # [V,3,3] world -> camera rotation
    t: np.ndarray          # [V,3]   camera position in the world ("USE_T" convention: the model's `centers`)
    f: np.ndarray          # [V,2]   focal length, pixels
    c: np.ndarray          # [V,2]   principal point, pixels
    image_size: tuple      # (w, h) pixels
    room: tuple            # (min_x, max_x, min_y, max_y) metres

    @property
    def num_views(self) -> int:
        return self.R.shape[0]


# rig kind -> (focal length px, image (w, h) px, room (min_x, max_x, min_y, max_y) m)
RIG_KINDS = {"h36m": (1145.0, (1000, 1000), (-1.0, 1.0, -1.5, 2.0)),   # hm_0 yaml:47-50,89-91
             "cmu": (1400.0, (1920, 1080), (-2.0, 0.3, -0.8, 0.8))}     # cmu_0 yaml:85-87


def rig_kind(kind: str) -> tuple:
    """(f0, (w, h), room) of a rig kind."""
    if kind not in RIG_KINDS:
        raise ValueError(f"unknown rig kind {kind!r}")
    return RIG_KINDS[kind]


def make_rig(num_views: int, kind: str = "h36m") -> Rig:
    """Ring of cameras, radius 4.5 m, height 1.5 m, looking at the room centre.

    kind "h36m": f=1145 px, 1000x1000 image, room -1..1 x -1.5..2  (hm_0 yaml:47-50,89-91)
    kind "cmu" : f=1400 px, 1920x1080 image, room -2..0.3 x -0.8..0.8 (cmu_0 yaml:85-87)
    """
    f0, (w, h), room = rig_kind(kind)
    centre = np.array([(room[0] + room[1]) / 2, (room[2] + room[3]) / 2, 0.9])
    Rs, ts = [], []
    for v in range(num_views):
        ang = 2 * math.pi * v / num_views + 0.3
        pos = np.array([centre[0] + 4.5 * math.cos(ang), centre[1] + 4.5 * math.sin(ang), 1.5])
        z = centre - pos
        z /= np.linalg.norm(z)                       # optical axis
        x = np.cross(z, np.array([0.0, 0.0, 1.0]))
        x /= np.linalg.norm(x)
        y = np.cross(z, x)                           # image y points down
        Rs.append(np.stack([x, y, z]))               # rows = camera axes in world coords
        ts.append(pos)
    V = num_views
    return Rig(R=np.stack(Rs), t=np.stack(ts), f=np.full((V, 2), f0), c=np.tile([w / 2.0, h / 2.0], (V, 1)),
               image_size=(w, h), room=room)


def cameras_from_uniforms(U, f0: float, image_size, room) -> np.ndarray:
    """[..., V, 18] calibrations (`inputs.pack_calibration` rows) of the camera model of `mpl_synth_cameras` from U [..., V, 6].

    Azimuth 2 pi (v + 0.8 (U0 - 0.5)) / V + 0.3, horizontal distance 4.5 (0.75 + 0.5 U1) m from the look-at point, height
    0.9 + 1.2 U2 m, look-at point the room centre at height 0.9 shifted by 0.5 (U3 - 0.5) in x and 0.5 (U4 - 0.5) in y,
    fx = fy = f0 (0.8 + 0.4 U5), principal point at the image centre, R the look-at rotation of `make_rig`.  Every U = 0.5
    gives `make_rig`'s camera.
    """
    U = np.asarray(U, dtype=np.float64)
    V = U.shape[-2]
    w, h = (float(x) for x in image_size)
    v = np.arange(V, dtype=np.float64)
    ang = 2 * math.pi * (v + 0.8 * (U[..., 0] - 0.5)) / V + 0.3
    dist = 4.5 * (0.75 + 0.5 * U[..., 1])
    at = np.stack([np.broadcast_to((room[0] + room[1]) / 2 + 0.5 * (U[..., 3] - 0.5), ang.shape),
                   np.broadcast_to((room[2] + room[3]) / 2 + 0.5 * (U[..., 4] - 0.5), ang.shape),
                   np.full(ang.shape, 0.9)], axis=-1)
    pos = np.stack([at[..., 0] + dist * np.cos(ang), at[..., 1] + dist * np.sin(ang), 0.9 + 1.2 * U[..., 2]], axis=-1)
    z = at - pos
    z /= np.linalg.norm(z, axis=-1, keepdims=True)
    x = np.cross(z, np.array([0.0, 0.0, 1.0]))
    x /= np.linalg.norm(x, axis=-1, keepdims=True)
    y = np.cross(z, x)
    f = f0 * (0.8 + 0.4 * U[..., 5:6])
    lead = U.shape[:-1]
    return np.concatenate([x, y, z, pos, f, f, np.broadcast_to([w / 2, h / 2, w, h], lead + (4,))], axis=-1)


def random_cameras(batch: int, num_views: int, kind: str = "h36m", seed: int = 0, start: int = 0) -> np.ndarray:
    """Host twin of `mpl_synth_cameras`: [B, V, 18] float64 calibrations of poses [start, start + batch), random camera
    setups around the room of rig `kind` (`cameras_from_uniforms`).  U0..U5 of (pose i, view v) come from the Philox4x64-10
    stream under key (seed, 2) (pose i owns counter blocks [i nb, (i+1) nb), nb = ceil(6 V / 4), slot 6 v + m is U_m), so
    pose i's cameras depend only on (seed, start + i)."""
    f0, image_size, room = rig_kind(kind)
    U = _uniforms(seed, start, batch, 6 * num_views, key1=2).reshape(batch, num_views, 6)
    return cameras_from_uniforms(U, f0, image_size, room)


def so3_exp(w) -> np.ndarray:
    """Rodrigues' formula Exp(w) = I + sin t / t [w]x + (1 - cos t) / t^2 [w]x^2, t = |w|, for w [..., 3] -> [..., 3, 3]; below
    t^2 = 1e-2 the coefficients come from their Taylor series through t^8, as on the device."""
    w = np.asarray(w, dtype=np.float64)
    t2 = (w * w).sum(-1)
    small = t2 < 1e-2
    with np.errstate(invalid="ignore", divide="ignore"):
        t = np.sqrt(t2)
        a = np.where(small, 1.0 - t2 / 6.0 * (1.0 - t2 / 20.0 * (1.0 - t2 / 42.0 * (1.0 - t2 / 72.0))), np.sin(t) / t)
        b = np.where(small, 0.5 * (1.0 - t2 / 12.0 * (1.0 - t2 / 30.0 * (1.0 - t2 / 56.0 * (1.0 - t2 / 90.0)))),
                     (1.0 - np.cos(t)) / t2)
    K = np.zeros(w.shape[:-1] + (3, 3))
    K[..., 0, 1], K[..., 0, 2], K[..., 1, 2] = -w[..., 2], w[..., 1], -w[..., 0]
    K[..., 1, 0], K[..., 2, 0], K[..., 2, 1] = w[..., 2], -w[..., 1], w[..., 0]
    K2 = w[..., :, None] * w[..., None, :] - t2[..., None, None] * np.eye(3)
    return np.eye(3) + a[..., None, None] * K + b[..., None, None] * K2


def calibration_noise(calib, seed: int, start: int, sigma_rot: float, sigma_pos: float) -> np.ndarray:
    """Host twin of `mpl_synth_calib_noise`: calib [V, 18] (a fixed rig, drawn as pose `start`) or [B, V, 18] (poses
    [start, start + B)) perturbed.  U0..U5 of (pose i, view v) come from the Philox4x64-10 stream under key (seed, 3)
    (slot layout of `random_cameras`); Box-Muller gives n_2k = r cos(2 pi U_2k+1), n_2k+1 = r sin(2 pi U_2k+1),
    r = sqrt(-2 ln max(U_2k, 1e-12)); R' = Exp(sigma_rot n0..2) R and t' = t + sigma_pos n3..5.  The intrinsics are copied, and a
    zero sigma keeps its field bit for bit."""
    calib = np.asarray(calib, dtype=np.float64)
    rig = calib.ndim == 2
    c = calib[None] if rig else calib
    B, V = c.shape[:2]
    U = _uniforms(seed, start, B, 6 * V, key1=3).reshape(B, V, 6)
    r = np.sqrt(-2.0 * np.log(np.maximum(U[..., 0::2], 1e-12)))
    th = 2 * math.pi * U[..., 1::2]
    n = np.empty((B, V, 6))
    n[..., 0::2], n[..., 1::2] = r * np.cos(th), r * np.sin(th)
    out = c.copy()
    if sigma_rot != 0:
        out[..., 0:9] = (so3_exp(sigma_rot * n[..., 0:3]) @ c[..., 0:9].reshape(B, V, 3, 3)).reshape(B, V, 9)
    if sigma_pos != 0:
        out[..., 9:12] = c[..., 9:12] + sigma_pos * n[..., 3:6]
    return out[0] if rig else out


def people_permutations(seed: int, start: int, frames: int, people: int, num_views: int) -> np.ndarray:
    """perm [F, V, P] int32 of `mpl_synth_people`: for frame start + f and view v, the person in each detection slot.  Frame
    i owns the counter blocks [i nb, (i + 1) nb), nb = ceil(V P / 4), of the Philox4x64-10 stream under key (seed, 4), and
    perm[f, v] is the stable ascending argsort of its uniforms in slots v P .. v P + P - 1."""
    U = _uniforms(seed, start, frames, num_views * people, key1=4).reshape(frames, num_views, people)
    return np.argsort(U, axis=-1, kind="stable").astype(np.int32)


def synth_people(pix, people: int, seed: int, start: int) -> tuple:
    """Host twin of `mpl_synth_people`: pix [F P, V, J, 3] with person p of frame f in row f P + p -> (scene [F, P, V, J, 3]
    with scene[f, s, v] = pix[f P + perm[f, v, s], v], perm [F, V, P] of `people_permutations`)."""
    pix = np.asarray(pix)
    B, V = pix.shape[:2]
    F = B // people
    perm = people_permutations(seed, start, F, people, V)
    rows = np.arange(F)[:, None, None] * people + perm                  # [F, V, P]
    scene = pix[rows, np.arange(V)[None, :, None]]                       # [F, V, P, J, 3]
    return np.ascontiguousarray(scene.transpose(0, 2, 1, 3, 4)), perm


def motion_joints(seed: int, start: int, sequences: int, frames: int, people: int, room, fps: float = 30.0,
                  num_joints: int = NUM_JOINTS) -> np.ndarray:
    """The 3D joints of `mpl_synth_motion`, fp64 [S, T, P, J, 3], for sequences [start, start + S).

    (sequence i, person p) owns the counter blocks of g = i P + p in the Philox4x64-10 stream under key (seed, 5), uniform
    slots U0..U8 then the Box-Muller pairs (u1_m, u2_m) at 9 + m and 9 + 3 (J - 1) + m.  With tau = t / fps:
    root x = (x0 + x1) / 2 + (0.25 + 0.25 U0) w_x sin(2 pi (0.03 + 0.07 U2) tau + 2 pi U4), y likewise with U1, U3, U5,
    z = 0.8 + 0.2 U6; heading theta = 2 pi U7 + (U8 - 0.5) tau; X_j = root + Rz(theta) o_j with synth_project's body o_j."""
    J = num_joints
    n = 3 * (J - 1)
    U = _uniforms(seed, start * people, sequences * people, 9 + 2 * n, key1=5).reshape(sequences, 1, people, 9 + 2 * n)
    x0, x1, y0, y1 = (float(r) for r in room)
    tau = (np.arange(frames, dtype=np.float64) / fps)[None, :, None]
    two_pi = 2 * math.pi
    ax, ay = (0.25 + 0.25 * U[..., 0]) * (x1 - x0), (0.25 + 0.25 * U[..., 1]) * (y1 - y0)
    fx, fy = 0.03 + 0.07 * U[..., 2], 0.03 + 0.07 * U[..., 3]
    px0, py0 = two_pi * U[..., 4], two_pi * U[..., 5]
    rx = 0.5 * (x0 + x1) + ax * np.sin(two_pi * fx * tau + px0)                      # [S, T, P]
    ry = 0.5 * (y0 + y1) + ay * np.sin(two_pi * fy * tau + py0)
    rz = np.broadcast_to(0.8 + 0.2 * U[..., 6], rx.shape)
    theta = two_pi * U[..., 7] + (U[..., 8] - 0.5) * tau
    c, s = np.cos(theta)[..., None], np.sin(theta)[..., None]
    u1 = np.maximum(U[..., 9:9 + n], 1e-12)
    u2 = U[..., 9 + n:9 + 2 * n]
    o = np.concatenate([np.zeros(U.shape[:-1] + (3,)), 0.25 * (np.sqrt(-2.0 * np.log(u1)) * np.cos(two_pi * u2))], axis=-1)
    o = o.reshape(U.shape[:-1] + (J, 3))                                              # [S, 1, P, J, 3]
    X = np.empty((sequences, frames, people, J, 3))
    X[..., 0] = rx[..., None] + (c * o[..., 0] - s * o[..., 1])
    X[..., 1] = ry[..., None] + (s * o[..., 0] + c * o[..., 1])
    X[..., 2] = rz[..., None] + o[..., 2]
    return X


def synth_motion(seed: int, start: int, sequences: int, frames: int, people: int, calib, room, fps: float = 30.0,
                 conf_mode: str = "uniform", num_joints: int = NUM_JOINTS) -> tuple:
    """Host twin of `mpl_synth_motion` -> (pix [S T P, V, J, 3] fp32, target [S T P, J, 3] fp32).

    Row r = ((start + s) T + t) P + p holds person p in frame t of sequence start + s (`motion_joints`), projected like
    `mpl_synth_project` through calib [V, 18] or one calibration per row [S T P, V, 18] (x_cam = R (X - t),
    u = f x_cam / z + c, no clipping, conf 0 behind the camera); conf 1 with conf_mode "ones", otherwise 0.3 + 0.7 U of
    `mpl_synth_project`'s confidence slots of pose r."""
    J = num_joints
    X = motion_joints(seed, start, sequences, frames, people, room, fps, J).reshape(-1, J, 3)
    B = len(X)
    calib = np.asarray(calib, dtype=np.float64)
    c = calib[None] if calib.ndim == 2 else calib                                     # [1 or B, V, 18]
    V = c.shape[1]
    R, t = c[..., :9].reshape(c.shape[0], V, 3, 3), c[..., 9:12]
    d = X[:, None, :, :] - t[:, :, None, :]                                           # [B, V, J, 3]
    xc = [R[:, :, None, r, 0] * d[..., 0] + R[:, :, None, r, 1] * d[..., 1] + R[:, :, None, r, 2] * d[..., 2] for r in range(3)]
    with np.errstate(divide="ignore", invalid="ignore"):
        u = xc[0] / xc[2] * c[:, :, None, 12] + c[:, :, None, 14]
        w = xc[1] / xc[2] * c[:, :, None, 13] + c[:, :, None, 15]
    if conf_mode == "ones":
        conf = np.ones((B, V, J))
    elif conf_mode == "uniform":
        n = 3 * (J - 1)
        conf = 0.3 + 0.7 * _uniforms(seed, start * frames * people, B, 3 + 2 * n + V * J)[:, 3 + 2 * n:].reshape(B, V, J)
    else:
        raise ValueError(conf_mode)
    conf = np.where(xc[2] > 0.0, conf, 0.0)
    pix = np.stack([u, w, conf], axis=-1).astype(np.float32)
    return pix, X.astype(np.float32)


def _uniforms(seed: int, start: int, count: int, per_pose: int, key1: int = 0) -> np.ndarray:
    """[count, per_pose] uniforms in [0,1); row i depends only on (seed, start+i).  Philox key (seed, key1)."""
    blocks = (per_pose + 3) // 4                      # Philox4x64: 4 outputs per counter step
    bg = np.random.Philox(key=seed if key1 == 0 else np.array([seed, key1], dtype=np.uint64))
    bg.advance(start * blocks)
    raw = bg.random_raw(count * blocks * 4).reshape(count, blocks * 4)[:, :per_pose]
    return (raw >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def make_batch(batch: int, rig: Rig, seed: int = 0, start: int = 0, conf_mode: str = "uniform",
               dtype=np.float32) -> dict:
    """Model inputs for poses [start, start+batch).

    Returns dict with `poses [B,V,17,3]` (x̂, ŷ, conf), `rays [B,V,17,3]`, `centers [B,V,1,3]`,
    `target [B,17,3]` (metres, OUTPUT_IN_METER convention) — all `dtype`.
    """
    V, J = rig.num_views, NUM_JOINTS
    per_pose = 3 + 2 * 3 * (J - 1) + V * J
    u = _uniforms(seed, start, batch, per_pose)
    room = rig.room
    root = np.stack([room[0] + u[:, 0] * (room[1] - room[0]),
                     room[2] + u[:, 1] * (room[3] - room[2]),
                     0.8 + 0.2 * u[:, 2]], axis=1)                         # [B,3]
    n = 3 * (J - 1)
    u1 = np.maximum(u[:, 3:3 + n], 1e-12)
    u2 = u[:, 3 + n:3 + 2 * n]
    gauss = np.sqrt(-2.0 * np.log(u1)) * np.cos(2 * math.pi * u2)          # Box-Muller, fixed draw count
    target = np.concatenate([root[:, None, :], root[:, None, :] + 0.25 * gauss.reshape(batch, J - 1, 3)], axis=1)
    conf_u = u[:, 3 + 2 * n:].reshape(batch, V, J)

    w, h = rig.image_size
    # world -> camera -> pixels (calib.py:42-77), per view
    x_cam = np.einsum("vij,bkj->bvki", rig.R, target) - np.einsum("vij,vj->vi", rig.R, rig.t)[None, :, None, :]
    z = x_cam[..., 2:3]
    px = x_cam[..., :2] / z * rig.f[None, :, None, :] + rig.c[None, :, None, :]      # [B,V,J,2]
    # clip + confidence zeroing (joints_dataset_mpl.py:701-715)
    inside = (px[..., 0] > 0) & (px[..., 0] < w - 1) & (px[..., 1] > 0) & (px[..., 1] < h - 1) & (z[..., 0] > 0)
    if conf_mode == "uniform":
        conf = 0.3 + 0.7 * conf_u
    elif conf_mode == "ones":
        conf = np.ones_like(conf_u)
    else:
        raise ValueError(conf_mode)
    conf = np.where(inside, conf, 0.0)
    px = np.stack([np.clip(px[..., 0], 0, w - 1), np.clip(px[..., 1], 0, h - 1)], axis=-1)
    # screen normalisation (joints_dataset_mpl.py:817-820) of joints and intrinsics (:615-623)
    norm = np.array([1.0, h / w])
    xy = px / w * 2 - norm
    c_hat = rig.c / w * 2 - norm                                            # [V,2]
    f_hat = rig.f / w * 2
    # rays (joints_dataset_mpl.py:872-898) with USE_T: R^T [x, y, 1] + t ; centers = t^T (:645-646)
    cam_dir = np.concatenate([(xy - c_hat[None, :, None, :]) / f_hat[None, :, None, :],
                              np.ones((batch, V, J, 1))], axis=-1)
    rays = np.einsum("vji,bvkj->bvki", rig.R, cam_dir) + rig.t[None, :, None, :]
    centers = np.broadcast_to(rig.t[None, :, None, :], (batch, V, 1, 3))
    poses = np.concatenate([xy, conf[..., None]], axis=-1)
    return {"poses": np.ascontiguousarray(poses, dtype=dtype), "rays": np.ascontiguousarray(rays, dtype=dtype),
            "centers": np.ascontiguousarray(centers, dtype=dtype), "target": np.ascontiguousarray(target, dtype=dtype)}


def detector_noise(pix, image_size, seed: int, start: int, sigma_px: float, p_outlier: float, p_miss: float) -> np.ndarray:
    """Host twin of `mpl_synth_detector_noise`: the detector-error model applied to raw pixels of poses [start, start+B).

    pix [B,V,J,3] (u, v, conf) as `mpl_synth_project` writes them; image_size (w, h).  Returns a perturbed float32 copy.
    Entries with conf == 0 are kept.  Every other entry draws U0..U5 from the Philox4x64-10 stream under key (seed, 1)
    (pose i owns counter blocks [i nb, (i+1) nb), nb = ceil(6 V J / 4), slot (v J + j) 6 + m is U_m):
    U0 < p_miss -> conf = 0; U0 < p_miss + p_outlier -> (u, v) = (U3 (w-1), U4 (h-1)), conf = 0.3 + 0.7 U5;
    otherwise (u, v) += sigma_px / conf * sqrt(-2 ln max(U1, 1e-12)) (cos, sin)(2 pi U2).  The parameters are rounded to
    float32 first, as the C call receives them.
    """
    pix = np.asarray(pix, dtype=np.float32)
    B, V, J, _ = pix.shape
    w, h = (float(x) for x in image_size)
    sigma, po, pm = (float(np.float32(x)) for x in (sigma_px, p_outlier, p_miss))
    U = _uniforms(seed, start, B, 6 * V * J, key1=1).reshape(B, V, J, 6)
    u, v, conf = (pix[..., k].astype(np.float64) for k in range(3))
    live = conf != 0
    miss = live & (U[..., 0] < pm)
    out = live & ~miss & (U[..., 0] < pm + po)
    noisy = live & ~miss & ~out
    s = sigma / np.where(noisy, conf, 1.0) * np.sqrt(-2.0 * np.log(np.maximum(U[..., 1], 1e-12)))
    theta = 2 * math.pi * U[..., 2]
    res = pix.copy()
    res[..., 0] = np.where(out, U[..., 3] * (w - 1), np.where(noisy, u + s * np.cos(theta), u)).astype(np.float32)
    res[..., 1] = np.where(out, U[..., 4] * (h - 1), np.where(noisy, v + s * np.sin(theta), v)).astype(np.float32)
    res[..., 2] = np.where(miss, 0.0, np.where(out, 0.3 + 0.7 * U[..., 5], conf)).astype(np.float32)
    return res


def lens_map(k, x, y) -> tuple:
    """OpenCV's 5-coefficient model D(x, y) on normalised coordinates and its Jacobian: (xd, yd, a, b, d), J = [[a, b], [b, d]].
    k = (k1, k2, p1, p2, k3), each broadcastable against x, y; the arithmetic of `mpl_distort_pixels` in the same order."""
    k1, k2, p1, p2, k3 = k
    r2 = x * x + y * y
    rho = 1.0 + r2 * (k1 + r2 * (k2 + r2 * k3))
    drho = k1 + r2 * (2.0 * k2 + r2 * (3.0 * k3))
    xd = x * rho + 2.0 * p1 * x * y + p2 * (r2 + 2.0 * x * x)
    yd = y * rho + p1 * (r2 + 2.0 * y * y) + 2.0 * p2 * x * y
    a = rho + 2.0 * x * x * drho + 2.0 * p1 * y + 6.0 * p2 * x
    b = 2.0 * x * y * drho + 2.0 * p1 * x + 2.0 * p2 * y
    d = rho + 2.0 * y * y * drho + 6.0 * p1 * y + 2.0 * p2 * x
    return xd, yd, a, b, d


def lens_valid(k, x, y) -> np.ndarray:
    """The validity rule of include/mpl_b200.h: det J > 0 and the radial map r -> r rho(r) increasing on [0, |x|], i.e.
    g(s) = 1 + 3 k1 s + 5 k2 s^2 + 7 k3 s^3 > 0 at s = r^2 and at the roots of g' strictly inside (0, r^2)."""
    k1, k2, p1, p2, k3 = (np.asarray(c, dtype=np.float64) for c in k)
    x, y = np.asarray(x, dtype=np.float64), np.asarray(y, dtype=np.float64)
    _, _, a, b, d = lens_map((k1, k2, p1, p2, k3), x, y)
    r2 = x * x + y * y

    def g(s):
        return 1.0 + s * (3.0 * k1 + s * (5.0 * k2 + s * (7.0 * k3)))

    with np.errstate(invalid="ignore", divide="ignore"):
        ok = (a * d - b * b > 0.0) & (g(r2) > 0.0) & (r2 < np.inf)
        disc = 100.0 * k2 * k2 - 252.0 * k1 * k3
        sq = np.sqrt(np.where(disc >= 0.0, disc, 0.0))
        cubic, quad = (k3 != 0.0) & (disc >= 0.0), (k3 == 0.0) & (k2 != 0.0)
        roots = [np.where(cubic, (-10.0 * k2 - sq) / (42.0 * k3), np.where(quad, -3.0 * k1 / (10.0 * k2), np.nan)),
                 np.where(cubic, (-10.0 * k2 + sq) / (42.0 * k3), np.nan)]
        for s in roots:
            inside = (s > 0.0) & (s < r2)
            ok &= ~inside | (g(np.where(inside, s, 0.0)) > 0.0)
    return ok


def distort_pixels(pix, calib, dist) -> np.ndarray:
    """Host twin of `mpl_distort_pixels`: ideal pinhole pixels -> those a camera with lens `dist` records.

    pix [B, V, J, 3] (u, v, conf); calib [V, 18] or [B, V, 18] (`inputs.pack_calibration` rows); dist (k1, k2, p1, p2, k3)
    per view, [V, 5] or [B, V, 5].  Returns a float32 copy: each entry with conf != 0 at x = ((u - cx) / fx, (v - cy) / fy)
    moves to u + fx (x_d - x), v + fy (y_d - y), (x_d, y_d) = `lens_map`(x), or gets conf = 0 (pixel kept) where x fails
    `lens_valid`.  Entries with conf == 0, and entries whose five coefficients are all 0, are kept.
    """
    pix = np.asarray(pix, dtype=np.float32)
    calib = np.asarray(calib, dtype=np.float64)
    dist = np.asarray(dist, dtype=np.float64)
    c = calib[..., :, None, :] if calib.ndim == 3 else calib[None, :, None, :]      # [B or 1, V, 1, 18]
    k = dist[..., :, None, :] if dist.ndim == 3 else dist[None, :, None, :]
    k = tuple(k[..., m] for m in range(5))
    fx, fy, cx, cy = (c[..., m] for m in range(12, 16))
    u, v, conf = (pix[..., m].astype(np.float64) for m in range(3))
    x, y = (u - cx) / fx, (v - cy) / fy
    with np.errstate(invalid="ignore", over="ignore"):
        xd, yd, _, _, _ = lens_map(k, x, y)
        live = (conf != 0) & ~((k[0] == 0) & (k[1] == 0) & (k[2] == 0) & (k[3] == 0) & (k[4] == 0))
        ok = live & lens_valid(k, x, y)
        res = pix.copy()
        res[..., 0] = np.where(ok, u + fx * (xd - x), u).astype(np.float32)
        res[..., 1] = np.where(ok, v + fy * (yd - y), v).astype(np.float32)
    res[..., 2] = np.where(live & ~ok, np.float32(0.0), pix[..., 2])
    return res


def named_weights(shapes: dict, seed: int = 0, pos_std: float = 0.02) -> dict:
    """Deterministic weights keyed by parameter NAME (order independent, numpy only).

    Distributions follow the PyTorch defaults the reference relies on (SURVEY.md §3.2-Q5):
    Linear/Conv1d weight and bias ~ U(±1/sqrt(fan_in)); LayerNorm/BatchNorm weight 1 + small noise,
    bias small noise (so the affine paths are exercised); learned position embeddings ~ N(0, pos_std²)
    (zeros at reference init — randomised so the add paths are tested); BN running stats non-trivial.
    `shapes`: name -> (shape tuple, kind) with kind in {linear_w, linear_b, norm_w, norm_b, pos, bn_mean, bn_var, count}.
    """
    import zlib
    out = {}
    for name, (shape, kind, fan_in) in shapes.items():
        key = (zlib.crc32(name.encode()) << 20) ^ (seed & 0xFFFFF)
        rng = np.random.Generator(np.random.Philox(key=key))
        size = int(np.prod(shape)) if len(shape) else 1
        if kind in ("linear_w", "linear_b"):
            bound = 1.0 / math.sqrt(fan_in)
            a = (rng.random(size) * 2 - 1) * bound
        elif kind == "norm_w":
            a = 1.0 + 0.1 * (rng.random(size) * 2 - 1)
        elif kind == "norm_b":
            a = 0.05 * (rng.random(size) * 2 - 1)
        elif kind == "pos":
            a = pos_std * rng.standard_normal(size)
        elif kind == "bn_mean":
            a = 0.1 * (rng.random(size) * 2 - 1)
        elif kind == "bn_var":
            a = 0.5 + rng.random(size)
        elif kind == "count":
            out[name] = np.zeros(shape, dtype=np.int64)
            continue
        else:
            raise ValueError(kind)
        out[name] = a.astype(np.float32).reshape(shape)
    return out
