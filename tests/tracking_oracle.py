"""numpy restatement of mpl_track_people and mpl_tracking_score (include/mpl_b200.h), rule for rule, one sequence and one
frame at a time.  The joint distances are sqrt((dx dx + dy dy) + dz dz) in fp64 with every operation rounded, as the device
computes them, so the costs, and with them every id, must agree bit for bit."""
import numpy as np


class Track:
    def __init__(self, tid, pos, has):
        self.id, self.pos, self.has, self.misses = tid, pos, has, 0


def used_joints(rows, mask):
    """rows [K, J, 3] fp32, mask [K, J] or None -> [K, J] bool: finite, and mask None or > 0."""
    ok = np.isfinite(rows).all(-1)
    return ok if mask is None else ok & (mask > 0)


def cost(track, row, used, min_joints):
    """Median joint distance over the joints used in the row and remembered by the track; +inf below min_joints."""
    sh = used & track.has
    n = int(sh.sum())
    if n < min_joints:
        return np.inf
    d = row[sh].astype(np.float64) - track.pos[sh].astype(np.float64)
    dist = np.sort(np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2]))
    lo, hi = dist[(n - 1) // 2], dist[n // 2]
    return lo if n % 2 else 0.5 * (lo + hi)


class Tracker:
    """One sequence's state; `step` tracks one frame."""

    def __init__(self, max_tracks, min_joints=3, max_dist=0.2, max_age=5):
        self.max_tracks, self.min_joints, self.max_dist, self.max_age = max_tracks, min_joints, max_dist, max_age
        self.tracks, self.next_id = [], 0

    def step(self, rows, mask=None):
        """rows [K, J, 3] fp32 -> ids [K] int32."""
        rows = np.asarray(rows, dtype=np.float32)
        K = len(rows)
        used = used_joints(rows, mask)
        det = used.sum(1) >= self.min_joints
        pairs = []
        for tr in self.tracks:
            for k in range(K):
                c = cost(tr, rows[k], used[k], self.min_joints)
                if c <= self.max_dist:
                    pairs.append((c, tr.id * K + k, tr, k))
        pairs.sort(key=lambda p: (p[0], p[1]))
        ids = np.full(K, -1, dtype=np.int32)
        matched = set()
        for _, _, tr, k in pairs:
            if id(tr) in matched or ids[k] >= 0:
                continue
            matched.add(id(tr))
            ids[k] = tr.id
            tr.pos = np.where(used[k][:, None], rows[k], tr.pos)
            tr.has = tr.has | used[k]
            tr.misses = 0
        alive = []
        for tr in self.tracks:
            if id(tr) not in matched:
                tr.misses += 1
                if tr.misses > self.max_age:
                    continue
            alive.append(tr)
        self.tracks = alive
        for k in range(K):
            if ids[k] >= 0 or not det[k] or len(self.tracks) >= self.max_tracks:
                continue
            self.tracks.append(Track(self.next_id, np.where(used[k][:, None], rows[k], np.float32(0)), used[k].copy()))
            ids[k] = self.next_id
            self.next_id += 1
        return ids


def track(points, joint_mask=None, max_tracks=None, min_joints=3, max_dist=0.2, max_age=5, trackers=None):
    """points [S, T, K, J, 3] -> (track_id [S, T, K] int32, the per-sequence Trackers, to continue a later chunk)."""
    points = np.asarray(points, dtype=np.float32)
    S, T, K = points.shape[:3]
    if trackers is None:
        trackers = [Tracker(2 * K if max_tracks is None else max_tracks, min_joints, max_dist, max_age) for _ in range(S)]
    out = np.empty((S, T, K), dtype=np.int32)
    for s in range(S):
        for t in range(T):
            out[s, t] = trackers[s].step(points[s, t], None if joint_mask is None else joint_mask[s, t])
    return out, trackers


def score(track_id, owner, people):
    """acc [11] of mpl_tracking_score."""
    track_id, owner = np.asarray(track_id), np.asarray(owner)
    S, T, K = track_id.shape
    acc = np.zeros(11)
    acc[0], acc[1], acc[2] = S, S * T, S * T * people
    for s in range(S):
        acc[10] += 1 + max(int(track_id[s].max()), -1)
        acc[5] += int((track_id[s] >= 0).sum())
        for q in range(people):
            prev, last, m = None, None, 0
            for t in range(T):
                ks = [k for k in range(K) if owner[s, t, k] == q and track_id[s, t, k] >= 0]
                if not ks:
                    continue
                h = track_id[s, t, ks[0]]
                m += 1
                if prev is not None and h != prev:
                    acc[6] += 1
                if last is not None and last != t - 1:
                    acc[7] += 1
                prev, last = h, t
            acc[3] += m
            acc[8] += 5 * m >= 4 * T
            acc[9] += 5 * m < T
    acc[4] = acc[2] - acc[3]
    acc[5] -= acc[3]
    return acc
