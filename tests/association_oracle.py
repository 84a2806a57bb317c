"""numpy restatement of mpl_associate_people and mpl_association_score (include/mpl_b200.h): the pair costs, the greedy
complete-linkage clustering, the ranking, the outputs and the score, one frame at a time.

`associate` also flags a frame as *near* when a decision could flip under the last-bit differences between this arithmetic
and the device's (fused multiply-adds, the order of the sums): a pair cost within 1e-9 (relative) of max_dist, or two
admissible costs within 1e-9 of each other (their order in the greedy pass).  Outside near frames the device's members,
labels and people must be this oracle's bit for bit."""
import numpy as np

NEAR_REL = 1e-9


def pair_costs(scene, calib, min_conf, min_joints):
    """One frame: scene [P, V, J, 3], calib [V, 18] -> (cost [M, M] fp64, symmetric, +inf where undefined; active [M] bool),
    detection m = s V + v."""
    P, V, J, _ = scene.shape
    M = P * V
    det = np.asarray(scene, dtype=np.float32).reshape(M, J, 3)
    view = np.arange(M) % V
    c = np.asarray(calib, dtype=np.float64)[view]                        # [M, 18]
    u, w = det[..., 0].astype(np.float64), det[..., 1].astype(np.float64)
    with np.errstate(invalid="ignore"):
        cand = ((det[..., 2] > np.float32(min_conf)) & (0.0 < u) & (u < c[:, 16:17] - 1.0) & (0.0 < w)
                & (w < c[:, 17:18] - 1.0))
        x = (u - c[:, 14:15]) / c[:, 12:13]
        y = (w - c[:, 15:16]) / c[:, 13:14]
    R = c[:, :9].reshape(M, 3, 3)
    d = x[..., None] * R[:, None, 0, :] + y[..., None] * R[:, None, 1, :] + R[:, None, 2, :]      # R^T (x, y, 1)
    active = cand.sum(1) >= min_joints
    cost = np.full((M, M), np.inf)
    a, b = np.triu_indices(M, 1)
    keep = (view[a] != view[b]) & active[a] & active[b]
    a, b = a[keep], b[keep]
    lo = np.where(view[a] < view[b], a, b)
    hi = a + b - lo
    shared = cand[lo] & cand[hi]                                         # [n, J]
    n = shared.sum(1)
    ok = n >= min_joints
    lo, hi, shared, n = lo[ok], hi[ok], shared[ok], n[ok]
    if len(lo) == 0:
        return cost, active
    dist = line_distances(c[hi, 9:12] - c[lo, 9:12], d[lo], d[hi])      # [n, J]
    dist = np.sort(np.where(shared, dist, np.inf), axis=1)
    i1, i2 = (n - 1) // 2, n // 2
    med = 0.5 * (np.take_along_axis(dist, i1[:, None], 1)[:, 0] + np.take_along_axis(dist, i2[:, None], 1)[:, 0])
    cost[lo, hi] = med
    cost[hi, lo] = med
    return cost, active


def line_distances(dc, d1, d2):
    """Distance between the lines c1 + a d1 and c2 + b d2 (dc = c2 - c1 [n, 3], d1 / d2 [n, J, 3]) -> [n, J]."""
    dc = dc[:, None, :]
    n = np.cross(d1, d2)
    nn = (n * n).sum(-1)
    a2, b2 = (d1 * d1).sum(-1), (d2 * d2).sum(-1)
    with np.errstate(invalid="ignore", divide="ignore"):
        skew = np.abs((dc * n).sum(-1)) / np.sqrt(nn)
        x = np.cross(np.broadcast_to(dc, d1.shape), d1)
        par = np.sqrt((x * x).sum(-1)) / np.sqrt(a2)
    return np.where(nn <= 1e-24 * a2 * b2, par, skew)


def cluster(cost, active, P, V, max_dist, K):
    """The clustering, ranking and outputs of one frame from its costs -> (members [K, V], labels [P, V], people)."""
    M = P * V
    view = np.arange(M) % V
    adm = cost <= max_dist
    a, b = np.nonzero(np.triu(adm, 1))
    lo = np.where(view[a] < view[b], a, b)
    hi = a + b - lo
    order = np.lexsort((lo * M + hi, cost[lo, hi]))
    cl = np.where(active, np.arange(M), -1)
    memb = {m: [m] for m in range(M) if active[m]}
    for e in order:
        ca, cb = cl[lo[e]], cl[hi[e]]
        if ca == cb or set(view[memb[ca]]) & set(view[memb[cb]]):
            continue
        if not adm[np.ix_(memb[ca], memb[cb])].all():
            continue
        memb[ca] = memb[ca] + memb[cb]
        for x in memb.pop(cb):
            cl[x] = ca
    persons = sorted((sorted(ms) for ms in memb.values() if len(ms) >= 2), key=lambda ms: (-len(ms), ms[0]))
    members = np.full((K, V), -1, dtype=np.int32)
    labels = np.where(active, -1, -2).astype(np.int32).reshape(P, V)
    for k, ms in enumerate(persons[:K]):
        for m in ms:
            members[k, m % V] = m // V
            labels[m // V, m % V] = k
    return members, labels, len(persons)


def near(cost, max_dist):
    """The frame's decisions could flip under last-bit differences of the costs (see the module docstring)."""
    c = cost[np.triu_indices(len(cost), 1)]
    c = c[np.isfinite(c)]
    if (np.abs(c - max_dist) <= NEAR_REL * max_dist).any():
        return True
    s = np.sort(c[c <= max_dist])
    return bool(len(s) > 1 and (np.diff(s) <= NEAR_REL * s[1:]).any())


def associate(scene, calib, min_conf=0.0, min_joints=3, max_dist=0.1, K=None):
    """scene [F, P, V, J, 3], calib [V, 18] or [F, V, 18] -> (members [F, K, V], labels [F, P, V], people [F], near [F])."""
    scene = np.asarray(scene)
    F, P, V = scene.shape[:3]
    K = P if K is None else K
    calib = np.asarray(calib, dtype=np.float64)
    members = np.empty((F, K, V), dtype=np.int32)
    labels = np.empty((F, P, V), dtype=np.int32)
    people = np.empty(F, dtype=np.int32)
    flags = np.empty(F, dtype=bool)
    for f in range(F):
        cost, active = pair_costs(scene[f], calib if calib.ndim == 2 else calib[f], min_conf, min_joints)
        members[f], labels[f], people[f] = cluster(cost, active, P, V, max_dist, K)
        flags[f] = near(cost, max_dist)
    return members, labels, people, flags


def score(members, labels, perm):
    """(owner [F, K], acc [8]) of mpl_association_score."""
    members, labels, perm = (np.asarray(a) for a in (members, labels, perm))
    F, K, V = members.shape
    P = labels.shape[1]
    owner = np.full((F, K), -1, dtype=np.int32)
    acc = np.zeros(8)
    acc[0] = F
    for f in range(F):
        cnt = np.zeros(P, dtype=np.int64)
        for s in range(P):
            for v in range(V):
                if labels[f, s, v] != -2:
                    cnt[perm[f, v, s]] += 1
        acc[1] += (cnt >= 2).sum()
        acc[7] += (cnt * (cnt - 1) // 2).sum()
        for k in range(K):
            true = [perm[f, v, members[f, k, v]] for v in range(V) if members[f, k, v] >= 0]
            n = len(true)
            if n == 0:
                continue
            counts = np.bincount(true, minlength=P)
            owner[f, k] = int(np.argmax(counts))                         # the first maximum: ties to the smaller index
            acc[2] += 1
            acc[5] += n * (n - 1) // 2
            acc[6] += (counts * (counts - 1) // 2).sum()
            if counts.max() == n:
                acc[3] += 1
                acc[4] += cnt[owner[f, k]] == n
    return owner, acc
