"""Oracle: size and orientation of map objects (pagnerf_b200.mapping.object_shape) on the CPU.  TEST INFRASTRUCTURE ONLY.

Restates the definitions of pagnerf_b200/mapping/panoptic_map.py with other means than the device's:
  * moments as Python integers: per-object int64 sums of 18-bit limbs (exact while the total weight stays below 2^33), combined
    without rounding;
  * covariance from float(num), Python's correctly rounded (nearest, ties to even) int -> float conversion, then the pinned order
    of float64 divisions;
  * axes by numpy.linalg.eigh with the pinned order and sign rules (a covariance with zero off-diagonal entries gives the world
    axes directly, as the Jacobi solver skips zero entries);
  * the box from GIVEN axes by the pinned float64 arithmetic (separate numpy operations, no FMA), minimum and maximum in the IEEE
    total order.
"""
import numpy as np

from .components import lattice_index

PAIRS = ((0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2))
LIMB = 18


def moments(j, component, K, weight=None):
    """-> (n, S, SS) of Python ints: n[o], S[o][a] = sum j_a, SS[o][p] = sum j_a j_b over PAIRS[p], over the points of object o in
    [0, K) (other components are skipped), each point counted weight[i] times (once without weight)."""
    j = np.asarray(j, np.int64).reshape(-1, 3)
    comp = np.asarray(component, np.int64).reshape(-1)
    w = np.ones(len(comp), np.int64) if weight is None else np.asarray(weight, np.int64).reshape(-1)
    sel = (comp >= 0) & (comp < K)
    j, comp, w = j[sel], comp[sel], w[sel]
    mask = (1 << LIMB) - 1

    def sums(v):
        out = np.zeros(K, np.int64)
        np.add.at(out, comp, w * v)
        return out

    n = [int(x) for x in sums(np.ones(len(comp), np.int64))]
    S = np.stack([sums(j[:, a]) for a in range(3)], 1)
    SS = []
    for a, b in PAIRS:
        p = j[:, a] * j[:, b]
        lo, hi = sums(p & mask), sums(p >> LIMB)
        SS.append([int(x) + (int(y) << LIMB) for x, y in zip(lo, hi)])
    return n, [[int(x) for x in row] for row in S], [[SS[p][o] for p in range(6)] for o in range(K)]


def covariance(n, S, SS, D):
    """-> f64 [K, 3, 3]: (((num / n) / n) * 4 / D) / D with num = n S_ab - S_a S_b exact and float(num) correctly rounded; NaN for
    objects without points"""
    K = len(n)
    cov = np.full((K, 3, 3), np.nan)
    for o in range(K):
        if n[o] == 0:
            continue
        for p, (a, b) in enumerate(PAIRS):
            num = n[o] * SS[o][p] - S[o][a] * S[o][b]
            cov[o, a, b] = cov[o, b, a] = float(num) / n[o] / n[o] * 4 / D / D
    return cov


def orient(e):
    """e signed so that its component of largest magnitude (the lowest index on ties) is positive, then unit length"""
    m = int(np.argmax(np.abs(e)))
    e = e if e[m] >= 0 else -e
    return e / np.sqrt((e[0] * e[0] + e[1] * e[1]) + e[2] * e[2])


def principal_axes(cov):
    """-> (variance f64 [K, 3] descending, axes f64 [K, 3, 3] rows) by the pinned rules; NaN rows for NaN covariances"""
    K = len(cov)
    var, axes = np.full((K, 3), np.nan), np.full((K, 3, 3), np.nan)
    for o in range(K):
        c = cov[o]
        if np.isnan(c).any():
            continue
        if c[0, 1] == 0 and c[0, 2] == 0 and c[1, 2] == 0:
            w, V = np.diag(c).copy(), np.eye(3)
        else:
            w, V = np.linalg.eigh(c)
        order = sorted(range(3), key=lambda i: -w[i])         # stable: ties keep the column order
        e0, e1 = orient(V[:, order[0]]), orient(V[:, order[1]])
        var[o] = w[order]
        axes[o] = np.stack([e0, e1, np.cross(e0, e1)])
    return var, axes


def total_key(v):
    """f64 -> u64 whose unsigned order is the IEEE total order (-0 < +0)"""
    b = np.asarray(v, np.float64).view(np.uint64)
    return np.where(b >> np.uint64(63), ~b, b | np.uint64(1 << 63))


def from_key(k):
    k = np.asarray(k, np.uint64)
    return np.where(k >> np.uint64(63), k & np.uint64((1 << 63) - 1), ~k).view(np.float64)


def box(j, component, K, axes, D):
    """The oriented box of each object along GIVEN axes f64 [K, 3, 3] (rows) -> (lo, hi, center, extent), f64 [K, 3] each, NaN for
    objects without points"""
    j = np.asarray(j, np.int64).reshape(-1, 3).astype(np.float64)
    comp = np.asarray(component, np.int64).reshape(-1)
    sel = (comp >= 0) & (comp < K)
    j, comp = j[sel], comp[sel]
    e = np.asarray(axes, np.float64)[comp]                    # [P', 3 axes, 3 coordinates]
    lo, hi = np.full((K, 3), np.nan), np.full((K, 3), np.nan)
    has = np.zeros(K, bool)
    has[comp] = True
    for a in range(3):
        p = (j[:, 0] * e[:, a, 0] + j[:, 1] * e[:, a, 1]) + j[:, 2] * e[:, a, 2]
        key = total_key(p)
        kl = np.full(K, np.iinfo(np.uint64).max, np.uint64)
        kh = np.zeros(K, np.uint64)
        np.minimum.at(kl, comp, key)
        np.maximum.at(kh, comp, key)
        lo[has, a], hi[has, a] = from_key(kl[has]), from_key(kh[has])
    extent = ((hi - lo) + 1.0) * 2.0 / D
    mid = (lo + hi) / 2.0
    ax = np.asarray(axes, np.float64)
    c = (mid[:, 0:1] * ax[:, 0] + mid[:, 1:2] * ax[:, 1]) + mid[:, 2:3] * ax[:, 2]
    center = (2.0 * c + 1.0) / D - 1.0
    return lo, hi, center, extent


def shape(xyz, k, level, component, K):
    """-> dict: covariance, variance, axes, center, extent, lo, hi (the device's definitions, the box along the oracle's own axes)
    and errors = dict(off_lattice, bad_components), the counts that make the device call raise"""
    D = int(k) << int(level)
    j, on = lattice_index(xyz, k, level)
    comp = np.asarray(component, np.int64).reshape(-1)
    bad = (comp < -1) | (comp >= K)
    use = np.where(on & ~bad, comp, -1)
    n, S, SS = moments(j, use, K)
    cov = covariance(n, S, SS, D)
    var, axes = principal_axes(cov)
    lo, hi, center, extent = box(j, use, K, axes, D)
    return dict(covariance=cov, variance=var, axes=axes, center=center, extent=extent, lo=lo, hi=hi, n=np.array(n, np.int64),
                errors=dict(off_lattice=int((~on).sum()), bad_components=int(bad.sum())))
