"""Oracle: lookups of 3-D points and rendered rays into a lattice map (pagnerf_b200.mapping.map_index / lookup_points /
lookup_rays) on the CPU.  TEST INFRASTRUCTURE ONLY.

Restates the definitions of pagnerf_b200/mapping/panoptic_map.py without a hash table: the packed lattice keys are sorted, and the
candidates of every window offset are found with np.searchsorted.  numpy evaluates each float64 / float32 operation separately
rounded, in the order written, so the distances, the window centre and the rays' surface points are the device's bit for bit.
"""
import itertools

import numpy as np

from .components import lattice_index, pack

MAX_RADIUS = 4


def index(xyz, k, level):
    """-> dict(keys: sorted packed lattice keys, points: the point of each key, D, errors=dict(off_lattice, duplicates))."""
    j, on = lattice_index(xyz, k, level)
    key = pack(j)
    idx = np.nonzero(on)[0]
    order = np.argsort(key[idx], kind="stable")
    sk, si = key[idx][order], idx[order]
    return dict(keys=sk, points=si, D=int(k) << int(level),
                errors=dict(off_lattice=int((~on).sum()), duplicates=int(idx.size - np.unique(sk).size)))


def query_position(x, D, radius):
    """xyz f32 [Q,3] -> (t f64 [Q,3], j0 i64 [Q,3], valid bool [Q]): t = ((x + 1) * D) * 0.5 - 0.5, j0 = floor(t + 0.5); valid iff
    every t is finite and in [-radius - 0.5, D - 0.5 + radius]."""
    x = np.asarray(x, dtype=np.float32).reshape(-1, 3).astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        t = ((x + 1.0) * float(D)) * 0.5 - 0.5
        valid = ((t >= -radius - 0.5) & (t <= (D - 0.5) + radius)).all(axis=1)
    t = np.where(valid[:, None], t, 0.0)
    return t, np.floor(t + 0.5).astype(np.int64), valid


def lookup_points(idx, xyz, radius, component=None):
    """-> (point i64 [Q], object i64 [Q] or None) by the definitions: nearest candidate by ((tx-jx)^2 + (ty-jy)^2) + (tz-jz)^2,
    then by point index."""
    D = idx["D"]
    sk, si = idx["keys"], idx["points"]
    t, j0, valid = query_position(xyz, D, radius)
    Q = t.shape[0]
    best_d = np.full(Q, np.inf)
    best_p = np.full(Q, -1, np.int64)
    for off in itertools.product(range(-radius, radius + 1), repeat=3) if sk.size else []:
        j = j0 + np.asarray(off, np.int64)
        ok = valid & ((j >= 0) & (j < D)).all(axis=1)
        key = pack(np.where(ok[:, None], j, 0))
        pos = np.minimum(np.searchsorted(sk, key), sk.size - 1)
        ok &= sk[pos] == key
        p = si[pos]
        dv = t - j.astype(np.float64)
        d2 = (dv[:, 0] * dv[:, 0] + dv[:, 1] * dv[:, 1]) + dv[:, 2] * dv[:, 2]
        better = ok & ((d2 < best_d) | ((d2 == best_d) & (p < best_p)))
        best_d = np.where(better, d2, best_d)
        best_p = np.where(better, p, best_p)
    obj = None
    if component is not None:
        component = np.asarray(component, np.int64)
        obj = np.where(best_p >= 0, component[np.maximum(best_p, 0)] if component.size else -1, -1)
    return best_p, obj


def surface_points(origins, dirs, depth, alpha, min_alpha):
    """-> (x f32 [N,3], valid bool [N]): s = depth / alpha, x = o + d * s in fp32 (separately rounded); valid iff
    alpha >= min_alpha (in fp32) and s is finite."""
    o = np.asarray(origins, np.float32).reshape(-1, 3)
    d = np.asarray(dirs, np.float32).reshape(-1, 3)
    a = np.asarray(alpha, np.float32).reshape(-1)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        s = np.asarray(depth, np.float32).reshape(-1) / a
        x = o + d * s[:, None]
    return x.astype(np.float32), (a >= np.float32(min_alpha)) & np.isfinite(s)


def lookup_rays(idx, origins, dirs, depth, alpha, radius, min_alpha, component=None):
    x, valid = surface_points(origins, dirs, depth, alpha, min_alpha)
    point, obj = lookup_points(idx, np.where(valid[:, None], x, np.float32(np.nan)), radius, component)
    return point, obj


def brute_force(xyz_map, k, level, queries, radius):
    """Every map point against every query: Chebyshev window around j0, then the smallest distance, then the smallest index."""
    j, on = lattice_index(xyz_map, k, level)
    assert on.all()
    D = int(k) << int(level)
    t, j0, valid = query_position(queries, D, radius)
    Q, P = t.shape[0], j.shape[0]
    out = np.full(Q, -1, np.int64)
    for q in range(Q):
        if not valid[q] or P == 0:
            continue
        cand = np.nonzero((np.abs(j - j0[q]) <= radius).all(axis=1))[0]
        if cand.size == 0:
            continue
        dv = t[q] - j[cand].astype(np.float64)
        d2 = (dv[:, 0] * dv[:, 0] + dv[:, 1] * dv[:, 1]) + dv[:, 2] * dv[:, 2]
        m = d2 == d2.min()
        out[q] = cand[m].min()
    return out
