"""Oracle: the objects of a labelled lattice map (pagnerf_b200.mapping.instance_components) on the CPU.  TEST INFRASTRUCTURE ONLY.

Restates the definitions of pagnerf_b200/mapping/panoptic_map.py with an independent algorithm -- no union-find, no hashing:
  * lattice recovery per axis by rounding (x + 1) D / 2 - 1/2, then the exact fp32 formula of oracle.mapping.cell_points decides;
  * neighbour pairs by sorting the packed lattice keys and np.searchsorted, every offset in both directions;
  * the closure by scipy.sparse.csgraph.connected_components;
  * numbering by each object's smallest point index;
  * statistics by oracle.mapping.summary on the object labels.
"""
import itertools

import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

from .mapping import summary

AXIS_BITS = 21


def lattice_index(xyz, k, level):
    """xyz f32 [P,3] -> (j i64 [P,3], on bool [P]): on[i] iff every coordinate of point i is, bit for bit, fl(fl((2j+1)/D) - 1)
    for some j in [0, D), D = k << level; j is that index (0 on axes where it is not)."""
    x = np.asarray(xyz, dtype=np.float32).reshape(-1, 3)
    D = int(k) << int(level)
    with np.errstate(invalid="ignore"):
        t = (x.astype(np.float64) + 1.0) * D * 0.5 - 0.5
        ok = (t > -0.5) & (t < D - 0.5)
    j = np.rint(np.where(ok, t, 0.0)).astype(np.int64)
    y = (2 * j + 1).astype(np.float32) / np.float32(D) - np.float32(1.0)
    ok &= y.astype(np.float32).view(np.uint32) == x.view(np.uint32)
    return np.where(ok, j, 0), ok.all(axis=1)


def pack(j):
    j = np.asarray(j, dtype=np.int64)
    return (j[:, 0] << (2 * AXIS_BITS)) | (j[:, 1] << AXIS_BITS) | j[:, 2]


def offsets(connectivity):
    """The neighbour offsets of a lattice point, both directions."""
    if connectivity == 6:
        return [d for d in itertools.product((-1, 0, 1), repeat=3) if sum(map(abs, d)) == 1]
    if connectivity == 26:
        return [d for d in itertools.product((-1, 0, 1), repeat=3) if d != (0, 0, 0)]
    raise ValueError(f"connectivity must be 6 or 26, got {connectivity}")


def components(xyz, semantic, instance, k, level, things, connectivity, min_points, rgb, num_instances, num_classes):
    """-> dict of numpy arrays: component [P], and per object count, instance, category, centroid, mean_rgb, bbox_min, bbox_max,
    votes, sum_xyz, sum_rgb; plus 'errors' = dict(off_lattice, duplicates, bad_labels), the counts that make the device call raise
    (the labelling is meaningless when one is non-zero)."""
    xyz = np.asarray(xyz, dtype=np.float32).reshape(-1, 3)
    P = xyz.shape[0]
    sem, inst = np.asarray(semantic, dtype=np.int64).reshape(P), np.asarray(instance, dtype=np.int64).reshape(P)
    Ci, Cs = int(num_instances), int(num_classes)
    D = int(k) << int(level)
    j, on = lattice_index(xyz, k, level)
    key = pack(j)
    bad = (sem < 0) | (sem >= Cs) | (inst < 0) | (inst >= Ci)
    errors = dict(off_lattice=int((~on).sum()), duplicates=int(on.sum() - np.unique(key[on]).size), bad_labels=int(bad.sum()))
    tm = np.zeros(Cs, bool)
    tm[list(things) if things is not None else slice(None)] = True
    active = on & ~bad & tm[np.clip(sem, 0, Cs - 1)]
    idx = np.nonzero(active)[0]
    order = np.argsort(key[idx], kind="stable")
    sk, si = key[idx][order], idx[order]
    rows, cols = [idx], [idx]          # self loops: every active point is in the graph
    for d in offsets(connectivity) if len(sk) else []:
        nj = j[idx] + np.asarray(d, dtype=np.int64)
        inside = ((nj >= 0) & (nj < D)).all(axis=1)
        nk = pack(np.where(inside[:, None], nj, 0))
        pos = np.minimum(np.searchsorted(sk, nk), len(sk) - 1)
        nb = si[pos]
        same = inside & (sk[pos] == nk) & (inst[nb] == inst[idx])
        rows.append(idx[same])
        cols.append(nb[same])
    r, c = np.concatenate(rows), np.concatenate(cols)
    _, lab = connected_components(coo_matrix((np.ones(r.size, np.int32), (r, c)), shape=(P, P)), directed=False)
    lab_a = lab[idx]
    n_lab = int(lab.max()) + 1 if P else 0
    size = np.bincount(lab_a, minlength=n_lab)
    first = np.full(n_lab, P, np.int64)
    np.minimum.at(first, lab_a, idx)
    kept = np.nonzero(size >= min_points)[0]
    kept = kept[np.argsort(first[kept], kind="stable")]
    new_id = np.full(n_lab, -1, np.int64)
    new_id[kept] = np.arange(kept.size)
    component = np.full(P, -1, np.int64)
    component[idx] = new_id[lab_a]
    K = int(kept.size)
    sel = component >= 0
    rgb = np.asarray(rgb, dtype=np.float32).reshape(-1, 3)
    out = summary(xyz[sel], rgb[sel], sem[sel], component[sel], K, Cs)
    obj_inst = np.full(K, -1, np.int64)
    obj_inst[component[sel]] = inst[sel]
    out.pop("errors")
    out.update(component=component, instance=obj_inst, errors=errors)
    return out
