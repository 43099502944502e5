"""Oracle: the panoptic point-map export (pagnerf_b200.mapping) on the CPU.  TEST INFRASTRUCTURE ONLY.

Restates the definitions of pagnerf_b200/mapping/panoptic_map.py step by step on oracle.field.FieldOracle:
  * sub-cell centres in fp32 numpy (exact-integer numerator and denominator, IEEE division: the bit-exact definition);
  * the field in float64: the encoders evaluated in float32 (their bit-exact definition, oracle/permuto.py, oracle/hashgrid.py),
    then every decoder, the view embedding, softmax and temperature in float64;
  * the density threshold on the float64 density;
  * labels = argmax of the float64 logits (lowest class on ties), scores = that class's value of the float64 output channel;
  * the per-instance summary as a per-point dictionary loop.
"""
import copy

import numpy as np
import torch
import torch.nn.functional as F

PRUNE_MIN_DENSITY = (0.01 * 512) / np.sqrt(3)


def cell_points(cells, level, k):
    """cells int [C,3] of `level` -> f32 [C*k^3, 3]; sub-point s = (ix*k + iy)*k + iz."""
    cells = np.asarray(cells, dtype=np.int64).reshape(-1, 3)
    sub = np.stack(np.meshgrid(np.arange(k), np.arange(k), np.arange(k), indexing="ij"), -1).reshape(-1, 3)
    num = 2 * (cells[:, None, :] * k + sub[None, :, :]) + 1
    xyz = num.astype(np.float32) / np.float32(k << level)
    return (xyz.astype(np.float32) - np.float32(1.0)).astype(np.float32).reshape(-1, 3)


def _dbl(module):
    return copy.deepcopy(module).double()


def evaluate(field, xyz, view_dir=(0.0, 0.0, -1.0)):
    """FieldOracle on points xyz f32 [P,3] seen along view_dir -> dict of float64 torch tensors: density [P], rgb [P,3],
    sem_logits / inst_logits [P,C] (instance logits already divided by the temperature) and the channels sem / inst [P,C] the
    nef returns."""
    with torch.no_grad():
        x32 = torch.from_numpy(np.ascontiguousarray(xyz, dtype=np.float32))
        lodw = field.lod_weights.double()
        feats = field.grid(x32).double() * lodw
        dfe = field.delta_grid(x32).double() * lodw if field.delta_grid is not None else None
        density_feats = _dbl(field.decoder_density)(feats)
        density = torch.relu(density_feats[:, 0])
        vd = torch.as_tensor(view_dir, dtype=torch.float32).double()
        vd = vd / vd.norm()
        ve = _dbl(field.view_embedder)(-vd[None]).expand(feats.shape[0], -1)
        rgb = torch.sigmoid(_dbl(field.decoder_color)(torch.cat([density_feats, ve], -1)))
        panop = feats + dfe if dfe is not None else feats
        s = _dbl(field.decoder_semantics)(panop)
        e = _dbl(field.decoder_inst)(panop)
        if field.inst_soft_temperature > 0.0:
            e = e / field.inst_soft_temperature
        return dict(density=density, rgb=rgb, sem_logits=s, inst_logits=e,
                    sem=F.softmax(s, -1) if field.sem_softmax else s, inst=F.softmax(e, -1) if field.inst_softmax else e)


def labels(logits, channel):
    """-> (label i64 [P], score f64 [P], relative gap between the two largest logits [P]) -- argmax takes the lowest index on ties."""
    z = logits.numpy()
    lab = np.argmax(z, axis=1)
    score = np.take_along_axis(channel.numpy(), lab[:, None], 1)[:, 0]
    if z.shape[1] > 1:
        top2 = -np.sort(-z, axis=1)[:, :2]
        gap = (top2[:, 0] - top2[:, 1]) / np.maximum(np.abs(top2[:, 0]), 1e-30)
    else:
        gap = np.full(z.shape[0], np.inf)
    return lab.astype(np.int64), score, gap


def extract(field, cells, level, k, min_density=None, view_dir=(0.0, 0.0, -1.0)):
    """The map of `field` on the leaf cells `cells` (in the octree's order) -> dict of numpy arrays: every point's xyz / density
    ('all_xyz', 'all_density') and the kept points' xyz, rgb, density, semantic, semantic_score, semantic_gap, instance,
    instance_score, instance_gap."""
    thr = PRUNE_MIN_DENSITY if min_density is None else float(min_density)
    xyz = cell_points(cells, level, k)
    out = evaluate(field, xyz, view_dir)
    dens = out["density"].numpy()
    keep = dens > thr
    kt = torch.from_numpy(keep)
    sl, ss, sg = labels(out["sem_logits"][kt], out["sem"][kt])
    il, is_, ig = labels(out["inst_logits"][kt], out["inst"][kt])
    return dict(all_xyz=xyz, all_density=dens, xyz=xyz[keep], rgb=out["rgb"].numpy()[keep], density=dens[keep], semantic=sl,
                semantic_score=ss, semantic_gap=sg, instance=il, instance_score=is_, instance_gap=ig)


def summary(xyz, rgb, semantic, instance, num_instances, num_classes, things=None):
    """Per-instance summary by a per-point dictionary loop -> dict of numpy arrays (count, sum_xyz, centroid, bbox_min, bbox_max,
    sum_rgb, mean_rgb, votes, category) plus 'errors', the number of points with an out-of-range label (skipped)."""
    Ci, Cs = int(num_instances), int(num_classes)
    things = set(range(Cs)) if things is None else set(things)
    acc = {}
    errors = 0
    for p, c, s, q in zip(np.asarray(xyz, np.float32).tolist(), np.asarray(rgb, np.float32).tolist(),
                          np.asarray(semantic).tolist(), np.asarray(instance).tolist()):
        if not (0 <= s < Cs and 0 <= q < Ci):
            errors += 1
            continue
        if s not in things:
            continue
        a = acc.setdefault(q, dict(n=0, sx=[0.0] * 3, sr=[0.0] * 3, lo=[np.inf] * 3, hi=[-np.inf] * 3, votes={}))
        a["n"] += 1
        for i in range(3):
            a["sx"][i] += p[i]
            a["sr"][i] += c[i]
            a["lo"][i] = min(a["lo"][i], p[i])
            a["hi"][i] = max(a["hi"][i], p[i])
        a["votes"][s] = a["votes"].get(s, 0) + 1
    count = np.zeros(Ci, np.int64)
    sum_xyz, sum_rgb = np.zeros((Ci, 3)), np.zeros((Ci, 3))
    bmin, bmax = np.full((Ci, 3), np.inf, np.float32), np.full((Ci, 3), -np.inf, np.float32)
    votes = np.zeros((Ci, Cs), np.int64)
    category = np.full(Ci, -1, np.int64)
    for q, a in acc.items():
        count[q] = a["n"]
        sum_xyz[q], sum_rgb[q] = a["sx"], a["sr"]
        bmin[q], bmax[q] = a["lo"], a["hi"]
        for s, v in a["votes"].items():
            votes[q, s] = v
        best = max(a["votes"].values())
        category[q] = min(s for s, v in a["votes"].items() if v == best)
    with np.errstate(invalid="ignore", divide="ignore"):
        centroid, mean_rgb = sum_xyz / count[:, None], sum_rgb / count[:, None]
    return dict(count=count, sum_xyz=sum_xyz, centroid=centroid, bbox_min=bmin, bbox_max=bmax, sum_rgb=sum_rgb, mean_rgb=mean_rgb,
                votes=votes, category=category, errors=errors)
