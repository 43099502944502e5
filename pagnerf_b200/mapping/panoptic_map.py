"""Labelled 3-D panoptic point map of a trained field, on the device: what the reference's utils/render_map.py exports by calling the
nef on the octree, without the [P, C] probability tensors, the per-thread decoder kernels or the host-side argmax.

    pts = extract_panoptic_map(nef, samples_per_axis=2)        # PanopticPoints of CUDA tensors, P kept points
    summ = instance_summary(pts, num_instances=nef.num_instances, num_classes=nef.num_classes, things={0})
    write_ply("map.ply", pts)

Definitions (the CPU oracle, oracle/mapping.py, and the tests follow them exactly):
  * Points.  Every occupied leaf cell of nef.grid.blas at nef.grid.blas_level (spc.unbatched_get_level_points, Morton order) gets
    k^3 sub-cell centres, k = samples_per_axis in [1, 8].  Sub-point s = (ix*k + iy)*k + iz (the axis order of
    pag_octree_level_bits); per axis, in fp32 with IEEE division, x = (float)(2*(p*k + i) + 1) / (float)(k << L) - 1.0f for the
    cell's integer coordinate p at level L.  Numerator and denominator are exact integers, there is no jitter: the map is
    deterministic.  Output order is cell order, then sub-point order, filtered by the density test; it does not depend on
    chunk_points.
  * Density and colour come from the colour branch: the density head after its ReLU, and the colour seen along the single
    direction view_dir (normalised here).  The default (0, 0, -1) is the look direction of the synthetic robot pass of bench.py
    and the tests; with real data pass the mean viewing direction.  All LODs are used (lod_idx = num_lods - 1), exact fp32, no
    autocast, like validation.  PanopticDDensityNeF's panoptic density is not used: the map's geometry is the colour density for
    every field.
  * A point is kept iff density > min_density.  The default is prune()'s cell threshold 0.01 * 512 / sqrt(3): "in the map" means
    what "kept by prune" means.
  * Labels are the argmax over the channel the nef's forward returns (logits times 1/T when inst_soft_temperature T > 0), taken on
    the logits, lowest class index on ties.  The score is the winning class's value of that channel: 1 / sum_c exp((z_c - z_max) * s)
    with a softmax head, z_max * s without one.
  * The heads read _panoptic_inputs(feats, coords, lod_idx, rows), the (a + b) * lod_weights the fused render uses; the delta grid
    is looked up for the kept rows only.
  * Supported fields: those whose heads the fused kernels serve (PanopticNeF._fused_heads_unsupported): plain heads, detached,
    'cat', feature width <= 48 and a multiple of 4, <= 16 classes, <= 208 instances.  Anything else raises NotImplementedError
    with the reason; a field on the CPU raises RuntimeError (no CPU fallback).
  * Host reads: one per chunk, the kept count (the size of that chunk's output, torch.nonzero).

instance_summary counts a point toward instance `inst` only when its semantic class is in `things` (every class when None), and
returns centroid = sum_xyz / count in float64 (NaN where count == 0; bbox_min / bbox_max stay +inf / -inf there).

instance_components splits the map into objects:

    comps = instance_components(pts, samples_per_axis=2, level=nef.grid.blas_level, num_instances=nef.num_instances,
                                num_classes=nef.num_classes, things={0}, connectivity=26, min_points=20)
    comps.count.numel()             # number of objects; comps.component[i] = object of point i or -1

  * Lattice.  D = k << level.  A point has lattice index j in [0, D)^3 iff each coordinate equals, bit for bit,
    fl(fl((2j+1)/D) - 1) (the point formula above), so every map of extract_panoptic_map(nef, k) is on the lattice of
    (k, nef.grid.blas_level).  Points off the lattice, and points whose lattice index another point has, raise ValueError with
    their number.  xyz must be float32.
  * Active points: semantic class in `things` (every class when None).  Labels outside [0, num_classes) / [0, num_instances) raise
    ValueError with their number, as in instance_summary.
  * Adjacency: two active points are adjacent iff their lattice indices differ by a vector of {-1,0,1}^3 \\ {0} (connectivity=26)
    or by one unit step along one axis (connectivity=6), and their instance labels are equal.  Objects are the transitive closure.
  * Numbering: objects of fewer than min_points points are dropped; their points and inactive points get component -1.  The others
    are numbered 0..K-1 in the order of their smallest point index.  The result does not depend on thread scheduling, and the
    partition does not depend on point order.
  * Statistics per object: count, centroid = float64 sum / count, bbox_min / bbox_max in float32, mean_rgb (float64), votes
    [K, num_classes], category = argmax of votes (lowest class on ties) and instance, the label the object's points share.
  * Host reads: one per call (the error counts and K).  Device memory: at most 12 C + 24 P + 12 ceil(P / 1024) + 8 bytes for the
    labelling (C = the smallest power of two >= 2P: a hash table of 12-byte slots, 16 bytes of workspace per point and the i64
    component, so at most 72 bytes per point) plus (160 + 8 num_classes) bytes per object; 11.2 M points take 0.65 GB.

map_index, lookup_points and lookup_rays answer which map point, and so which object, a 3-D point or a rendered pixel lies on:

    index = map_index(pts, samples_per_axis=2, level=nef.grid.blas_level)               # MapIndex; one host read (error counts)
    hit = lookup_points(index, xyz, radius=1, component=comps.component)                # MapLookup(point i64[Q], object i64[Q])
    hit = lookup_rays(index, rays.origins, rays.dirs, rb.depth, rb.alpha, radius=1, min_alpha=0.5, component=comps.component)

  * Index.  The lattice rules of instance_components (D = k << level; every point on the lattice bit for bit, no two points with one
    lattice index, else ValueError with the same messages; xyz float32, P <= 2^30).  Labels are not read: every map point is
    indexed, stuff and floater points included, so a leaf in front of a fruit resolves to the leaf, not to the fruit behind it.
  * Query position.  Per axis, in float64 with explicitly rounded operations (no FMA contraction): t = ((x + 1) * D) * 0.5 - 0.5,
    window centre j0 = floor(t + 0.5).
  * Candidates.  Map points whose lattice index j lies in [0, D)^3 and differs from j0 by at most `radius` (an integer in [0, 4])
    per axis.
  * Choice.  The candidate with the smallest ((tx-jx)^2 + (ty-jy)^2) + (tz-jz)^2 (float64, in this order, no FMA), then the
    smallest point index; point = -1 with no candidate, for a non-finite coordinate, and for t outside
    [-radius - 0.5, D - 0.5 + radius] in any axis.
  * Object.  object = component[point] where point >= 0, else -1 (so floaters and inactive points give -1 with a valid point);
    component must have shape [P] of the indexed map.  Without component, MapLookup.object is None.
  * Rays.  The surface point of a rendered ray, in fp32 with IEEE rounding: s = depth / alpha, then x = o + d * s per axis as a
    separately rounded mul and add (the marcher's sample-position convention).  Rays with alpha < min_alpha (min_alpha in (0, 1],
    compared in fp32) or a non-finite s give -1; a ray with alpha == min_alpha is looked up.  depth and alpha may be [N] or [N, 1],
    as the tracer returns them.
  * Host traffic.  Lookups make no host read and no host synchronisation; their launch geometry depends on Q and radius only, so
    they can be captured in a CUDA graph.  The result depends only on the inputs: the same for any query order and on every run.
  * Memory.  The index is the table alone: 12 C bytes (u64 key + u32 point per slot, C = the smallest power of two >= 2P), plus
    the 4-entry info tensor; 2^25 slots, about 0.4 GB, for the 11.2 M points of a k = 4 map.  A lookup allocates only its outputs
    (16 bytes per query with component, 8 without) when its inputs are contiguous.

project_map answers, from the map alone, which map point, at what depth and which object each pixel of a camera sees:

    mv = project_map(pts, samples_per_axis=2, level=nef.grid.blas_level, view=V, intrinsics=K, height=H, width=W,
                     component=comps.component)                                         # MapView(point, depth, object), [B, H, W]

  * Cameras.  view f32 [B, 4, 4] world-to-camera matrices (BAPipeline's and bench.make_cameras' layout; rows 0..2 are read),
    intrinsics f32 [B, 4] = (fx, fy, cx, cy) in pixels, both CUDA tensors.  The camera looks down its -z axis; the pixel in column c
    and row r has the camera-space ray direction ((c + 0.5 - cx) / fx, (r + 0.5 - cy) / fy, -1), rows growing with +y (the
    convention of bench.make_frame_rays).
  * Arithmetic.  fp32, every operation separately rounded (no FMA contraction), in the order written.
  * Transform.  Per row q of view: p_q = ((V[q,0] x + V[q,1] y) + V[q,2] z) + V[q,3]; the point's depth is z = -p_2.
  * Pixel position.  u = fx (p_0 / z) + cx, v = fy (p_1 / z) + cy (the division, then the product, then the sum).
  * Footprint.  A map point stands for its lattice cell, of half-size h = fl(1 / D), D = samples_per_axis << level (exact when
    samples_per_axis is a power of two).  Half-sizes in pixels su = min((fx h) / z, max_radius), sv = min((fy h) / z, max_radius),
    NaN propagating.  The point covers every pixel the closed square [u - su, u + su] x [v - sv, v + sv] touches: columns
    floor(u - su) .. floor(u + su), rows floor(v - sv) .. floor(v + sv), clipped to the image.  With max_radius = 0 a point covers
    exactly the pixel containing (u, v).  max_radius is an integer in [0, 32]; a point tests at most (2 max_radius + 2)^2 pixels
    (2 max_radius + 1 per axis but for the rounding of u +- su).
  * Dropped points.  A point is projected only if z > near, u and v are finite and su >= 0 and sv >= 0 (false for NaN; a negative
    focal length gives an empty square).  Floors are clamped to the image in float before the conversion to an integer, so a point
    far off-screen cannot overflow it.  Camera values are not validated (that would be a host read); they are used as defined here.
  * Visibility.  Each pixel gets the covering point with the smallest z, then the smallest point index, whatever the thread schedule.
  * Outputs.  point i64 [B, H, W] (-1 where no point covers the pixel), depth f32 [B, H, W] (its z, +inf where point == -1) and, with
    component (i64 [P], e.g. InstanceComponents.component), object = component[point], -1 where point == -1.
  * Lattice.  (samples_per_axis, level) only set the footprint; the points need not lie on the lattice and are not checked.
  * Limits.  P <= 2^30, B <= 65535, height and width integers in [1, 16384], near a finite number > 0 (also in fp32).
  * Host traffic.  None: the launch geometry depends on P, B, H, W and max_radius only, so the call can be captured in a CUDA graph.
  * Memory.  The outputs and a u64 depth buffer of B H W entries: 28 bytes per pixel with component, 20 without.

object_visibility answers, per map object and camera view, how much of the object the view sees, how much of it is hidden and where:

    vis = object_visibility(pts, samples_per_axis=2, level=nef.grid.blas_level, view=V, intrinsics=K, height=H, width=W,
                            component=comps.component, num_objects=comps.count.numel())   # ObjectVisibility, [B, K] tensors
    best = vis.visible.argmax(0)                          # the view that shows each object best; vis.bbox[best[o], o] crops it
    occluded = 1 - vis.visible / vis.silhouette           # NaN where the view covers none of the object

  * Arguments.  pts, samples_per_axis, level, view, intrinsics, height, width, max_radius and near mean exactly what they mean
    for project_map, with its checks and limits.  component i64 [P]: each point's object in [0, num_objects) or -1; components
    outside [-1, num_objects) raise ValueError with their number.  num_objects = K, an integer >= 0.
  * Coverage.  Pixel (b, r, c) is covered by point i iff project_map's footprint rule covers it: the same fp32 arithmetic, the same
    dropped points (near plane, non-finite, negative half-size, off-screen) and clamping before the integer conversion.
  * visible[b, o]: the pixels of view b whose project_map point (smallest depth, then smallest index) has component o.
  * silhouette[b, o]: the pixels of view b covered by at least one point with component o, at any depth; visible[b, o] of a
    projection of object o's points alone.
  * bbox[b, o] = (col_min, row_min, col_max, row_max) of the visible pixels, (-1, -1, -1, -1) where visible[b, o] == 0.
  * Points with component -1 (stuff, floaters, inactive points) occlude but own no row.  So visible <= silhouette, and visible[b]
    sums to the pixels of view b with MapView.object >= 0.  The occluded fraction and the best view are left to the caller.
  * Host traffic.  One host read per call (the silhouette bitmaps' size and the error count); the call cannot be captured in a
    CUDA graph.  The result depends only on the inputs: the same for any split of the cameras into calls and on every run.
  * Memory.  The u64 depth buffer (8 B H W bytes, freed before the silhouettes), 32 bytes of outputs and 28 of workspace per
    (view, object) pair plus 16 bytes, and the silhouette bitmaps: one bit per pixel of each pair's footprint box, rows padded to
    32-bit words, at most VISIBILITY_BITMAP_BYTES (256 MiB).  When the bitmaps exceed it the silhouettes are built in rounds,
    each a pass over the points and cameras.
"""
import math
from typing import NamedTuple, Optional

import numpy as np
import torch

from .. import ops, spc
from ..pc_nerf import PanopticNeF
from ..pc_nerf.panoptic_nef import _decoder_tensors

MAX_SAMPLES_PER_AXIS = 8
PRUNE_MIN_DENSITY = (0.01 * 512) / math.sqrt(3)      # PanopticNeF.prune()'s cell threshold
MAX_SUMMARY_CLASSES = 32                             # thing mask: one bit per class
MAX_LEVEL = 15                                       # pag_map_cell_points' octree levels
MAX_COMPONENT_POINTS = 1 << 30                       # i32 union-find parents, u32 table values
MAX_LOOKUP_RADIUS = 4                                # a (2r+1)^3 window: 729 probes per query at most
MAX_PROJECT_RADIUS = 32                              # a footprint of at most 66 x 66 pixels
MAX_PROJECT_SIDE = 16384
MAX_PROJECT_CAMERAS = 65535                          # one grid row per camera
VISIBILITY_BITMAP_BYTES = 256 << 20                  # silhouette bitmaps of one round; >= 32 MiB, one 16384 x 16384 view's


class PanopticPoints(NamedTuple):
    xyz: torch.Tensor              # f32 [P, 3]
    rgb: torch.Tensor              # f32 [P, 3]
    density: torch.Tensor          # f32 [P]
    semantic: torch.Tensor         # i64 [P]
    semantic_score: torch.Tensor   # f32 [P]
    instance: torch.Tensor         # i64 [P]
    instance_score: torch.Tensor   # f32 [P]


class InstanceComponents(NamedTuple):
    component: torch.Tensor        # i64 [P]: object of each point, -1 if the point is in no object
    count: torch.Tensor            # i64 [K]
    instance: torch.Tensor         # i64 [K]: the instance label all points of the object share
    category: torch.Tensor         # i64 [K]: argmax of votes (lowest class on ties)
    centroid: torch.Tensor         # f64 [K, 3]
    mean_rgb: torch.Tensor         # f64 [K, 3]
    bbox_min: torch.Tensor         # f32 [K, 3]
    bbox_max: torch.Tensor         # f32 [K, 3]
    votes: torch.Tensor            # i64 [K, Cs]


class MapIndex(NamedTuple):
    keys: torch.Tensor             # i64 [C]: packed lattice index + 1 per slot, 0 = empty (C = the smallest power of two >= 2P)
    points: torch.Tensor           # i32 [C]: the map point of each filled slot
    k: int                         # samples_per_axis of the map's lattice
    level: int
    P: int                         # points of the indexed map


class MapLookup(NamedTuple):
    point: torch.Tensor                    # i64 [Q]: the nearest map point in the window, -1 if none
    object: Optional[torch.Tensor]         # i64 [Q]: component[point], -1 where there is no point or it is in no object


class MapView(NamedTuple):
    point: torch.Tensor                    # i64 [B, H, W]: the visible map point of each pixel, -1 if none
    depth: torch.Tensor                    # f32 [B, H, W]: its camera-space depth z (> near), +inf where point == -1
    object: Optional[torch.Tensor]         # i64 [B, H, W]: component[point], -1 where point == -1 or the point is in no object


class ObjectVisibility(NamedTuple):
    visible: torch.Tensor                  # i64 [B, K]: pixels of view b whose front map point belongs to object o
    silhouette: torch.Tensor               # i64 [B, K]: pixels of view b covered by object o's points at any depth
    bbox: torch.Tensor                     # i32 [B, K, 4]: (col_min, row_min, col_max, row_max) of the visible pixels, -1s if none


class InstanceSummary(NamedTuple):
    count: torch.Tensor            # i64 [Ci]
    centroid: torch.Tensor         # f64 [Ci, 3]
    bbox_min: torch.Tensor         # f32 [Ci, 3]
    bbox_max: torch.Tensor         # f32 [Ci, 3]
    mean_rgb: torch.Tensor         # f64 [Ci, 3]
    votes: torch.Tensor            # i64 [Ci, Cs]
    category: torch.Tensor         # i64 [Ci]: argmax of votes (lowest class on ties), -1 where count == 0


def _empty_points(device):
    f = lambda *s: torch.empty(*s, dtype=torch.float32, device=device)
    i = lambda *s: torch.empty(*s, dtype=torch.int64, device=device)
    return PanopticPoints(f(0, 3), f(0, 3), f(0), i(0), f(0), i(0), f(0))


def _check_field(nef):
    if not isinstance(nef, PanopticNeF):
        raise NotImplementedError(f"map export serves PanopticNeF and its subclasses, not {type(nef).__name__}")
    if nef.position_input:
        raise NotImplementedError("map export: position_input fields are not served by the fused decoders")
    reason = nef._fused_heads_unsupported()
    if reason is not None:
        raise NotImplementedError(f"map export: the label kernel does not serve {reason}")
    if not nef.decoder_density.lout.weight.is_cuda:
        raise RuntimeError("pagnerf_b200 map export runs on CUDA fields only (no CPU fallback)")


def extract_panoptic_map(nef, samples_per_axis=2, min_density=None, view_dir=(0.0, 0.0, -1.0), chunk_points=1 << 21):
    """-> PanopticPoints of the k^3 sub-cell centres of every occupied leaf cell whose density exceeds min_density (see the module
    docstring for the exact definitions).  Works in chunks of at most max(chunk_points, k^3) points; one host read per chunk."""
    k = samples_per_axis
    if isinstance(k, bool) or not isinstance(k, (int, np.integer)) or not 1 <= k <= MAX_SAMPLES_PER_AXIS:
        raise ValueError(f"samples_per_axis must be an integer in [1, {MAX_SAMPLES_PER_AXIS}], got {k!r}")
    k = int(k)
    if int(chunk_points) < 1:
        raise ValueError(f"chunk_points must be positive, got {chunk_points}")
    _check_field(nef)
    dev = nef.decoder_density.lout.weight.device
    vd = torch.as_tensor(view_dir, dtype=torch.float32).reshape(3)
    if not torch.isfinite(vd).all() or float(vd.norm()) == 0.0:
        raise ValueError(f"view_dir must be a finite non-zero 3-vector, got {view_dir}")
    vd = (vd / vd.norm()).reshape(1, 3).to(dev)
    thr = PRUNE_MIN_DENSITY if min_density is None else float(min_density)
    grid = nef.grid
    level = int(grid.blas_level)
    blas = grid.blas.to(dev)
    cells = spc.unbatched_get_level_points(blas.points, blas.pyramid, level)
    C = cells.shape[0]
    if C == 0:
        return _empty_points(dev)
    kk = k ** 3
    cells_per_chunk = max(1, int(chunk_points) // kk)
    lod_idx = nef.num_lods - 1
    w_dc = _decoder_tensors(nef.decoder_density, 1) + _decoder_tensors(nef.decoder_color, 2)
    w_pan = _decoder_tensors(nef.decoder_semantics, 1) + _decoder_tensors(nef.decoder_inst, 2)
    Cs, Ci = int(nef.num_classes), int(nef.num_instances)
    temp = float(getattr(nef, 'inst_soft_temperature', 0.0))
    parts = []
    with torch.no_grad(), torch.autocast('cuda', enabled=False):
        lodw = nef._lodw(dev)
        for c0 in range(0, C, cells_per_chunk):
            xyz = ops.map_cell_points(cells[c0:c0 + cells_per_chunk], level, k)
            coords = xyz[:, None]
            feats = nef._encode(grid, coords, lod_idx)
            n = xyz.shape[0]
            # one ray carrying the chunk's points: every point is seen along view_dir
            sigma, rgb = ops.DecodeDCFn.apply(feats, lodw, vd, n, True, 'tiled', *w_dc)
            rows = torch.nonzero(sigma > thr).reshape(-1)          # the chunk's one host read: its output size
            if rows.numel() == 0:
                continue
            a, b = nef._panoptic_inputs(feats, coords, lod_idx, rows)
            del feats
            sl, ss, il, is_ = ops.pan_labels_f32(a, b, lodw, Cs, Ci, bool(nef.sem_softmax), bool(nef.inst_softmax), temp, *w_pan)
            del a, b
            parts.append((xyz.index_select(0, rows), rgb.index_select(0, rows), sigma.index_select(0, rows), sl, ss, il, is_))
    if not parts:
        return _empty_points(dev)
    if len(parts) == 1:
        return PanopticPoints(*parts[0])
    return PanopticPoints(*(torch.cat(col) for col in zip(*parts)))


def _thing_mask(num_instances, num_classes, things):
    """-> (Ci, Cs, thing mask with one bit per class in `things`, every class when None)."""
    Ci, Cs = int(num_instances), int(num_classes)
    if Ci < 1 or not 1 <= Cs <= MAX_SUMMARY_CLASSES:
        raise ValueError(f"num_instances must be >= 1 and num_classes in [1, {MAX_SUMMARY_CLASSES}], got {Ci}, {Cs}")
    if things is None:
        return Ci, Cs, (1 << Cs) - 1
    things = set(int(c) for c in things)
    if not all(0 <= c < Cs for c in things):
        raise ValueError(f"things must be classes in [0, {Cs}), got {sorted(things)}")
    return Ci, Cs, sum(1 << c for c in things)


def instance_summary(pts, num_instances, num_classes, things=None):
    """Per-instance statistics of a labelled map (csrc/mapping.cu, one launch + one host read for the error count) -> InstanceSummary.
    A point counts toward its instance only when its semantic class is in `things` (every class when None).  Raises ValueError if a
    point carries a semantic label outside [0, num_classes) or an instance label outside [0, num_instances)."""
    Ci, Cs, mask = _thing_mask(num_instances, num_classes, things)
    if not pts.xyz.is_cuda:
        raise RuntimeError("pagnerf_b200 map export runs on CUDA tensors only (no CPU fallback)")
    count, sum_xyz, sum_rgb, votes, bmin, bmax, errors = ops.map_instance_stats(pts.xyz, pts.rgb, pts.semantic, pts.instance, Cs, Ci, mask)
    bad = int(errors.item())
    if bad:
        raise ValueError(f"{bad} points carry a semantic label outside [0, {Cs}) or an instance label outside [0, {Ci})")
    n = count.to(torch.float64)[:, None]
    category = torch.where(count > 0, votes.argmax(dim=1), torch.full_like(count, -1))
    return InstanceSummary(count, sum_xyz / n, bmin, bmax, sum_rgb / n, votes, category)


def _is_int(v):
    return not isinstance(v, bool) and isinstance(v, (int, np.integer))


def _check_lattice(k, level):
    if not _is_int(k) or not 1 <= k <= MAX_SAMPLES_PER_AXIS:
        raise ValueError(f"samples_per_axis must be an integer in [1, {MAX_SAMPLES_PER_AXIS}], got {k!r}")
    if not _is_int(level) or not 0 <= level <= MAX_LEVEL:
        raise ValueError(f"level must be an integer in [0, {MAX_LEVEL}], got {level!r}")


def _lattice_errors(off, dup, k, level):
    errors = []
    if off:
        errors.append(f"{off} points are not on the lattice of samples_per_axis={k}, level={level}")
    if dup:
        errors.append(f"{dup} points repeat the lattice index of another point")
    return errors


def instance_components(pts, samples_per_axis, level, num_instances, num_classes, things=None, connectivity=26, min_points=1):
    """Objects of a labelled lattice map: connected components of equal instance labels (csrc/mapping.cu, one host read) ->
    InstanceComponents.  See the module docstring for the exact definitions and the memory bound.  Raises ValueError for points off
    the lattice of (samples_per_axis, level), for two points with the same lattice index and for out-of-range labels, with the
    number of points affected."""
    k = samples_per_axis
    _check_lattice(k, level)
    Ci, Cs, mask = _thing_mask(num_instances, num_classes, things)
    if connectivity not in (6, 26) or isinstance(connectivity, bool):
        raise ValueError(f"connectivity must be 6 or 26, got {connectivity!r}")
    if not _is_int(min_points) or min_points < 1:
        raise ValueError(f"min_points must be an integer >= 1, got {min_points!r}")
    if not pts.xyz.is_cuda:
        raise RuntimeError("pagnerf_b200 map export runs on CUDA tensors only (no CPU fallback)")
    if pts.xyz.shape[0] > MAX_COMPONENT_POINTS:
        raise ValueError(f"instance_components serves up to {MAX_COMPONENT_POINTS} points, got {pts.xyz.shape[0]}")
    k, level = int(k), int(level)
    component, info = ops.map_components(pts.xyz, pts.semantic, pts.instance, level, k, Cs, Ci, mask, int(connectivity),
                                         int(min_points))
    K, off, dup, bad = info.tolist()                # the call's one host read: the error counts and the output size
    errors = _lattice_errors(off, dup, k, level)
    if bad:
        errors.append(f"{bad} points carry a semantic label outside [0, {Cs}) or an instance label outside [0, {Ci})")
    if errors:
        raise ValueError("; ".join(errors))
    count, sum_xyz, sum_rgb, votes, bmin, bmax, inst = ops.map_component_stats(pts.xyz, pts.rgb, pts.semantic, pts.instance, component,
                                                                              Cs, K)
    n = count.to(torch.float64)[:, None]
    return InstanceComponents(component, count, inst, votes.argmax(dim=1), sum_xyz / n, sum_rgb / n, bmin, bmax, votes)


def _hash_slots(P):
    """C of the index table: the smallest power of two >= 2P (at least 2), include/pagnerf_b200.h pag_map_index_bytes"""
    return max(2, 1 << (2 * P - 1).bit_length()) if P > 0 else 2


def _check_tensor(name, t, shapes, dtype):
    """t must be a tensor of one of `shapes` (None = any size on that axis) and of `dtype`"""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a tensor, got {type(t).__name__}")
    ok = any(t.dim() == len(s) and all(w is None or t.shape[i] == w for i, w in enumerate(s)) for s in shapes)
    if not ok:
        want = " or ".join("[" + ", ".join("N" if w is None else str(w) for w in s) + "]" for s in shapes)
        raise ValueError(f"{name} must have shape {want}, got {list(t.shape)}")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")


def map_index(pts, samples_per_axis, level):
    """Lattice index of a map (csrc/mapping.cu, one launch + one host read for the error counts) -> MapIndex.  pts: PanopticPoints or
    its xyz f32 [P, 3].  Every point is indexed, whatever its labels.  Raises ValueError for points off the lattice of
    (samples_per_axis, level) and for two points with the same lattice index, with their number.  See the module docstring for the
    definitions and the memory bound (12 C bytes)."""
    k = samples_per_axis
    _check_lattice(k, level)
    xyz = pts.xyz if isinstance(pts, PanopticPoints) else pts
    _check_tensor("xyz", xyz, [(None, 3)], torch.float32)
    P = int(xyz.shape[0])
    if P > MAX_COMPONENT_POINTS:
        raise ValueError(f"map_index serves up to {MAX_COMPONENT_POINTS} points, got {P}")
    if not xyz.is_cuda:
        raise RuntimeError("pagnerf_b200 map lookups run on CUDA tensors only (no CPU fallback)")
    k, level = int(k), int(level)
    keys, points, info = ops.map_index(xyz, level, k)
    _, off, dup, _ = info.tolist()                  # the call's one host read: the error counts
    errors = _lattice_errors(off, dup, k, level)
    if errors:
        raise ValueError("; ".join(errors))
    return MapIndex(keys, points, k, level, P)


def _check_lookup(index, radius, component):
    if not isinstance(index, MapIndex):
        raise TypeError(f"index must be a MapIndex (map_index), got {type(index).__name__}")
    C = _hash_slots(index.P)
    if index.keys.shape != (C,) or index.points.shape != (C,) or index.keys.dtype != torch.int64 or index.points.dtype != torch.int32:
        raise ValueError(f"index is not the table of a {index.P}-point map: keys / points must be int64 / int32 [{C}]")
    if not _is_int(radius) or not 0 <= radius <= MAX_LOOKUP_RADIUS:
        raise ValueError(f"radius must be an integer in [0, {MAX_LOOKUP_RADIUS}], got {radius!r}")
    if component is not None:
        if not isinstance(component, torch.Tensor) or tuple(component.shape) != (index.P,):
            shape = list(component.shape) if isinstance(component, torch.Tensor) else type(component).__name__
            raise ValueError(f"component must have shape [{index.P}] (the indexed map's points), got {shape}")
        if component.dtype != torch.int64:
            raise TypeError(f"component must be torch.int64, got {component.dtype}")


def _check_cuda(*tensors):
    if not all(t.is_cuda for t in tensors if t is not None):
        raise RuntimeError("pagnerf_b200 map lookups run on CUDA tensors only (no CPU fallback)")


def lookup_points(index, xyz, radius=1, component=None):
    """Nearest map point in the (2 radius + 1)^3 lattice window around each query xyz f32 [Q, 3], and its object when component
    (i64 [P], e.g. InstanceComponents.component) is given -> MapLookup (csrc/mapping.cu, one launch, no host read).  See the module
    docstring for the exact definitions."""
    _check_lookup(index, radius, component)
    _check_tensor("xyz", xyz, [(None, 3)], torch.float32)
    _check_cuda(index.keys, index.points, xyz, component)
    point, obj = ops.map_lookup_points(index.keys, index.points, index.level, index.k, xyz, int(radius), component)
    return MapLookup(point, obj)


def lookup_rays(index, origins, dirs, depth, alpha, radius=1, min_alpha=0.5, component=None):
    """lookup_points for the surface point o + d * (depth / alpha) of each rendered ray (origins / dirs f32 [N, 3], depth / alpha
    f32 [N] or [N, 1], e.g. a tracer's rb.depth / rb.alpha); rays with alpha < min_alpha resolve to -1 -> MapLookup (one launch,
    no host read)."""
    _check_lookup(index, radius, component)
    if isinstance(min_alpha, bool) or not isinstance(min_alpha, (int, float, np.integer, np.floating)) or \
            not (0.0 < float(np.float32(min_alpha)) and float(min_alpha) <= 1.0):
        raise ValueError(f"min_alpha must be a number in (0, 1], got {min_alpha!r}")
    _check_tensor("origins", origins, [(None, 3)], torch.float32)
    N = int(origins.shape[0])
    _check_tensor("dirs", dirs, [(N, 3)], torch.float32)
    _check_tensor("depth", depth, [(N,), (N, 1)], torch.float32)
    _check_tensor("alpha", alpha, [(N,), (N, 1)], torch.float32)
    _check_cuda(index.keys, index.points, origins, dirs, depth, alpha, component)
    point, obj = ops.map_lookup_rays(index.keys, index.points, index.level, index.k, origins, dirs, depth, alpha, float(min_alpha),
                                     int(radius), component)
    return MapLookup(point, obj)


def _check_projection(fn, pts, k, level, view, intrinsics, height, width, max_radius, near, component):
    """The arguments project_map and object_visibility share -> (xyz, h, near) as the kernels take them"""
    _check_lattice(k, level)
    xyz = pts.xyz if isinstance(pts, PanopticPoints) else pts
    _check_tensor("xyz", xyz, [(None, 3)], torch.float32)
    P = int(xyz.shape[0])
    if P > MAX_COMPONENT_POINTS:
        raise ValueError(f"{fn} serves up to {MAX_COMPONENT_POINTS} points, got {P}")
    _check_tensor("view", view, [(None, 4, 4)], torch.float32)
    B = int(view.shape[0])
    if B > MAX_PROJECT_CAMERAS:
        raise ValueError(f"{fn} serves up to {MAX_PROJECT_CAMERAS} cameras per call, got {B}")
    _check_tensor("intrinsics", intrinsics, [(B, 4)], torch.float32)
    for name, n in (("height", height), ("width", width)):
        if not _is_int(n) or not 1 <= n <= MAX_PROJECT_SIDE:
            raise ValueError(f"{name} must be an integer in [1, {MAX_PROJECT_SIDE}], got {n!r}")
    if not _is_int(max_radius) or not 0 <= max_radius <= MAX_PROJECT_RADIUS:
        raise ValueError(f"max_radius must be an integer in [0, {MAX_PROJECT_RADIUS}], got {max_radius!r}")
    if isinstance(near, bool) or not isinstance(near, (int, float, np.integer, np.floating)) or \
            not (np.isfinite(np.float32(near)) and np.float32(near) > 0):
        raise ValueError(f"near must be a finite number > 0, got {near!r}")
    if component is not None:
        if not isinstance(component, torch.Tensor) or tuple(component.shape) != (P,):
            shape = list(component.shape) if isinstance(component, torch.Tensor) else type(component).__name__
            raise ValueError(f"component must have shape [{P}] (the projected map's points), got {shape}")
        if component.dtype != torch.int64:
            raise TypeError(f"component must be torch.int64, got {component.dtype}")
    if not all(t.is_cuda for t in (xyz, view, intrinsics, component) if t is not None):
        raise RuntimeError("pagnerf_b200 map projection runs on CUDA tensors only (no CPU fallback)")
    return xyz, float(np.float32(1.0) / np.float32(int(k) << int(level))), float(np.float32(near))


def project_map(pts, samples_per_axis, level, view, intrinsics, height, width, max_radius=8, near=0.01, component=None):
    """Z-buffered splatting of a map's points into B camera views (view f32 [B, 4, 4] world-to-camera, intrinsics f32 [B, 4] =
    (fx, fy, cx, cy)): per pixel the nearest covering map point, its depth and, with component (i64 [P]), its object -> MapView of
    [B, height, width] tensors (csrc/mapping.cu, a fill and two launches, no host read).  pts: PanopticPoints or its xyz f32 [P, 3].
    See the module docstring for the exact definitions."""
    xyz, h, near = _check_projection("project_map", pts, samples_per_axis, level, view, intrinsics, height, width, max_radius, near,
                                     component)
    point, depth, obj = ops.map_project(xyz, view, intrinsics, int(height), int(width), h, near, int(max_radius), component)
    return MapView(point, depth, obj)


def object_visibility(pts, samples_per_axis, level, view, intrinsics, height, width, component, num_objects, max_radius=8, near=0.01):
    """How much of each map object each of B camera views sees: per (view, object) the visible area, the unoccluded silhouette and
    the visible pixels' box -> ObjectVisibility (csrc/mapping.cu, one host read).  The arguments shared with project_map mean and
    are checked as there; component i64 [P] (e.g. InstanceComponents.component) gives each point's object in [0, num_objects) or
    -1.  Raises ValueError with their number for components outside [-1, num_objects).  See the module docstring for the exact
    definitions and the memory bound."""
    if component is None:
        raise TypeError("object_visibility needs component (i64 [P], each point's object or -1)")
    if not _is_int(num_objects) or not 0 <= num_objects <= MAX_COMPONENT_POINTS:
        raise ValueError(f"num_objects must be an integer in [0, {MAX_COMPONENT_POINTS}], got {num_objects!r}")
    xyz, h, near = _check_projection("object_visibility", pts, samples_per_axis, level, view, intrinsics, height, width, max_radius,
                                     near, component)
    K = int(num_objects)
    visible, silhouette, bbox, bad, _ = ops.map_visibility(xyz, view, intrinsics, int(height), int(width), h, near, int(max_radius),
                                                           component, K, VISIBILITY_BITMAP_BYTES)
    if bad:
        raise ValueError(f"{bad} points carry a component outside [-1, {K})")
    return ObjectVisibility(visible, silhouette, bbox)


PLY_PROPERTIES = [("x", "float", "<f4"), ("y", "float", "<f4"), ("z", "float", "<f4"),
                  ("red", "uchar", "u1"), ("green", "uchar", "u1"), ("blue", "uchar", "u1"),
                  ("density", "float", "<f4"), ("semantic", "int", "<i4"), ("semantic_score", "float", "<f4"),
                  ("instance", "int", "<i4"), ("instance_score", "float", "<f4")]


def write_ply(path, pts, component=None):
    """Binary little-endian PLY of a map, one vertex per point: x y z (float), red green blue (uchar, round(255 * clamp(rgb, 0, 1))),
    density, semantic (int), semantic_score, instance (int), instance_score, and with `component` (i64 [P], e.g.
    InstanceComponents.component) a last int property `component`."""
    P = int(pts.xyz.shape[0])
    props = PLY_PROPERTIES + ([("component", "int", "<i4")] if component is not None else [])
    rec = np.empty(P, dtype=[(n, t) for n, _, t in props])
    xyz = pts.xyz.detach().cpu().numpy().astype(np.float32)
    rgb = np.rint(np.clip(pts.rgb.detach().cpu().numpy().astype(np.float64), 0.0, 1.0) * 255.0).astype(np.uint8)
    for i, n in enumerate("xyz"):
        rec[n] = xyz[:, i]
    for i, n in enumerate(("red", "green", "blue")):
        rec[n] = rgb[:, i]
    rec["density"] = pts.density.detach().cpu().numpy()
    rec["semantic"] = pts.semantic.detach().cpu().numpy()
    rec["semantic_score"] = pts.semantic_score.detach().cpu().numpy()
    rec["instance"] = pts.instance.detach().cpu().numpy()
    rec["instance_score"] = pts.instance_score.detach().cpu().numpy()
    if component is not None:
        if tuple(component.shape) != (P,):
            raise ValueError(f"component must have shape ({P},), got {tuple(component.shape)}")
        rec["component"] = component.detach().cpu().numpy()
    header = ["ply", "format binary_little_endian 1.0", f"element vertex {P}"]
    header += [f"property {t} {n}" for n, t, _ in props]
    header += ["end_header"]
    with open(path, "wb") as f:
        f.write(("\n".join(header) + "\n").encode("ascii"))
        f.write(rec.tobytes())
