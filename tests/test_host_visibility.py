"""CPU: the per-object visibility oracle (oracle/visibility.py) against an independent route (the projection of each object's points
alone), a hand-computed known answer, argument validation of pagnerf_b200.mapping.object_visibility and its C ABI entries."""
import numpy as np
import pytest
import torch

from oracle import projection as op
from oracle import visibility as ov
from tests.test_host_projection import _cameras, _cloud


@pytest.mark.parametrize("max_radius", [0, 1, 3, 8])
@pytest.mark.parametrize("seed,k,level,H,W", [(0, 2, 2, 9, 13), (1, 1, 3, 12, 10), (2, 4, 1, 7, 16)])
def test_oracle_matches_projection_per_object(max_radius, seed, k, level, H, W):
    """silhouette[b, o] is the visible count of a projection of object o's points alone; visible and bbox follow the object image
    of the projection of all points.  The cloud has ties, near-plane, off-screen, NaN and inf points, and clamped footprints."""
    near = 0.0625
    x = _cloud(seed, 70, near)
    V, K = _cameras(W, H)
    comp = np.random.default_rng(seed).integers(-1, 5, 70)
    n_obj = 6                                                         # object 5 has no point
    visible, silhouette, bbox = ov.visibility(x, k, level, V, K, H, W, comp, n_obj, max_radius, near)
    _, _, obj = op.project(x, k, level, V, K, H, W, max_radius, near, comp)
    for o in range(n_obj):
        alone = op.project(x[comp == o], k, level, V, K, H, W, max_radius, near)[0]
        assert np.array_equal(silhouette[:, o], (alone >= 0).sum((1, 2)))
        for b in range(len(V)):
            m = obj[b] == o
            assert visible[b, o] == m.sum()
            if m.any():
                r, c = np.nonzero(m)
                assert bbox[b, o].tolist() == [c.min(), r.min(), c.max(), r.max()]
            else:
                assert (bbox[b, o] == -1).all()
    assert (visible <= silhouette).all() and (visible < silhouette).any() and (silhouette[:, 5] == 0).all()
    assert np.array_equal(visible.sum(1), (obj >= 0).sum((1, 2)))


def test_known_answer_occluded_square():
    """max_radius = 0, one point per pixel: a 4 x 4 square of object 0 at z = 1 behind a 2 x 3 patch of object 1 at z = 0.5 and one
    stuff point (-1) at z = 0.25 in front of both."""
    V = np.eye(4, dtype=np.float32)[None].copy()
    V[0, 2, 3] = -1.0                                                 # camera at (0, 0, 1) looking down -z
    K = np.array([[1.0, 1.0, 0.0, 0.0]], np.float32)
    pts, comp = [], []
    def put(c, r, z, o):                                               # a point projecting to the centre of pixel (r, c) at depth z
        pts.append([(c + 0.5) * z, (r + 0.5) * z, 1.0 - z])
        comp.append(o)
    for r in range(2, 6):
        for c in range(3, 7):
            put(c, r, 1.0, 0)
    for r in range(1, 3):
        for c in range(5, 8):
            put(c, r, 0.5, 1)
    put(3, 5, 0.25, -1)
    x = np.array(pts, np.float32)
    visible, silhouette, bbox = ov.visibility(x, 2, 2, V, K, 8, 10, np.array(comp), 3, max_radius=0)
    # the patch hides square pixels (2, 5) and (2, 6), the stuff point (5, 3): 16 - 3 = 13 visible; the patch is all visible
    assert visible.tolist() == [[13, 6, 0]] and silhouette.tolist() == [[16, 6, 0]]
    assert bbox.tolist() == [[[3, 2, 6, 5], [5, 1, 7, 2], [-1, -1, -1, -1]]]


def _cpu_args(P=10, B=2):
    return dict(pts=torch.zeros(P, 3), samples_per_axis=2, level=3, view=torch.eye(4).repeat(B, 1, 1), intrinsics=torch.ones(B, 4),
                height=8, width=8, component=torch.zeros(P, dtype=torch.int64), num_objects=3)


@pytest.mark.parametrize("kwargs,err,match", [
    (dict(samples_per_axis=0), ValueError, "samples_per_axis"), (dict(level=16), ValueError, "level"),
    (dict(pts=torch.zeros(4, 2)), ValueError, "xyz"), (dict(pts=torch.zeros(4, 3, dtype=torch.float64)), TypeError, "xyz"),
    (dict(view=torch.eye(4)), ValueError, "view"), (dict(view=torch.zeros(65536, 4, 4)), ValueError, "cameras"),
    (dict(intrinsics=torch.ones(3, 4)), ValueError, "intrinsics"), (dict(height=0), ValueError, "height"),
    (dict(width=16385), ValueError, "width"), (dict(max_radius=33), ValueError, "max_radius"), (dict(near=0), ValueError, "near"),
    (dict(near=float("nan")), ValueError, "near"), (dict(component=None), TypeError, "component"),
    (dict(component=torch.zeros(9, dtype=torch.int64)), ValueError, "component"),
    (dict(component=torch.zeros(10, dtype=torch.int32)), TypeError, "component"),
    (dict(num_objects=-1), ValueError, "num_objects"), (dict(num_objects=2.0), ValueError, "num_objects"),
    (dict(num_objects=True), ValueError, "num_objects"), (dict(num_objects=None), ValueError, "num_objects"),
    (dict(num_objects=(1 << 30) + 1), ValueError, "num_objects")])
def test_argument_validation(kwargs, err, match):
    from pagnerf_b200.mapping import object_visibility
    args = _cpu_args()
    args.update(kwargs)
    with pytest.raises(err, match=match):
        object_visibility(**args)


def test_cpu_tensors_are_refused():
    from pagnerf_b200.mapping import object_visibility
    with pytest.raises(RuntimeError, match="CUDA"):
        object_visibility(**_cpu_args())


def test_bitmap_rounds():
    """One round when the bitmaps fit the cap; otherwise windows of cap - (largest bitmap) words"""
    from pagnerf_b200 import ops
    from pagnerf_b200.mapping import panoptic_map
    assert panoptic_map.VISIBILITY_BITMAP_BYTES >= 16384 * 16384 // 8
    assert ops.silhouette_bitmap_words(0, 8, 8, 1 << 20) == (0, 0)
    assert ops.silhouette_bitmap_words(1000, 8, 40, 4000) == (1000, 1)
    assert ops.silhouette_bitmap_words(1001, 8, 40, 4000) == (1000, -(-1001 // 984))
    with pytest.raises(ValueError, match="largest bitmap"):
        ops.silhouette_bitmap_words(1001, 500, 40, 4000)


def test_visibility_entry_points_in_the_header_and_the_library():
    from pagnerf_b200 import _lib
    protos = _lib.parse_header()
    assert len(protos["pag_map_visibility"]) == 20 and len(protos["pag_map_visibility_silhouette"]) == 20
    assert _lib.KERNELS_PER_CALL["pag_map_visibility"] == 6
    assert {"pag_map_visibility", "pag_map_visibility_silhouette"} <= set(_lib.exported_symbols())
