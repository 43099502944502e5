"""CPU: the object-shape oracle (oracle/shape.py) on hand-computed shapes, argument validation of pagnerf_b200.mapping.object_shape
and its C ABI entry."""
import numpy as np
import pytest
import torch

from oracle import shape as osh

K_, LEVEL = 2, 4
D = K_ << LEVEL                                                       # 32


def _xyz(j):
    return ((2 * np.asarray(j, np.int64) + 1).astype(np.float32) / np.float32(D) - np.float32(1.0)).reshape(-1, 3)


def _shape(j, comp=None, K=1):
    j = np.asarray(j, np.int64).reshape(-1, 3)
    return osh.shape(_xyz(j), K_, LEVEL, np.zeros(len(j), np.int64) if comp is None else comp, K)


def _world(c):
    return (2.0 * np.asarray(c, np.float64) + 1.0) / D - 1.0


def test_single_point():
    r = _shape([[5, 9, 30]])
    assert r["errors"] == dict(off_lattice=0, bad_components=0)
    assert (r["covariance"] == 0).all() and (r["variance"] == 0).all()
    assert np.array_equal(r["axes"][0], np.eye(3))
    assert np.array_equal(r["extent"][0], np.full(3, 2.0 / D))      # one cell
    assert np.array_equal(r["center"][0], _world([5, 9, 30]))


def test_two_points_along_an_axis():
    """j = (3, 4, 4) and (3, 8, 4): lattice variance 4 along y, 0 elsewhere; the zero eigenvalues keep the x, z order"""
    r = _shape([[3, 4, 4], [3, 8, 4]])
    cov = np.zeros((3, 3))
    cov[1, 1] = 4.0 * 4 / D / D
    assert np.array_equal(r["covariance"][0], cov)
    assert np.array_equal(r["variance"][0], [cov[1, 1], 0.0, 0.0])
    assert np.array_equal(r["axes"][0], [[0, 1, 0], [1, 0, 0], [0, 0, -1]])       # axes[2] = e_y x e_x
    assert np.array_equal(r["extent"][0], np.array([5.0, 1.0, 1.0]) * 2.0 / D)
    assert np.allclose(r["center"][0], _world([3, 6, 4]), rtol=0, atol=1e-15)


@pytest.mark.parametrize("radius", [1, 3, 5])
def test_lattice_ball_is_isotropic(radius):
    """A lattice ball is symmetric under axis reflections and permutations: its covariance is exactly diagonal with equal entries,
    so the axes are the world axes and the box is the (2r + 1)-cell cube around the centre"""
    c = np.array([15, 16, 14])
    off = np.stack(np.meshgrid(*[np.arange(-radius, radius + 1)] * 3, indexing="ij"), -1).reshape(-1, 3)
    r = _shape(c + off[(off ** 2).sum(1) <= radius * radius])
    cov = r["covariance"][0]
    assert (cov[~np.eye(3, dtype=bool)] == 0).all() and cov[0, 0] == cov[1, 1] == cov[2, 2] > 0
    assert np.array_equal(r["axes"][0], np.eye(3))
    assert np.array_equal(r["extent"][0], np.full(3, (2 * radius + 1) * 2.0 / D))
    assert np.array_equal(r["center"][0], _world(c))


def test_axis_aligned_box():
    """5 x 7 x 3 points: lattice variances (n^2 - 1) / 12 = 2, 4, 2/3, so the order is y, x, z"""
    j = np.argwhere(np.ones((5, 7, 3), bool)) + [2, 10, 20]
    r = _shape(j)
    assert np.array_equal(r["covariance"][0][~np.eye(3, dtype=bool)], np.zeros(6))
    assert np.array_equal(np.diag(r["covariance"][0]), [2.0 * 4 / D / D, 4.0 * 4 / D / D, (70 / 105) * 4 / D / D])
    assert np.array_equal(r["axes"][0], [[0, 1, 0], [1, 0, 0], [0, 0, -1]])
    assert np.array_equal(r["extent"][0], np.array([7.0, 5.0, 3.0]) * 2.0 / D)
    assert np.array_equal(r["center"][0], _world([4, 13, 21]))


def test_rotated_segment_gets_its_length():
    """21 points on a 45-degree diagonal in the x-y plane: the axis-aligned box is 21 cells on x and y, the principal box
    20 sqrt(2) + 1 cells long and one cell across; the variance along it is 2 (21^2 - 1) / 12 lattice units"""
    t = np.arange(-10, 11)
    r = _shape(np.stack([t + 15, t + 15, np.full(21, 7)], 1))
    u = np.array([1.0, 1.0, 0.0]) / np.sqrt(2.0)
    assert np.allclose(r["variance"][0], [2 * (21 ** 2 - 1) / 12 * 4 / D / D, 0, 0], rtol=1e-14, atol=1e-18)
    assert np.allclose(r["axes"][0][0], u, atol=1e-15)
    assert np.allclose(r["extent"][0], np.array([20 * np.sqrt(2.0) + 1, 1, 1]) * 2.0 / D, rtol=1e-14)
    assert np.allclose(r["center"][0], _world([15, 15, 7]), atol=1e-14)
    assert np.allclose(np.cross(r["axes"][0][0], r["axes"][0][1]), r["axes"][0][2], atol=1e-15)


def test_rotated_box_axes_follow_the_symmetry():
    """A box rotated by 45 degrees about z is mapped to itself by the reflection x <-> y and by z -> -z: its eigenvectors are
    exactly (1, 1, 0) / sqrt(2), (1, -1, 0) / sqrt(2) and z, with the longer side first"""
    g = np.stack(np.meshgrid(*[np.arange(32)] * 3, indexing="ij"), -1).reshape(-1, 3)
    d = g - [15, 15, 15]
    u, v = (d[:, 0] + d[:, 1]) / np.sqrt(2), (d[:, 0] - d[:, 1]) / np.sqrt(2)
    j = g[(np.abs(u) <= 12) & (np.abs(v) <= 5) & (np.abs(d[:, 2]) <= 2)]
    r = _shape(j)
    s = 1 / np.sqrt(2.0)
    assert np.allclose(np.abs(r["axes"][0]), [[s, s, 0], [s, s, 0], [0, 0, 1]], atol=1e-15)
    assert r["axes"][0][1][0] > 0 > r["axes"][0][1][1]                 # the sign rule: the lowest index wins the magnitude tie
    assert r["variance"][0][0] > r["variance"][0][1] > r["variance"][0][2]


def test_empty_objects_and_skipped_points():
    j = np.array([[1, 2, 3], [4, 5, 6], [7, 8, 9]])
    r = _shape(j, np.array([2, -1, 2]), K=3)
    for key in ("covariance", "variance", "axes", "center", "extent"):
        assert np.isnan(r[key][:2]).all() and not np.isnan(r[key][2]).any(), key
    assert r["n"].tolist() == [0, 0, 2]
    bad = _shape(j, np.array([3, -2, 0]), K=3)
    assert bad["errors"] == dict(off_lattice=0, bad_components=2)
    x = _xyz(j)
    x[0, 1] = np.nextafter(x[0, 1], np.float32(2))
    assert osh.shape(x, K_, LEVEL, np.zeros(3, np.int64), 1)["errors"]["off_lattice"] == 1


def test_weighted_moments_are_repeated_points():
    j = np.array([[1, 2, 3], [30, 0, 17], [8, 8, 8]])
    w = np.array([3, 1, 2])
    assert osh.moments(j, np.zeros(3, np.int64), 1, w) == osh.moments(np.repeat(j, w, 0), np.zeros(6, np.int64), 1)


def test_box_total_order_and_keys():
    v = np.array([-np.inf, -2.5, -0.0, 0.0, 1e-300, 3.0, np.inf])
    k = osh.total_key(v)
    assert (np.diff(k.astype(object)) > 0).all()
    assert np.array_equal(osh.from_key(k).view(np.uint64), v.view(np.uint64))


def _cpu_args(P=10):
    return dict(pts=torch.zeros(P, 3), samples_per_axis=2, level=3, component=torch.zeros(P, dtype=torch.int64), num_objects=3)


@pytest.mark.parametrize("kwargs,err,match", [
    (dict(samples_per_axis=0), ValueError, "samples_per_axis"), (dict(samples_per_axis=9), ValueError, "samples_per_axis"),
    (dict(level=16), ValueError, "level"), (dict(level=1.0), ValueError, "level"),
    (dict(pts=torch.zeros(4, 2)), ValueError, "xyz"), (dict(pts=torch.zeros(4, 3, dtype=torch.float64)), TypeError, "xyz"),
    (dict(pts=[[0.0, 0.0, 0.0]]), TypeError, "xyz"), (dict(component=None), TypeError, "component"),
    (dict(component=torch.zeros(9, dtype=torch.int64)), ValueError, "component must have shape \\[10\\]"),
    (dict(component=torch.zeros(10, dtype=torch.int32)), TypeError, "component"),
    (dict(num_objects=-1), ValueError, "num_objects"), (dict(num_objects=2.0), ValueError, "num_objects"),
    (dict(num_objects=True), ValueError, "num_objects"), (dict(num_objects=(1 << 30) + 1), ValueError, "num_objects")])
def test_argument_validation(kwargs, err, match):
    from pagnerf_b200.mapping import object_shape
    args = _cpu_args()
    args.update(kwargs)
    with pytest.raises(err, match=match):
        object_shape(**args)


def test_cpu_tensors_are_refused():
    from pagnerf_b200.mapping import object_shape
    with pytest.raises(RuntimeError, match="CUDA"):
        object_shape(**_cpu_args())


def test_shape_entry_point_in_the_header_and_the_library():
    from pagnerf_b200 import _lib, ops
    from pagnerf_b200.mapping import panoptic_map
    protos = _lib.parse_header()
    assert len(protos["pag_map_shape"]) == 14
    assert _lib.KERNELS_PER_CALL["pag_map_shape"] == 4
    assert "pag_map_shape" in _lib.exported_symbols()
    assert ops.SHAPE_ACC_WORDS == 22 and panoptic_map.SHAPE_WORKSPACE_BYTES == 176
