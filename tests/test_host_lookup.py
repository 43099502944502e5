"""CPU: the map-lookup oracle (oracle/lookup.py) against brute force over every map point, its ray form against its point form,
and argument validation of pagnerf_b200.mapping.map_index / lookup_points / lookup_rays."""
import numpy as np
import pytest
import torch

from oracle import lookup as ol


def _random_map(seed, k, level, fill):
    """Points on the (k, level) lattice in random order -> (xyz f32 [P,3], lattice indices [P,3])."""
    rng = np.random.default_rng(seed)
    D = k << level
    j = np.argwhere(rng.random((D, D, D)) < fill)
    j = j[rng.permutation(len(j))]
    return (2 * j + 1).astype(np.float32) / np.float32(D) - np.float32(1.0), j


def _queries(seed, D, n=400):
    """Lattice centres, points on sub-cell faces, edges and corners (t = j + 0.5: the tie cases), points just outside the cube,
    uniform points, NaN and inf."""
    rng = np.random.default_rng(seed)
    f32 = np.float32
    centre = lambda j: (2 * j + 1).astype(f32) / f32(D) - f32(1.0)
    face = lambda j: (2 * (j + 1)).astype(f32) / f32(D) - f32(1.0)          # t = j + 0.5 exactly
    j = rng.integers(-1, D + 1, (n, 3))
    q = [centre(j), face(j)]
    mixed = centre(j)
    pick = rng.random((n, 3)) < 0.5
    mixed[pick] = face(j)[pick]
    q.append(mixed)
    outside = rng.uniform(-1, 1, (n, 3)).astype(f32)
    axis = rng.integers(0, 3, n)
    outside[np.arange(n), axis] = rng.choice([-1, 1], n) * rng.uniform(1.0, 1.0 + 12.0 / D, n).astype(f32)
    q.append(outside)
    q.append(rng.uniform(-1.2, 1.2, (n, 3)).astype(f32))
    special = rng.uniform(-1, 1, (12, 3)).astype(f32)
    special[0, 0], special[1, 1], special[2, 2] = np.nan, np.inf, -np.inf
    special[3] = np.nan
    special[4, :] = [np.inf, 0, 0]
    q.append(special)
    return np.concatenate(q).astype(f32)


@pytest.mark.parametrize("radius", [0, 1, 2, 3])
@pytest.mark.parametrize("seed,k,level,fill", [(0, 1, 3, 0.3), (1, 2, 2, 0.15), (2, 2, 3, 0.05)])
def test_oracle_matches_brute_force(radius, seed, k, level, fill):
    xyz, _ = _random_map(seed, k, level, fill)
    D = k << level
    q = _queries(seed + 10 * radius, D)
    idx = ol.index(xyz, k, level)
    assert idx["errors"] == dict(off_lattice=0, duplicates=0)
    comp = np.random.default_rng(seed).integers(-1, 5, len(xyz))
    point, obj = ol.lookup_points(idx, q, radius, comp)
    want = ol.brute_force(xyz, k, level, q, radius)
    assert np.array_equal(point, want)
    assert np.array_equal(obj, np.where(want >= 0, comp[np.maximum(want, 0)], -1))
    assert (point >= 0).any() and (point < 0).any()
    assert (point[-12:-7] == -1).all()                      # non-finite coordinates
    assert ol.lookup_points(idx, q, radius)[1] is None


def test_ties_go_to_the_smallest_point_index():
    D, k, level = 8, 2, 2
    j = np.array([[4, 4, 4], [3, 4, 4], [4, 3, 4], [3, 3, 4]])
    for order in (np.arange(4), np.arange(4)[::-1]):
        xyz = (2 * j[order] + 1).astype(np.float32) / np.float32(D) - np.float32(1.0)
        idx = ol.index(xyz, k, level)
        # t = (3.5, 3.5, 4): all four at the same distance 0.5
        q = np.array([[2 * 4 / D - 1, 2 * 4 / D - 1, (2 * 4 + 1) / D - 1]], np.float32)
        point, _ = ol.lookup_points(idx, q, 1)
        assert point.tolist() == [0]
        assert ol.brute_force(xyz, k, level, q, 1).tolist() == [0]


def test_window_bounds_and_empty_map():
    k, level = 1, 3
    D = 8
    xyz = np.array([[(2 * 0 + 1) / D - 1] * 3], np.float32)                  # lattice index (0, 0, 0)
    idx = ol.index(xyz, k, level)
    for radius in range(4):
        # t = -radius - 0.5 is inside the window range, just below it is not
        edge = np.float32((-radius - 0.5 + 0.5) * 2 / D - 1)
        below = np.nextafter(edge, np.float32(-2))
        q = np.array([[edge, xyz[0, 1], xyz[0, 2]], [below, xyz[0, 1], xyz[0, 2]]], np.float32)
        point, _ = ol.lookup_points(idx, q, radius)
        assert point.tolist() == [0, -1]
        assert np.array_equal(point, ol.brute_force(xyz, k, level, q, radius))
    empty = ol.index(np.zeros((0, 3), np.float32), k, level)
    assert ol.lookup_points(empty, xyz, 2)[0].tolist() == [-1]


@pytest.mark.parametrize("radius", [0, 1, 2])
def test_ray_form_equals_point_form(radius):
    xyz, _ = _random_map(3, 2, 3, 0.2)
    idx = ol.index(xyz, 2, 3)
    rng = np.random.default_rng(radius)
    N = 3000
    o = rng.uniform(-1, 1, (N, 3)).astype(np.float32)
    d = rng.normal(size=(N, 3)).astype(np.float32)
    depth = rng.uniform(0, 1.5, N).astype(np.float32)
    alpha = rng.uniform(0, 1, N).astype(np.float32)
    min_alpha = 0.4
    alpha[:50] = np.float32(min_alpha)                       # looked up
    alpha[50:60] = 0.0                                       # s = inf or NaN: -1
    depth[60:70] = np.inf
    comp = rng.integers(-1, 9, len(xyz))
    point, obj = ol.lookup_rays(idx, o, d, depth, alpha, radius, min_alpha, comp)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        s = depth / alpha
        x = (o + d * s[:, None]).astype(np.float32)
    valid = (alpha >= np.float32(min_alpha)) & np.isfinite(s)
    want_p, want_o = ol.lookup_points(idx, x, radius, comp)
    assert np.array_equal(point, np.where(valid, want_p, -1))
    assert np.array_equal(obj, np.where(valid, want_o, -1))
    assert (point[:50] >= 0).any() and (point[50:70] == -1).all()
    assert np.array_equal(point, ol.brute_force(xyz, 2, 3, np.where(valid[:, None], x, np.nan), radius))


def test_index_error_counts():
    xyz, _ = _random_map(4, 2, 2, 0.3)
    bad = np.concatenate([xyz, xyz[:3]])
    bad[5, 1] = np.nextafter(bad[5, 1], np.float32(2))
    assert ol.index(bad, 2, 2)["errors"] == dict(off_lattice=1, duplicates=3)


def test_hash_slots_matches_the_library_rule():
    from pagnerf_b200.mapping.panoptic_map import _hash_slots
    for P in list(range(0, 70)) + [1 << 20, (1 << 20) + 1, 11_200_000, 1 << 30]:
        c = 2
        while c < 2 * P:
            c <<= 1
        assert _hash_slots(P) == c, P


def _cpu_index(P=10):
    from pagnerf_b200.mapping import MapIndex
    from pagnerf_b200.mapping.panoptic_map import _hash_slots
    C = _hash_slots(P)
    return MapIndex(torch.zeros(C, dtype=torch.int64), torch.zeros(C, dtype=torch.int32), 2, 3, P)


def _rays(N=5):
    return (torch.zeros(N, 3), torch.ones(N, 3), torch.ones(N, 1), torch.ones(N, 1))


@pytest.mark.parametrize("radius", [-1, 5, 1.0, True, "1", None])
def test_radius_validation(radius):
    from pagnerf_b200.mapping import lookup_points, lookup_rays
    with pytest.raises(ValueError, match="radius"):
        lookup_points(_cpu_index(), torch.zeros(4, 3), radius=radius)
    with pytest.raises(ValueError, match="radius"):
        lookup_rays(_cpu_index(), *_rays(), radius=radius)


@pytest.mark.parametrize("min_alpha", [0, 0.0, -0.5, 1.0000001, 2, float("nan"), 1e-60, True, "0.5", None])
def test_min_alpha_validation(min_alpha):
    from pagnerf_b200.mapping import lookup_rays
    with pytest.raises(ValueError, match="min_alpha"):
        lookup_rays(_cpu_index(), *_rays(), min_alpha=min_alpha)


def test_shape_and_dtype_validation():
    from pagnerf_b200.mapping import lookup_points, lookup_rays
    idx = _cpu_index()
    with pytest.raises(ValueError, match="xyz"):
        lookup_points(idx, torch.zeros(4, 2))
    with pytest.raises(ValueError, match="xyz"):
        lookup_points(idx, torch.zeros(12))
    with pytest.raises(TypeError, match="xyz"):
        lookup_points(idx, torch.zeros(4, 3, dtype=torch.float64))
    o, d, t, a = _rays(5)
    for args, err, match in [((o[:4], d, t, a), ValueError, "dirs"), ((o, d[:, :2], t, a), ValueError, "dirs"),
                             ((o, d, t[:4], a), ValueError, "depth"), ((o, d, torch.ones(5, 2), a), ValueError, "depth"),
                             ((o, d, t, a.reshape(1, 5)), ValueError, "alpha"), ((o.double(), d, t, a), TypeError, "origins"),
                             ((o, d, t.half(), a), TypeError, "depth"), ((o, d, t, a.double()), TypeError, "alpha")]:
        with pytest.raises(err, match=match):
            lookup_rays(idx, *args)
    with pytest.raises(TypeError, match="index"):
        lookup_points(tuple(idx), torch.zeros(4, 3))
    with pytest.raises(ValueError, match="table"):
        lookup_points(idx._replace(P=100), torch.zeros(4, 3))
    with pytest.raises(ValueError, match="table"):
        lookup_points(idx._replace(points=idx.points.long()), torch.zeros(4, 3))


def test_component_validation():
    from pagnerf_b200.mapping import lookup_points, lookup_rays
    idx = _cpu_index(10)
    for comp in (torch.zeros(9, dtype=torch.int64), torch.zeros(11, dtype=torch.int64), torch.zeros(10, 1, dtype=torch.int64),
                 [0] * 10):
        with pytest.raises(ValueError, match="component"):
            lookup_points(idx, torch.zeros(4, 3), component=comp)
        with pytest.raises(ValueError, match="component"):
            lookup_rays(idx, *_rays(), component=comp)
    with pytest.raises(TypeError, match="component"):
        lookup_points(idx, torch.zeros(4, 3), component=torch.zeros(10, dtype=torch.int32))


def test_cpu_tensors_are_refused():
    from pagnerf_b200.mapping import PanopticPoints, map_index, lookup_points, lookup_rays
    idx = _cpu_index(10)
    with pytest.raises(RuntimeError, match="CUDA"):
        lookup_points(idx, torch.zeros(4, 3), component=torch.zeros(10, dtype=torch.int64))
    with pytest.raises(RuntimeError, match="CUDA"):
        lookup_rays(idx, *_rays(), radius=0, min_alpha=1.0)
    xyz, _ = _random_map(0, 2, 2, 0.3)
    with pytest.raises(RuntimeError, match="CUDA"):
        map_index(torch.from_numpy(xyz), samples_per_axis=2, level=2)
    P = len(xyz)
    pts = PanopticPoints(torch.from_numpy(xyz), torch.zeros(P, 3), torch.zeros(P), torch.zeros(P, dtype=torch.int64), torch.zeros(P),
                         torch.zeros(P, dtype=torch.int64), torch.zeros(P))
    with pytest.raises(RuntimeError, match="CUDA"):
        map_index(pts, samples_per_axis=2, level=2)


@pytest.mark.parametrize("kwargs,err,match", [
    (dict(samples_per_axis=0), ValueError, "samples_per_axis"), (dict(samples_per_axis=9), ValueError, "samples_per_axis"),
    (dict(samples_per_axis=2.0), ValueError, "samples_per_axis"), (dict(level=-1), ValueError, "level"),
    (dict(level=16), ValueError, "level"), (dict(level=True), ValueError, "level"),
    (dict(xyz=torch.zeros(4, 2)), ValueError, "xyz"), (dict(xyz=torch.zeros(4, 3, dtype=torch.float64)), TypeError, "xyz")])
def test_map_index_argument_validation(kwargs, err, match):
    from pagnerf_b200.mapping import map_index
    xyz = kwargs.pop("xyz", torch.zeros(4, 3))
    args = dict(samples_per_axis=2, level=3)
    args.update(kwargs)
    with pytest.raises(err, match=match):
        map_index(xyz, **args)
