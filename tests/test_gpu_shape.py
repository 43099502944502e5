"""GPU: size and orientation of map objects (pagnerf_b200.mapping.object_shape; csrc/mapping.cu) against the CPU oracle
(oracle/shape.py): bit-exact covariance (also past 2^64 sums and on f64 rounding ties), eigen-decomposition within stated
tolerances, the box bit for bit along the device's axes, exact answers on lattice balls and boxes, planted rotated shapes,
invariances, edge cases, errors, host reads, memory and the golden fields' maps."""
import gc

import numpy as np
import pytest
import torch

from oracle import shape as osh
from oracle.components import lattice_index
from tests.test_gpu_components import _coords, _synthetic
from tests.util import load_golden, build_cuda_nef

pytestmark = pytest.mark.gpu
DEV = "cuda"
FIELDS = ("covariance", "variance", "axes", "center", "extent")


@pytest.fixture(autouse=True)
def _collect_device_garbage():
    """Free device tensors held in reference cycles (the tracebacks of the ValueError tests) when each test ends, so they are not
    freed inside a later test's peak-memory window"""
    yield
    gc.collect()


def _t(a, dt=torch.float32):
    return torch.as_tensor(np.asarray(a)).to(dt).to(DEV)


def _run(xyz, k, level, comp, K):
    from pagnerf_b200.mapping import object_shape
    return object_shape(xyz, samples_per_axis=k, level=level, component=comp, num_objects=K)


def _bits_equal(a, b):
    """equal bit for bit where not NaN, NaN at the same places"""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint64), b[~nb].view(np.uint64))


def _check_eigen(var, axes, ref_var, ref_axes, cov):
    """variance and axes against the oracle's numpy.linalg.eigh.

    Tolerances: Jacobi and eigh are both backward stable, so each computed eigenvalue lies within a small multiple of
    eps ||C||_2 (eps = 2^-52) of the exact one, and an eigenvector (or the projector on a cluster of eigenvalues) within a small
    multiple of eps ||C||_2 / gap of the exact one, gap = the distance to the other eigenvalues.  Eigenvalues: |dv| <= 1e-12 ||C||
    (a margin of ~4000 eps).  Axes: compared only across relative eigengaps gap / ||C|| >= 1e-6, where the bound is ~1e-10; tolerance
    1e-8 on the projectors.  Eigenvalues closer than that form a cluster whose subspace is compared by its projector."""
    for o in range(len(cov)):
        if np.isnan(cov[o]).any():
            assert np.isnan(var[o]).all() and np.isnan(axes[o]).all() and np.isnan(ref_var[o]).all()
            continue
        scale = max(np.abs(ref_var[o]).max(), 1e-300)
        assert np.abs(var[o] - ref_var[o]).max() <= 1e-12 * scale, (o, var[o], ref_var[o])
        e = axes[o]
        assert np.abs(e @ e.T - np.eye(3)).max() <= 1e-12 and np.linalg.det(e) > 0, o
        for a in range(2):                                            # the sign rule, exactly
            m = int(np.argmax(np.abs(e[a])))
            assert e[a, m] > 0, (o, a)
        clusters, start = [], 0
        for a in range(1, 4):
            if a == 3 or ref_var[o, a - 1] - ref_var[o, a] >= 1e-6 * scale:
                clusters.append(list(range(start, a)))
                start = a
        for c in clusters:
            Pd, Pr = e[c].T @ e[c], ref_axes[o][c].T @ ref_axes[o][c]
            assert np.abs(Pd - Pr).max() <= 1e-8, (o, c)


def _check(xyz, k, level, comp, K, weight=None, j=None):
    """object_shape against the oracle: covariance bit for bit, eigen-decomposition by _check_eigen, the box (lo, hi from the
    workspace; center, extent) bit for bit by the oracle's box along the device's axes -> the result"""
    from pagnerf_b200 import ops
    got = _run(xyz, k, level, comp, K)
    cov, var, axes, center, extent, acc, errors = ops.map_shape(xyz, level, k, comp, K)
    assert errors.tolist() == [0, 0]
    for f, t in zip(FIELDS, (cov, var, axes, center, extent)):
        g = getattr(got, f)
        assert g.dtype == torch.float64 and g.is_cuda and _bits_equal(g.cpu().numpy(), t.cpu().numpy()), f
    D = k << level
    c = comp.cpu().numpy()
    if j is None:
        j, on = lattice_index(xyz.cpu().numpy(), k, level)
        assert on.all()
    n, S, SS = osh.moments(j, c, K, weight)
    ref_cov = osh.covariance(n, S, SS, D)
    assert _bits_equal(got.covariance.cpu().numpy(), ref_cov)
    ref_var, ref_axes = osh.principal_axes(ref_cov)
    _check_eigen(got.variance.cpu().numpy(), got.axes.cpu().numpy(), ref_var, ref_axes, ref_cov)
    dev_axes = got.axes.cpu().numpy()
    lo, hi, ref_center, ref_extent = osh.box(j, c, K, dev_axes, D)
    keys = acc.cpu().numpy().view(np.uint64)
    empty = np.array(n) == 0
    assert _bits_equal(np.where(empty[:, None], np.nan, osh.from_key(keys[:, 16:19])), lo)
    assert _bits_equal(np.where(empty[:, None], np.nan, osh.from_key(keys[:, 19:22])), hi)
    assert _bits_equal(got.center.cpu().numpy(), ref_center)
    assert _bits_equal(got.extent.cpu().numpy(), ref_extent)
    return got


def _objects(pts, k, level, Ci, Cs, min_points=1):
    from pagnerf_b200.mapping import instance_components
    comps = instance_components(pts, samples_per_axis=k, level=level, num_instances=Ci, num_classes=Cs, min_points=min_points)
    return comps.component, int(comps.count.numel())


@pytest.mark.parametrize("seed,level,k,fill", [(0, 4, 2, 0.35), (1, 4, 2, 0.35), (2, 3, 3, 0.5), (3, 5, 2, 0.2)])
def test_matches_oracle_on_synthetic_maps(cuda_lib, seed, level, k, fill):
    pts, Ci, Cs = _synthetic(seed, level=level, k=k, fill=fill)
    comp, K = _objects(pts, k, level, Ci, Cs)
    assert K > 3
    _check(pts.xyz, k, level, comp, K)


# Objects of two point clusters each, on the D = 2^18 lattice (k = 8, level 15): m1 copies of j1 and m2 of j2 = j1 - delta, so
# num_ab = m1 m2 delta_a delta_b.  Object 0 holds 2^28 + 2^26 + 1 points near the far corner: its sums S_ab pass 2^64.  The deltas
# of objects 1-4 were searched so that a numerator lies exactly half-way between two f64 values with an odd / even last bit
# (rounds up / down) and one unit above / below such a half-way point; object 4's delta mixes signs (a negative numerator).
BIG_M1 = (1 << 28) + (1 << 26) + 1
SMALL_M1 = (1 << 20) + 1
CLUSTERS = [(BIG_M1, (5852, 6671, 170275)), (SMALL_M1, (250619, 226259, 248468)), (SMALL_M1, (222575, 14825, 24009)),
            (SMALL_M1, (22249, 94650, 219022)), (SMALL_M1, (-44325, 192931, 212065))]


def _rounding_class(num):
    num = abs(num)
    t = num.bit_length() - 53
    if t <= 0:
        return "exact"
    rem, half = num & ((1 << t) - 1), 1 << (t - 1)
    return {half: "tie_up" if (num >> t) & 1 else "tie_down", half + 1: "above", half - 1: "below"}.get(rem, "other")


def test_sums_past_2_64_and_rounding_ties(cuda_lib):
    k, level = 8, 15
    D = k << level
    js, comps, weights = [], [], []
    for o, (m1, delta) in enumerate(CLUSTERS):
        j1 = np.array([0 if d < 0 else D - 1 for d in delta])
        js += [j1, j1 - np.array(delta)]
        comps += [o, o]
        weights += [m1, 3]
    j, comp, w = np.array(js), np.array(comps), np.array(weights)
    assert ((j >= 0) & (j < D)).all()
    K = len(CLUSTERS)
    n, S, SS = osh.moments(j, comp, K, w)
    assert max(max(s) for s in SS) >= 1 << 64                          # the carry words are used
    classes = {_rounding_class(n[o] * SS[o][p] - S[o][a] * S[o][b]) for o in range(K) for p, (a, b) in enumerate(osh.PAIRS)}
    assert {"tie_up", "tie_down", "above", "below"} <= classes
    assert any(n[o] * SS[o][p] < S[o][a] * S[o][b] for o in range(K) for p, (a, b) in enumerate(osh.PAIRS))
    reps = _t(w, torch.int64)
    xyz = torch.repeat_interleave(_t(_coords(j, D)), reps, dim=0)
    c = torch.repeat_interleave(_t(comp, torch.int64), reps)
    assert xyz.shape[0] == sum(weights) <= 1 << 30
    # the oracle works on the distinct points with their multiplicities (the box does not depend on repeats)
    from pagnerf_b200 import ops
    got = _run(xyz, k, level, c, K)
    ref_cov = osh.covariance(n, S, SS, D)
    assert _bits_equal(got.covariance.cpu().numpy(), ref_cov)
    ref_var, ref_axes = osh.principal_axes(ref_cov)
    _check_eigen(got.variance.cpu().numpy(), got.axes.cpu().numpy(), ref_var, ref_axes, ref_cov)
    *_, acc, _ = ops.map_shape(xyz, level, k, c, K)
    acc = acc.cpu().numpy().view(np.uint64)
    assert acc[:, 0].tolist() == n
    assert [[int(acc[o, 4 + p]) + (int(acc[o, 10 + p]) << 64) for p in range(6)] for o in range(K)] == SS
    _, _, center, extent = osh.box(j, comp, K, got.axes.cpu().numpy(), D)
    assert _bits_equal(got.center.cpu().numpy(), center) and _bits_equal(got.extent.cpu().numpy(), extent)
    del xyz, c


def test_lattice_balls_get_world_axes_and_exact_extent(cuda_lib):
    """components_bench.fruit_map: balls of radius 4, each symmetric under axis reflections and permutations, so the covariance is
    exactly diagonal with equal entries: the axes are the world axes and the box is the 9-cell cube around the centre"""
    from tools.components_bench import fruit_map
    k, level = 2, 6
    D = k << level
    pts, n_balls = fruit_map(60000, k, level)
    comp, K = _objects(pts, k, level, 200, 6)
    assert K == n_balls > 100
    got = _check(pts.xyz, k, level, comp, K)
    cov = got.covariance.cpu().numpy()
    assert (cov[:, ~np.eye(3, dtype=bool)] == 0).all()
    assert (cov[:, 0, 0] == cov[:, 1, 1]).all() and (cov[:, 1, 1] == cov[:, 2, 2]).all()
    assert (got.axes.cpu().numpy() == np.eye(3)).all()
    assert (got.extent.cpu().numpy() == 9 * 2.0 / D).all()
    cen = torch.zeros(K, 3, dtype=torch.float64, device=DEV).index_add_(0, comp, pts.xyz.double()) / 257
    assert torch.allclose(got.center, cen, rtol=0, atol=1e-12)


def test_axis_aligned_boxes_get_exact_sides(cuda_lib):
    """Solid boxes of distinct sides in every axis order: diagonal covariance, so the axes are the world axes sorted by side
    (the longest first; axes[2] = axes[0] x axes[1]) and the extents are the sides in cells, exactly"""
    k, level = 2, 5
    D = k << level
    sides = [(9, 5, 3), (3, 9, 5), (5, 3, 9), (11, 7, 4), (4, 11, 7), (7, 4, 11)]
    js, comp = [], []
    for o, s in enumerate(sides):
        origin = np.array([(o % 3) * 20 + 2, (o // 3) * 20 + 2, 5 + o])
        js.append(np.argwhere(np.ones(s, bool)) + origin)
        comp += [o] * int(np.prod(s))
    got = _check(_t(_coords(np.concatenate(js), D)), k, level, _t(comp, torch.int64), len(sides))
    for o, s in enumerate(sides):
        order = np.argsort(-np.array(s), kind="stable")
        e0, e1 = np.eye(3)[order[0]], np.eye(3)[order[1]]
        assert np.array_equal(got.axes[o].cpu().numpy(), np.stack([e0, e1, np.cross(e0, e1)])), o
        assert np.array_equal(got.extent[o].cpu().numpy(), np.array(s, np.float64)[order] * 2.0 / D), o
        assert (got.variance[o, :-1] > got.variance[o, 1:]).all()


def _rotation(rng):
    q = rng.normal(size=4)
    q /= np.linalg.norm(q)
    w, x, y, z = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def test_planted_rotated_boxes_and_ellipsoids(cuda_lib):
    """Solid boxes (half sides h) and ellipsoids (semi-axes h) with random rotations R and unequal axes, sampled on the lattice.

    Tolerances, from lattice quantisation:
      * Axes.  The ideal covariance is A = R diag(s) R^T, s = h^2 / 3 (box) or h^2 / 5 (ellipsoid), in lattice units.  The lattice
        sample's covariance is A + E, and E is computed here from the oracle's exact covariance.  By Weyl and the Davis-Kahan sin
        theta theorem, the angle between recovered axis a and R's column a obeys sin theta_a <= ||E|| / (gap_a - ||E||), gap_a =
        the distance of s_a to the other s.
      * Extents.  Every point of space lies within sqrt(3)/2 of a lattice point.  The ball of radius sqrt(3)/2 centred sqrt(3)/2
        inside the shape's tip along axis a lies inside the shape (the other half sides, and the ellipsoid's radii of curvature at
        its tips, exceed sqrt(3)/2), so some lattice point inside projects within sqrt(3) of the tip: along the true axis hi - lo
        lies in [2 h_a - 2 sqrt(3), 2 h_a], and the extent in cells in [2 h_a + 1 - 2 sqrt(3), 2 h_a + 1].  Along the recovered axis
        every projection moves by at most |e - u| rho <= sqrt(2) sin theta rho, rho = the largest distance of a point from the
        centre, which widens the interval by 2 sqrt(2) sin theta rho on each side.
      * Centre.  Along each true axis the box's midpoint lies within sqrt(3)/2 of the shape's centre, and within sqrt(2) sin theta
        rho more along the recovered axis: |centre - c| <= sqrt(3) (sqrt(3)/2 + sqrt(2) max sin theta rho) cells."""
    k, level = 2, 6
    D = k << level
    rng = np.random.default_rng(11)
    shapes = [("box", (20.0, 12.0, 6.0)), ("box", (26.0, 9.0, 4.5)), ("ellipsoid", (24.0, 14.0, 8.0)), ("ellipsoid", (22.0, 12.0, 6.5))]
    js, comp, planted = [], [], []
    for o, (kind, h) in enumerate(shapes):
        R = _rotation(rng)
        c = np.array([32.0, 32.0, 32.0]) + (0.5 * (o % 2), 0.25 * o, 0.0) + ((o % 2) * 64, (o // 2) * 64, 0)
        r = int(np.ceil(np.linalg.norm(h))) + 1
        g = np.stack(np.meshgrid(*[np.arange(-r, r + 1)] * 3, indexing="ij"), -1).reshape(-1, 3) + np.floor(c).astype(np.int64)
        u = (g - c) @ R                                              # coordinates along R's columns
        inside = (np.abs(u) <= h).all(1) if kind == "box" else ((u / h) ** 2).sum(1) <= 1
        js.append(g[inside])
        comp += [o] * int(inside.sum())
        planted.append((kind, np.array(h), R, c, g[inside]))
    j = np.concatenate(js)
    assert ((j >= 0) & (j < D)).all()
    got = _check(_t(_coords(j, D)), k, level, _t(comp, torch.int64), len(shapes))
    n, S, SS = osh.moments(j, np.array(comp), len(shapes))
    lattice_cov = osh.covariance(n, S, SS, D) * (D * D / 4.0)
    axes, extent, center = got.axes.cpu().numpy(), got.extent.cpu().numpy() * D / 2.0, got.center.cpu().numpy()
    for o, (kind, h, R, c, pts) in enumerate(planted):
        s = h ** 2 / (3.0 if kind == "box" else 5.0)
        E = lattice_cov[o] - R @ np.diag(s) @ R.T
        normE = np.linalg.norm(E, 2)
        rho = np.linalg.norm(pts - c, axis=1).max()
        sins = []
        for a in range(3):
            gap = min(abs(s[a] - s[b]) for b in range(3) if b != a)
            assert gap > 2 * normE, (o, a, gap, normE)
            sin = normE / (gap - normE)
            sins.append(sin)
            assert abs(axes[o, a] @ R[:, a]) >= np.sqrt(1 - sin ** 2) - 1e-12, (o, a)
            widen = 2 * np.sqrt(2) * sin * rho
            assert 2 * h[a] + 1 - 2 * np.sqrt(3) - widen <= extent[o, a] <= 2 * h[a] + 1 + widen, (o, a, extent[o, a])
        centre_cells = (center[o] + 1.0) * D / 2.0 - 0.5
        assert np.linalg.norm(centre_cells - c) <= np.sqrt(3) * (np.sqrt(3) / 2 + np.sqrt(2) * max(sins) * rho), o


def test_order_relabelling_and_repeats_change_nothing(cuda_lib):
    pts, Ci, Cs = _synthetic(5, fill=0.5)
    comp, K = _objects(pts, 2, 4, Ci, Cs, min_points=3)
    ref = _run(pts.xyz, 2, 4, comp, K)
    again = _run(pts.xyz, 2, 4, comp, K)
    assert all(_bits_equal(getattr(ref, f).cpu().numpy(), getattr(again, f).cpu().numpy()) for f in FIELDS)
    perm = torch.randperm(pts.xyz.shape[0], generator=torch.Generator().manual_seed(0)).to(DEV)
    shuf = _run(pts.xyz[perm], 2, 4, comp[perm], K)
    assert all(_bits_equal(getattr(ref, f).cpu().numpy(), getattr(shuf, f).cpu().numpy()) for f in FIELDS)
    relabel = torch.randperm(K, generator=torch.Generator().manual_seed(1)).to(DEV)
    comp2 = torch.where(comp >= 0, relabel[comp.clamp(min=0)], comp)
    rel = _run(pts.xyz, 2, 4, comp2, K)
    for f in FIELDS:
        assert _bits_equal(getattr(rel, f)[relabel].cpu().numpy(), getattr(ref, f).cpu().numpy()), f


def test_edge_cases(cuda_lib):
    k, level = 2, 3
    D = k << level
    empty = _run(_t(np.zeros((0, 3))), k, level, _t(np.zeros(0), torch.int64), 3)
    for f in FIELDS:
        assert np.isnan(getattr(empty, f).cpu().numpy()).all() and getattr(empty, f).shape[0] == 3, f
    none = _run(_t(_coords([[1, 2, 3]], D)), k, level, _t([-1], torch.int64), 0)
    assert [tuple(getattr(none, f).shape) for f in FIELDS] == [(0, 3, 3), (0, 3), (0, 3, 3), (0, 3), (0, 3)]
    j = np.array([[1, 2, 3], [4, 6, 3], [7, 7, 7], [9, 1, 14]])
    got = _check(_t(_coords(j, D)), k, level, _t([1, 1, 3, -1], torch.int64), 4)   # objects 0 and 2 empty; 1: two points; 3: one
    for f in FIELDS:
        v = getattr(got, f).cpu().numpy()
        assert np.isnan(v[[0, 2]]).all() and not np.isnan(v[[1, 3]]).any(), f
    assert (got.covariance[3] == 0).all() and (got.axes[3].cpu() == torch.eye(3, dtype=torch.float64)).all()
    assert (got.extent[3] == 2.0 / D).all() and got.center[3].tolist() == ((2 * j[2] + 1) / D - 1).tolist()
    d = (j[1] - j[0]).astype(np.float64)
    assert np.allclose(got.axes[1, 0].cpu().numpy(), d / np.linalg.norm(d), atol=1e-15)
    assert np.allclose(got.extent[1].cpu().numpy(), np.array([np.linalg.norm(d) + 1, 1, 1]) * 2 / D, rtol=1e-14)
    unused = _run(_t(_coords(j, D)), k, level, _t([-1] * 4, torch.int64), 2)
    assert all(np.isnan(getattr(unused, f).cpu().numpy()).all() for f in FIELDS)


def test_errors_raise_with_counts(cuda_lib):
    pts, Ci, Cs = _synthetic(0)
    comp, K = _objects(pts, 2, 4, Ci, Cs)
    xyz = pts.xyz.clone()
    xyz[3, 0] = torch.nextafter(xyz[3, 0], torch.tensor(2.0, device=DEV))
    xyz[10, 2] = 1.5
    with pytest.raises(ValueError, match="^2 points are not on the lattice"):
        _run(xyz, 2, 4, comp, K)
    with pytest.raises(ValueError, match="not on the lattice"):
        _run(pts.xyz, 2, 3, comp, K)                                # the wrong level
    bad = comp.clone()
    bad[[0, 5, 9]] = torch.tensor([K, -2, K + 7], device=DEV)
    with pytest.raises(ValueError, match=f"^3 points carry a component outside \\[-1, {K}\\)"):
        _run(pts.xyz, 2, 4, bad, K)
    with pytest.raises(ValueError, match=f"^{int((comp >= 0).sum())} points carry"):
        _run(pts.xyz, 2, 4, comp, 0)                                # no object at all
    with pytest.raises(RuntimeError, match="CUDA"):
        _run(pts.xyz, 2, 4, comp.cpu(), K)


def test_one_host_read(cuda_lib, monkeypatch):
    pts, Ci, Cs = _synthetic(1)
    comp, K = _objects(pts, 2, 4, Ci, Cs)
    _run(pts.xyz, 2, 4, comp, K)
    reads = []
    for name in ("item", "tolist", "cpu"):
        orig = getattr(torch.Tensor, name)

        def counted(self, *a, _orig=orig, _name=name, **kw):
            if self.is_cuda:
                reads.append(_name)
            return _orig(self, *a, **kw)
        monkeypatch.setattr(torch.Tensor, name, counted)
    got = _run(pts.xyz, 2, 4, comp, K)
    monkeypatch.undo()
    assert len(reads) == 1, reads
    assert got.extent.shape == (K, 3)


def test_memory_within_documented_bound(cuda_lib):
    """Peak allocation growth of a call <= the outputs (216 bytes per object) + SHAPE_WORKSPACE_BYTES per object + 16 bytes"""
    from pagnerf_b200.mapping import panoptic_map
    pts, Ci, Cs = _synthetic(2, level=5, k=2, fill=0.6)
    comp, K = _objects(pts, 2, 5, Ci, Cs)
    _run(pts.xyz, 2, 5, comp, K)
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = _run(pts.xyz, 2, 5, comp, K)
    torch.cuda.synchronize()
    growth = torch.cuda.max_memory_allocated() - base
    assert panoptic_map.SHAPE_WORKSPACE_BYTES == 176
    bound = (216 + panoptic_map.SHAPE_WORKSPACE_BYTES) * K + 16
    assert growth <= bound + 7 * 512, (growth, bound)                # the caching allocator rounds each of 7 tensors to 512 bytes
    del out


@pytest.mark.parametrize("name", ["trace_delta_permuto_ray", "trace_nef_tcnn_ray", "trace_dd_permuto_ray"])
def test_golden_field_map_end_to_end(cuda_lib, name):
    from pagnerf_b200.mapping import extract_panoptic_map, instance_components
    g = load_golden(name)
    nef = build_cuda_nef(g, DEV)
    if "tcnn" in name:
        nef.grid.embedder.round_half = True
    level = int(nef.grid.blas_level)
    for k in (2, 3):
        pts = extract_panoptic_map(nef, k, min_density=-1.0)
        comps = instance_components(pts, samples_per_axis=k, level=level, num_instances=nef.num_instances,
                                    num_classes=nef.num_classes)
        K = int(comps.count.numel())
        assert K > 0
        got = _check(pts.xyz, k, level, comps.component, K)
        assert (got.extent > 0).all()
