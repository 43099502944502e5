"""CPU: the map-object oracle (oracle/components.py) against scipy.ndimage.label on dense lattices, its lattice recovery against
oracle.mapping.cell_points, argument validation of pagnerf_b200.mapping.instance_components and the PLY writer's component column."""
import numpy as np
import pytest
import torch
from hypothesis import given, settings, strategies as st
from scipy import ndimage

from oracle import components as oc
from oracle import mapping as om


def _dense_map(n, occ):
    """One point per occupied voxel of an n^3 grid, in raster order -> (xyz, voxel index [P,3]).  Voxel v of an axis is sub-point
    v % k of cell v // k, so its coordinate is cell_points' fl(fl((2v+1)/n) - 1)."""
    ijk = np.argwhere(occ)
    return (2 * ijk + 1).astype(np.float32) / np.float32(n) - np.float32(1.0), ijk


@settings(max_examples=60, deadline=None)
@given(level=st.integers(1, 3), k=st.integers(1, 2), fill=st.floats(0.1, 0.9), n_labels=st.integers(1, 4), Cs=st.integers(1, 3),
       connectivity=st.sampled_from([6, 26]), use_things=st.booleans(), seed=st.integers(0, 2 ** 31 - 1))
def test_oracle_matches_ndimage_label(level, k, fill, n_labels, Cs, connectivity, use_things, seed):
    rng = np.random.default_rng(seed)
    n = k << level
    occ = rng.random((n, n, n)) < fill
    inst_grid = rng.integers(0, n_labels, (n, n, n))
    sem_grid = rng.integers(0, Cs, (n, n, n))
    things = set(rng.choice(Cs, size=rng.integers(0, Cs + 1), replace=False).tolist()) if use_things else None
    xyz, ijk = _dense_map(n, occ)
    perm = rng.permutation(len(xyz))                   # point order is arbitrary
    xyz, ijk = xyz[perm], ijk[perm]
    inst = inst_grid[tuple(ijk.T)]
    sem = sem_grid[tuple(ijk.T)]
    rgb = rng.random((len(xyz), 3)).astype(np.float32)
    got = oc.components(xyz, sem, inst, k, level, things, connectivity, 1, rgb, n_labels, Cs)
    assert got["errors"] == dict(off_lattice=0, duplicates=0, bad_labels=0)
    tm = np.zeros(Cs, bool)
    tm[list(things) if things is not None else slice(None)] = True
    active_grid = occ & tm[sem_grid]
    structure = ndimage.generate_binary_structure(3, 1 if connectivity == 6 else 3)
    # the same partition: per instance label, ndimage's components are exactly the oracle's objects of that label
    want_parts = set()
    for q in range(n_labels):
        lab, nl = ndimage.label(active_grid & (inst_grid == q), structure=structure)
        at = lab[tuple(ijk.T)]
        for c in range(1, nl + 1):
            want_parts.add(frozenset(np.nonzero(at == c)[0].tolist()))
    comp = got["component"]
    got_parts = {frozenset(np.nonzero(comp == c)[0].tolist()) for c in range(len(got["count"]))}
    assert got_parts == want_parts
    active = active_grid[tuple(ijk.T)]
    assert ((comp >= 0) == active).all()
    # numbering by smallest point index, counts and the shared instance label
    first = [np.nonzero(comp == c)[0].min() for c in range(len(got["count"]))]
    assert first == sorted(first)
    assert np.array_equal(got["count"], np.bincount(comp[comp >= 0], minlength=len(got["count"])))
    for c in range(len(got["count"])):
        assert (inst[comp == c] == got["instance"][c]).all()


@settings(max_examples=20, deadline=None)
@given(level=st.integers(1, 3), min_points=st.integers(1, 6), seed=st.integers(0, 2 ** 31 - 1))
def test_oracle_min_points_drops_small_objects(level, min_points, seed):
    rng = np.random.default_rng(seed)
    n = 1 << level
    occ = rng.random((n, n, n)) < 0.3
    xyz, ijk = _dense_map(n, occ)
    inst = rng.integers(0, 2, len(xyz))
    sem = np.zeros(len(xyz), np.int64)
    rgb = np.zeros((len(xyz), 3), np.float32)
    every = oc.components(xyz, sem, inst, 1, level, None, 26, 1, rgb, 2, 1)
    some = oc.components(xyz, sem, inst, 1, level, None, 26, min_points, rgb, 2, 1)
    keep = every["count"] >= min_points
    assert np.array_equal(some["count"], every["count"][keep])
    remap = np.full(len(keep), -1)
    remap[keep] = np.arange(keep.sum())
    want = np.where(every["component"] >= 0, remap[np.maximum(every["component"], 0)], -1)
    assert np.array_equal(some["component"], want)


@pytest.mark.parametrize("k", range(1, 9))
@pytest.mark.parametrize("level", [1, 3, 7])
def test_lattice_index_round_trips_cell_points(k, level):
    n = 1 << level
    rng = np.random.default_rng(k * 100 + level)
    cells = np.unique(np.concatenate([rng.integers(0, n, (6, 3)), [[0, 0, 0], [n - 1, n - 1, n - 1]]]), axis=0)
    xyz = om.cell_points(cells, level, k)
    j, on = oc.lattice_index(xyz, k, level)
    assert on.all()
    sub = np.stack(np.meshgrid(np.arange(k), np.arange(k), np.arange(k), indexing="ij"), -1).reshape(-1, 3)
    assert np.array_equal(j, (cells[:, None, :] * k + sub[None]).reshape(-1, 3))
    # one ulp off on one axis: off the lattice
    for direction in (np.inf, -np.inf):
        bumped = xyz.copy()
        bumped[:, 1] = np.nextafter(bumped[:, 1], np.float32(direction))
        assert not oc.lattice_index(bumped, k, level)[1].any()
    # outside [-1, 1] and NaN: off
    assert not oc.lattice_index(xyz[:1] * 0 + np.float32(2.0), k, level)[1].any()
    assert not oc.lattice_index(np.full((1, 3), np.nan, np.float32), k, level)[1].any()
    # duplicates: counted once per repeated point
    dup = np.concatenate([xyz, xyz[:3]])
    P = len(dup)
    res = oc.components(dup, np.zeros(P, np.int64), np.zeros(P, np.int64), k, level, None, 26, 1, np.zeros((P, 3), np.float32), 1, 1)
    assert res["errors"] == dict(off_lattice=0, duplicates=3, bad_labels=0)


def test_oracle_error_counts():
    xyz = om.cell_points(np.array([[0, 0, 0], [1, 1, 1]]), 2, 2)
    P = len(xyz)
    sem, inst = np.zeros(P, np.int64), np.zeros(P, np.int64)
    xyz[0, 0] = np.nextafter(xyz[0, 0], np.float32(1))
    sem[1], inst[2], inst[3] = 3, -1, 5
    res = oc.components(xyz, sem, inst, 2, 2, None, 26, 1, np.zeros((P, 3), np.float32), 5, 3)
    assert res["errors"] == dict(off_lattice=1, duplicates=0, bad_labels=3)


def _points(P, seed=0):
    from pagnerf_b200.mapping import PanopticPoints
    g = torch.Generator().manual_seed(seed)
    return PanopticPoints(torch.rand(P, 3, generator=g) * 2 - 1, torch.rand(P, 3, generator=g), torch.rand(P, generator=g) * 10,
                          torch.randint(0, 6, (P,), generator=g), torch.rand(P, generator=g),
                          torch.randint(0, 200, (P,), generator=g), torch.rand(P, generator=g))


@pytest.mark.parametrize("kwargs,match", [
    (dict(samples_per_axis=0), "samples_per_axis"), (dict(samples_per_axis=9), "samples_per_axis"),
    (dict(samples_per_axis=2.0), "samples_per_axis"), (dict(samples_per_axis=True), "samples_per_axis"),
    (dict(level=-1), "level"), (dict(level=16), "level"), (dict(level=3.0), "level"),
    (dict(connectivity=8), "connectivity"), (dict(connectivity=True), "connectivity"), (dict(connectivity="26"), "connectivity"),
    (dict(min_points=0), "min_points"), (dict(min_points=1.5), "min_points"),
    (dict(things={6}), "things"), (dict(num_classes=33), "num_classes"), (dict(num_instances=0), "num_instances")])
def test_instance_components_argument_validation(kwargs, match):
    from pagnerf_b200.mapping import instance_components
    args = dict(samples_per_axis=2, level=3, num_instances=200, num_classes=6)
    args.update(kwargs)
    with pytest.raises(ValueError, match=match):
        instance_components(_points(10), **args)


def test_instance_components_refuses_cpu_tensors():
    from pagnerf_b200.mapping import instance_components
    with pytest.raises(RuntimeError, match="CUDA"):
        instance_components(_points(10), samples_per_axis=2, level=3, num_instances=200, num_classes=6)


@pytest.mark.parametrize("P", [0, 1, 1000])
def test_write_ply_component_column(tmp_path, P):
    from pagnerf_b200.mapping import write_ply
    pts = _points(P, P)
    plain, with_comp = tmp_path / "a.ply", tmp_path / "b.ply"
    write_ply(str(plain), pts)
    write_ply(str(plain.with_suffix(".none")), pts, component=None)
    assert plain.read_bytes() == plain.with_suffix(".none").read_bytes()
    comp = torch.randint(-1, 50, (P,), generator=torch.Generator().manual_seed(P))
    write_ply(str(with_comp), pts, component=comp)
    raw_a, raw_b = plain.read_bytes(), with_comp.read_bytes()
    ha, hb = raw_a.index(b"end_header\n") + 11, raw_b.index(b"end_header\n") + 11
    assert raw_b[:hb] == raw_a[:ha].replace(b"property float instance_score\n", b"property float instance_score\nproperty int component\n")
    rec_a = np.frombuffer(raw_a[ha:], dtype=np.dtype([("v", "V35")]))
    rec_b = np.frombuffer(raw_b[hb:], dtype=np.dtype([("v", "V35"), ("component", "<i4")]))
    assert len(rec_b) == P and rec_a.tobytes() == rec_b["v"].tobytes()
    assert np.array_equal(rec_b["component"], comp.numpy())
    with pytest.raises(ValueError, match="component"):
        write_ply(str(with_comp), pts, component=comp[:-1] if P else torch.zeros(1, dtype=torch.int64))
