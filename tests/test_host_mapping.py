"""CPU: the point-map oracle (oracle/mapping.py) against direct constructions -- sub-cell coordinates and their order, the per-instance
summary on hypothesis-generated labels --, the PLY writer of pagnerf_b200.mapping and its argument validation."""
import numpy as np
import pytest
import torch
from hypothesis import given, settings, strategies as st

from oracle import mapping as om
from tests.util import load_golden, build_cuda_nef


@pytest.mark.parametrize("k", [1, 2, 3, 8])
@pytest.mark.parametrize("level", [1, 4, 7])
def test_cell_points_coordinates_and_order(k, level):
    n = 1 << level
    rng = np.random.default_rng(k * 10 + level)
    cells = np.concatenate([rng.integers(0, n, (5, 3)), [[0, 0, 0], [n - 1, n - 1, n - 1], [n - 1, 0, n - 1]]]).astype(np.int16)
    got = om.cell_points(cells, level, k)
    assert got.dtype == np.float32 and got.shape == (len(cells) * k ** 3, 3)
    want = []
    for p in cells.tolist():
        for ix in range(k):
            for iy in range(k):
                for iz in range(k):
                    want.append([np.float32(2 * (c * k + i) + 1) / np.float32(k * n) - np.float32(1.0) for c, i in zip(p, (ix, iy, iz))])
    want = np.array(want, dtype=np.float32)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    # sub-cell centres: strictly inside their cell, the far corner's last centre at 1 - 1/(k 2^L)
    lo = cells.astype(np.float64).repeat(k ** 3, 0) / n * 2 - 1
    assert (got > lo).all() and (got < lo + 2.0 / n).all()
    assert np.allclose(got[(len(cells) - 1) * k ** 3 - 1], 1 - 1 / (k * n), rtol=0, atol=1e-7)


def _vector_summary(xyz, rgb, sem, inst, Ci, Cs, things):
    """Independent restatement with numpy scatter operations."""
    ok = (sem >= 0) & (sem < Cs) & (inst >= 0) & (inst < Ci)
    errors = int((~ok).sum())
    tm = np.zeros(Cs, bool)
    tm[list(things) if things is not None else slice(None)] = True
    sel = ok.copy()
    sel[ok] = tm[sem[ok]]
    q, s = inst[sel], sem[sel]
    count = np.bincount(q, minlength=Ci).astype(np.int64)
    sum_xyz, sum_rgb = np.zeros((Ci, 3)), np.zeros((Ci, 3))
    np.add.at(sum_xyz, q, xyz[sel].astype(np.float64))
    np.add.at(sum_rgb, q, rgb[sel].astype(np.float64))
    bmin, bmax = np.full((Ci, 3), np.inf, np.float32), np.full((Ci, 3), -np.inf, np.float32)
    np.minimum.at(bmin, q, xyz[sel])
    np.maximum.at(bmax, q, xyz[sel])
    votes = np.zeros((Ci, Cs), np.int64)
    np.add.at(votes, (q, s), 1)
    category = np.where(count > 0, votes.argmax(1), -1)
    return dict(count=count, sum_xyz=sum_xyz, sum_rgb=sum_rgb, bbox_min=bmin, bbox_max=bmax, votes=votes, category=category, errors=errors)


@settings(max_examples=40, deadline=None)
@given(P=st.integers(0, 300), Ci=st.integers(1, 12), Cs=st.integers(1, 6), seed=st.integers(0, 2 ** 31 - 1),
       use_things=st.booleans(), bad=st.booleans())
def test_oracle_summary_against_vectorised(P, Ci, Cs, seed, use_things, bad):
    rng = np.random.default_rng(seed)
    xyz = rng.uniform(-1, 1, (P, 3)).astype(np.float32)
    rgb = rng.uniform(0, 1, (P, 3)).astype(np.float32)
    sem = rng.integers(0, Cs, P)
    inst = rng.integers(0, Ci, P)
    if bad and P:
        sem[rng.integers(0, P, 3)] = Cs
        inst[rng.integers(0, P, 2)] = -1
    things = set(rng.choice(Cs, size=rng.integers(0, Cs + 1), replace=False).tolist()) if use_things else None
    got = om.summary(xyz, rgb, sem, inst, Ci, Cs, things)
    want = _vector_summary(xyz, rgb, sem, inst, Ci, Cs, things)
    assert got["errors"] == want["errors"]
    for key in ("count", "votes", "category", "bbox_min", "bbox_max"):
        assert np.array_equal(got[key], want[key]), key
    for key in ("sum_xyz", "sum_rgb"):
        assert np.allclose(got[key], want[key], rtol=1e-12, atol=1e-12), key
    n = want["count"] > 0
    assert np.allclose(got["centroid"][n], want["sum_xyz"][n] / want["count"][n, None], rtol=1e-12)
    assert np.isnan(got["centroid"][~n]).all()


def _points(P, seed=0):
    from pagnerf_b200.mapping import PanopticPoints
    g = torch.Generator().manual_seed(seed)
    return PanopticPoints(torch.rand(P, 3, generator=g) * 2 - 1, torch.rand(P, 3, generator=g), torch.rand(P, generator=g) * 10,
                          torch.randint(0, 6, (P,), generator=g), torch.rand(P, generator=g),
                          torch.randint(0, 200, (P,), generator=g), torch.rand(P, generator=g))


@pytest.mark.parametrize("P", [0, 1, 1000])
def test_write_ply_round_trip(tmp_path, P):
    from pagnerf_b200.mapping import write_ply
    pts = _points(P, P)
    path = tmp_path / "map.ply"
    write_ply(str(path), pts)
    raw = path.read_bytes()
    header = ("ply\nformat binary_little_endian 1.0\nelement vertex %d\n"
              "property float x\nproperty float y\nproperty float z\n"
              "property uchar red\nproperty uchar green\nproperty uchar blue\n"
              "property float density\nproperty int semantic\nproperty float semantic_score\n"
              "property int instance\nproperty float instance_score\nend_header\n") % P
    assert raw[:len(header)] == header.encode("ascii")
    dt = np.dtype([("x", "<f4"), ("y", "<f4"), ("z", "<f4"), ("red", "u1"), ("green", "u1"), ("blue", "u1"), ("density", "<f4"),
                   ("semantic", "<i4"), ("semantic_score", "<f4"), ("instance", "<i4"), ("instance_score", "<f4")])
    assert len(raw) == len(header) + P * dt.itemsize == len(header) + P * 35
    rec = np.frombuffer(raw[len(header):], dtype=dt)
    assert np.array_equal(np.stack([rec["x"], rec["y"], rec["z"]], 1), pts.xyz.numpy())
    rgb8 = np.rint(np.clip(pts.rgb.numpy().astype(np.float64), 0, 1) * 255).astype(np.uint8)
    assert np.array_equal(np.stack([rec["red"], rec["green"], rec["blue"]], 1), rgb8)
    assert np.array_equal(rec["density"], pts.density.numpy())
    assert np.array_equal(rec["semantic"], pts.semantic.numpy()) and np.array_equal(rec["instance"], pts.instance.numpy())
    assert np.array_equal(rec["semantic_score"], pts.semantic_score.numpy())
    assert np.array_equal(rec["instance_score"], pts.instance_score.numpy())


@pytest.fixture(scope="module")
def cpu_nef():
    return build_cuda_nef(load_golden("trace_delta_permuto_ray"), "cpu")


@pytest.mark.parametrize("k", [0, 9, -1, 2.0, True])
def test_extract_rejects_samples_per_axis(cpu_nef, k):
    from pagnerf_b200.mapping import extract_panoptic_map
    with pytest.raises(ValueError, match="samples_per_axis"):
        extract_panoptic_map(cpu_nef, samples_per_axis=k)


@pytest.mark.parametrize("attr,value,match", [("sem_sigmoid", True, "sigmoid"), ("inst_normalize", True, "normalize"),
                                              ("sem_detach", False, "detached"), ("num_instances", 300, "instances"),
                                              ("num_classes", 17, "classes"), ("effective_feature_dim", 50, "feature width"),
                                              ("panoptic_features_type", "position", "panoptic_features_type")])
def test_extract_rejects_unsupported_fields(cpu_nef, attr, value, match):
    from pagnerf_b200.mapping import extract_panoptic_map
    old = getattr(cpu_nef, attr)
    setattr(cpu_nef, attr, value)
    try:
        with pytest.raises(NotImplementedError, match=match):
            extract_panoptic_map(cpu_nef)
    finally:
        setattr(cpu_nef, attr, old)


def test_extract_refuses_cpu_field(cpu_nef):
    from pagnerf_b200.mapping import extract_panoptic_map
    with pytest.raises(RuntimeError, match="CUDA"):
        extract_panoptic_map(cpu_nef)


def test_instance_summary_argument_validation():
    from pagnerf_b200.mapping import instance_summary
    pts = _points(10)
    with pytest.raises(ValueError, match="things"):
        instance_summary(pts, 200, 6, things={6})
    with pytest.raises(ValueError, match="num_classes"):
        instance_summary(pts, 200, 33)
    with pytest.raises(RuntimeError, match="CUDA"):
        instance_summary(pts, 200, 6)


def test_fused_panoptic_ok_unchanged_for_dd_field():
    """The shared shape helper serves the DD field for map export, but its fused render path stays off."""
    nef = build_cuda_nef(load_golden("trace_dd_permuto_ray"), "cpu")
    assert nef._fused_heads_unsupported() is None
    with torch.no_grad():
        assert nef.fused_panoptic_ok({'semantics', 'inst_embedding'}) is False
