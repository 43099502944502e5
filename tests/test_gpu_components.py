"""GPU: objects of a labelled map (pagnerf_b200.mapping.instance_components; csrc/mapping.cu) against the CPU oracle
(oracle/components.py), on known answers, union-find worst cases, error inputs, the golden fields' maps, memory and host reads."""
import numpy as np
import pytest
import torch

from oracle import components as oc
from oracle import mapping as om
from tests.util import load_golden, build_cuda_nef

pytestmark = pytest.mark.gpu
DEV = "cuda"
KEYS_EXACT = ("component", "count", "instance", "category", "votes", "bbox_min", "bbox_max")


def _coords(j, D):
    """lattice indices [P,3] -> xyz f32 [P,3] by the map's point formula"""
    return (2 * np.asarray(j, np.int64) + 1).astype(np.float32) / np.float32(D) - np.float32(1.0)


def _pts(xyz, sem, inst, rgb=None, seed=0):
    from pagnerf_b200.mapping import PanopticPoints
    P = len(xyz)
    g = torch.Generator().manual_seed(seed)
    rgb = torch.rand(P, 3, generator=g) if rgb is None else torch.as_tensor(rgb)
    t = lambda a, dt: torch.as_tensor(np.asarray(a)).to(dt).to(DEV)
    return PanopticPoints(t(xyz, torch.float32).reshape(P, 3), rgb.float().to(DEV), torch.ones(P, device=DEV), t(sem, torch.int64),
                          torch.ones(P, device=DEV), t(inst, torch.int64), torch.ones(P, device=DEV))


def _run(pts, k, level, Ci, Cs, things=None, connectivity=26, min_points=1):
    from pagnerf_b200.mapping import instance_components
    return instance_components(pts, samples_per_axis=k, level=level, num_instances=Ci, num_classes=Cs, things=things,
                               connectivity=connectivity, min_points=min_points)


def _oracle(pts, k, level, Ci, Cs, things=None, connectivity=26, min_points=1):
    return oc.components(pts.xyz.cpu().numpy(), pts.semantic.cpu().numpy(), pts.instance.cpu().numpy(), k, level, things,
                         connectivity, min_points, pts.rgb.cpu().numpy(), Ci, Cs)


def _assert_equal(got, ref):
    assert ref["errors"] == dict(off_lattice=0, duplicates=0, bad_labels=0)
    for key in KEYS_EXACT:
        g = getattr(got, key).cpu().numpy()
        assert g.shape == ref[key].shape and np.array_equal(g, ref[key]), key
    for key in ("centroid", "mean_rgb"):
        g = getattr(got, key)
        assert g.dtype == torch.float64
        assert np.allclose(g.cpu().numpy(), ref[key], rtol=1e-12, atol=1e-15), key


def _synthetic(seed, level=4, k=2, fill=0.35, n_labels=6, Cs=4):
    """A map on the (k, level) lattice in the map's order (by leaf cell, then by sub-point): blocky instance labels (so objects
    span many points) with noise, random classes."""
    rng = np.random.default_rng(seed)
    D = k << level
    block = rng.integers(0, n_labels, (4, 4, 4))
    j = np.argwhere(rng.random((D, D, D)) < fill)
    inst = block[tuple((j * 4 // D).T)]
    noise = rng.random(len(j)) < 0.05
    inst[noise] = rng.integers(0, n_labels, noise.sum())
    sem = rng.integers(0, Cs, len(j))
    cell = j // k
    perm = np.lexsort((j[:, 2], j[:, 1], j[:, 0], cell[:, 2], cell[:, 1], cell[:, 0]))
    return _pts(_coords(j[perm], D), sem[perm], inst[perm], seed=seed), n_labels, Cs


@pytest.mark.parametrize("seed", [0, 1])
@pytest.mark.parametrize("connectivity", [6, 26])
@pytest.mark.parametrize("min_points,things", [(1, None), (5, None), (8, {0, 2}), (1, {3})])
def test_components_match_oracle(cuda_lib, seed, connectivity, min_points, things):
    pts, Ci, Cs = _synthetic(seed)
    got = _run(pts, 2, 4, Ci, Cs, things, connectivity, min_points)
    ref = _oracle(pts, 2, 4, Ci, Cs, things, connectivity, min_points)
    assert len(ref["count"]) > 3
    _assert_equal(got, ref)


def test_planted_fruit(cuda_lib):
    """S separated balls with labels from a pool smaller than S, plus isolated speckle points: exactly S objects, each with its
    ball's label and centre; instance_summary on the same map merges the balls that share a label."""
    from pagnerf_b200.mapping import instance_summary
    rng = np.random.default_rng(7)
    k, level = 2, 5
    D = k << level                                       # 64
    S, pool, r = 27, 5, 3
    centres = np.stack(np.meshgrid(*[np.arange(3)] * 3, indexing="ij"), -1).reshape(-1, 3) * 12 + 6     # spaced 12 > 2r + 1
    labels = rng.integers(0, pool, S)
    labels[:pool] = np.arange(pool)
    off = np.stack(np.meshgrid(*[np.arange(-r, r + 1)] * 3, indexing="ij"), -1).reshape(-1, 3)
    ball = off[(off ** 2).sum(1) <= r * r]
    j = np.concatenate([c + ball for c in centres])
    inst = np.repeat(labels, len(ball))
    speck = np.stack(np.meshgrid(*[np.arange(44, 64, 2)] * 3, indexing="ij"), -1).reshape(-1, 3)     # 2 apart: never adjacent
    speck_inst = rng.integers(0, pool, len(speck))
    j = np.concatenate([j, speck])
    inst = np.concatenate([inst, speck_inst])
    perm = rng.permutation(len(j))
    pts = _pts(_coords(j[perm], D), np.zeros(len(j), np.int64), inst[perm])
    got = _run(pts, k, level, pool, 1, min_points=2)
    assert got.count.numel() == S
    assert (got.count == len(ball)).all()
    want_centre = (2 * centres.astype(np.float64) + 1) / D - 1
    cen = got.centroid.cpu().numpy()
    match = np.argmin(((cen[:, None] - want_centre[None]) ** 2).sum(-1), axis=1)
    assert sorted(match.tolist()) == list(range(S))
    assert np.allclose(cen, want_centre[match], atol=1e-6)
    assert np.array_equal(got.instance.cpu().numpy(), labels[match])
    assert _run(pts, k, level, pool, 1, min_points=1).count.numel() == S + len(speck)
    # what the per-label summary makes of the same map: one row per label, its balls and speckles merged
    summ = instance_summary(pts, pool, 1)
    per_label = np.bincount(labels, minlength=pool)
    assert (per_label > 1).any()
    want_count = per_label * len(ball) + np.bincount(speck_inst, minlength=pool)
    assert np.array_equal(summ.count.cpu().numpy(), want_count)
    ball_span = 2 * r * 2.0 / D
    span = (summ.bbox_max - summ.bbox_min).max(dim=1).values.cpu().numpy()
    assert (span > ball_span + 1e-6).all()                # every row spans more than one ball


def test_six_versus_twenty_six(cuda_lib):
    n = 50
    t = np.arange(n)
    j = np.stack([t, t, t], 1)
    pts = _pts(_coords(j, 64), np.zeros(n, np.int64), np.zeros(n, np.int64))
    assert _run(pts, 2, 5, 1, 1, connectivity=26).count.tolist() == [n]
    six = _run(pts, 2, 5, 1, 1, connectivity=6)
    assert six.count.tolist() == [1] * n and six.component.tolist() == list(range(n))


def _serpentine(rows=64, length=1 << 16):
    """A chain of 2^22 + 63 points: rows along x at y = 0, 2, 4, ..., joined at alternating ends by one point at odd y.  Under
    6-connectivity only consecutive points are adjacent (a path); 26-connectivity adds two diagonal edges at each joint."""
    pts = []
    for r in range(rows):
        x = np.arange(length) if r % 2 == 0 else np.arange(length)[::-1]
        pts.append(np.stack([x, np.full(length, 2 * r), np.zeros(length, np.int64)], 1))
        if r + 1 < rows:
            pts.append(np.array([[x[-1], 2 * r + 1, 0]]))
    return np.concatenate(pts)


@pytest.mark.parametrize("order", ["forward", "reversed", "shuffled"])
def test_long_path_is_one_object(cuda_lib, order):
    j = _serpentine()
    assert len(j) >= 1 << 22
    if order == "reversed":
        j = j[::-1]
    elif order == "shuffled":
        j = j[np.random.default_rng(0).permutation(len(j))]
    k, level = 8, 15                                     # D = 2^18
    P = len(j)
    pts = _pts(_coords(j, k << level), np.zeros(P, np.int64), np.zeros(P, np.int64))
    for conn in (6, 26):
        got = _run(pts, k, level, 1, 1, connectivity=conn)
        assert got.count.tolist() == [P]
        assert bool((got.component == 0).all())


def test_all_distinct_labels(cuda_lib):
    """K = P: every point its own object (labels all different), the statistics in global memory."""
    D = 64
    j = np.argwhere(np.ones((D, D, 25), bool))
    P = len(j)
    pts = _pts(_coords(j, D), np.arange(P) % 3, np.random.default_rng(1).permutation(P))
    got = _run(pts, 2, 5, P, 3)
    assert got.count.numel() == P
    _assert_equal(got, _oracle(pts, 2, 5, P, 3))


def test_instance_summary_many_instances(cuda_lib):
    """instance_summary with more instances than the shared-memory slots hold: the global-memory variant, against the oracle."""
    from pagnerf_b200.mapping import instance_summary
    pts, _, Cs = _synthetic(3, n_labels=6)
    Ci = 5000
    g = torch.Generator().manual_seed(0)
    pts = pts._replace(instance=torch.randint(0, 300, (pts.xyz.shape[0],), generator=g).to(DEV) * 16)
    for things in (None, {1, 2}):
        s = instance_summary(pts, Ci, Cs, things)
        ref = om.summary(pts.xyz.cpu().numpy(), pts.rgb.cpu().numpy(), pts.semantic.cpu().numpy(), pts.instance.cpu().numpy(), Ci, Cs,
                         things)
        for key in ("count", "votes", "category", "bbox_min", "bbox_max"):
            assert np.array_equal(getattr(s, key).cpu().numpy(), ref[key]), key
        n = ref["count"] > 0
        for key in ("centroid", "mean_rgb"):
            assert np.allclose(getattr(s, key).cpu().numpy()[n], ref[key][n], rtol=1e-12, atol=1e-15), key


def test_edge_sizes(cuda_lib):
    for P in (0, 1):
        j = np.zeros((P, 3), np.int64) + 5
        pts = _pts(_coords(j, 16), np.zeros(P, np.int64), np.zeros(P, np.int64))
        got = _run(pts, 2, 3, 1, 1)
        assert got.count.numel() == P and got.component.tolist() == list(range(P))
        assert got.centroid.shape == (P, 3) and got.votes.shape == (P, 1)
    pts, Ci, Cs = _synthetic(0)
    none = _run(pts, 2, 4, Ci, Cs, things=set())
    assert none.count.numel() == 0 and bool((none.component == -1).all())
    big = _run(pts, 2, 4, Ci, Cs, min_points=pts.xyz.shape[0] + 1)
    assert big.count.numel() == 0


def test_deterministic_and_order_free(cuda_lib):
    pts, Ci, Cs = _synthetic(5, fill=0.5)
    a, b = _run(pts, 2, 4, Ci, Cs, min_points=3), _run(pts, 2, 4, Ci, Cs, min_points=3)
    for x, y in zip(a, b):
        assert torch.equal(x, y) or torch.allclose(x, y, rtol=1e-15, atol=0)
    assert torch.equal(a.component, b.component) and torch.equal(a.count, b.count)
    perm = torch.randperm(pts.xyz.shape[0], generator=torch.Generator().manual_seed(0)).to(DEV)
    shuffled = pts._replace(**{f: getattr(pts, f)[perm] for f in pts._fields})
    c = _run(shuffled, 2, 4, Ci, Cs, min_points=3)
    parts = lambda comp, idx: {frozenset(idx[comp == q].tolist()) for q in np.unique(comp[comp >= 0])}
    ia = np.arange(pts.xyz.shape[0])
    assert parts(a.component.cpu().numpy(), ia) == parts(c.component.cpu().numpy(), perm.cpu().numpy())


def test_errors_raise_with_counts(cuda_lib):
    pts, Ci, Cs = _synthetic(0)
    xyz = pts.xyz.clone()
    xyz[3, 0] = torch.nextafter(xyz[3, 0], torch.tensor(2.0, device=DEV))
    xyz[10, 2] = 1.5
    with pytest.raises(ValueError, match="2 points are not on the lattice"):
        _run(pts._replace(xyz=xyz), 2, 4, Ci, Cs)
    with pytest.raises(ValueError, match="not on the lattice"):
        _run(pts, 2, 3, Ci, Cs)                              # the wrong level
    dup = pts._replace(**{f: torch.cat([getattr(pts, f), getattr(pts, f)[:4]]) for f in pts._fields})
    with pytest.raises(ValueError, match="4 points repeat"):
        _run(dup, 2, 4, Ci, Cs)
    sem, inst = pts.semantic.clone(), pts.instance.clone()
    sem[0], inst[1], inst[2] = Cs, -1, Ci
    with pytest.raises(ValueError, match="3 points carry"):
        _run(pts._replace(semantic=sem, instance=inst), 2, 4, Ci, Cs)
    ref = _oracle(pts._replace(semantic=sem, instance=inst), 2, 4, Ci, Cs)
    assert ref["errors"]["bad_labels"] == 3


@pytest.mark.parametrize("name", ["trace_delta_permuto_ray", "trace_nef_tcnn_ray", "trace_dd_permuto_ray"])
def test_golden_field_map_end_to_end(cuda_lib, name):
    from pagnerf_b200.mapping import extract_panoptic_map
    g = load_golden(name)
    nef = build_cuda_nef(g, DEV)
    if "tcnn" in name:
        nef.grid.embedder.round_half = True
    level = int(nef.grid.blas_level)
    for k, things, conn, mp in ((2, None, 26, 1), (3, {4, 5}, 6, 3)):
        pts = extract_panoptic_map(nef, k, min_density=-1.0)
        got = _run(pts, k, level, nef.num_instances, nef.num_classes, things, conn, mp)
        ref = _oracle(pts, k, level, nef.num_instances, nef.num_classes, things, conn, mp)
        assert len(ref["count"]) > 0
        _assert_equal(got, ref)


def test_memory_within_documented_bound(cuda_lib):
    """Peak allocation growth of a call <= 12 C + 24 P bytes (C = smallest power of two >= 2P) + 12 per 1024 points + the
    per-object outputs, (160 + 8 Cs) bytes each."""
    pts, Ci, Cs = _synthetic(2, level=5, k=2, fill=0.6)      # ~157 k points
    _run(pts, 2, 5, Ci, Cs)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    got = _run(pts, 2, 5, Ci, Cs)
    torch.cuda.synchronize()
    P, K = pts.xyz.shape[0], got.count.numel()
    C = 2
    while C < 2 * P:
        C *= 2
    bound = 12 * C + 24 * P + 12 * (P // 1024 + 1) + 8 + (160 + 8 * Cs) * K
    growth = torch.cuda.max_memory_allocated() - base
    assert growth <= bound + (1 << 16), (growth, bound)          # + the caching allocator's 512-byte rounding of a few tensors


def test_one_host_read(cuda_lib, monkeypatch):
    pts, Ci, Cs = _synthetic(1)
    _run(pts, 2, 4, Ci, Cs)
    reads = []
    for name in ("item", "tolist", "cpu"):
        orig = getattr(torch.Tensor, name)

        def counted(self, *a, _orig=orig, _name=name, **kw):
            if self.is_cuda:
                reads.append(_name)
            return _orig(self, *a, **kw)
        monkeypatch.setattr(torch.Tensor, name, counted)
    got = _run(pts, 2, 4, Ci, Cs)
    monkeypatch.undo()
    assert len(reads) == 1, reads
    assert got.count.numel() > 0
