"""GPU: per-object visibility of a map in camera views (pagnerf_b200.mapping.object_visibility; csrc/mapping.cu) against the CPU
oracle (oracle/visibility.py) and project_map, a planted-fruit scene with an occluder, silhouette rounds, camera-split invariance,
edge cases, out-of-range components, the golden fields' maps and memory."""
import gc

import numpy as np
import pytest
import torch

from oracle import visibility as ov
from tests.test_gpu_projection import _analytic_camera, _coords, _lattice_map, _pass_cameras, _planted_scene, _t
from tests.util import load_golden, build_cuda_nef

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(autouse=True)
def _collect_device_garbage():
    """Free device tensors held in reference cycles (the tracebacks of the ValueError tests hold the call's frames) when each test
    ends, so they are not freed inside a later test's peak-memory window"""
    yield
    gc.collect()


def _objects(xyz, k, level, seed, n_labels=8):
    """instance_components of the map with random instance labels, every point a thing -> (component i64 [P] on the device, K)"""
    from pagnerf_b200.mapping import PanopticPoints, instance_components
    P = len(xyz)
    one = torch.ones(P, device=DEV)
    inst = _t(np.random.default_rng(seed).integers(0, n_labels, P), torch.int64)
    pts = PanopticPoints(_t(xyz), torch.rand(P, 3, device=DEV), one, torch.zeros(P, dtype=torch.int64, device=DEV), one, inst, one)
    comps = instance_components(pts, samples_per_axis=k, level=level, num_instances=n_labels, num_classes=1, min_points=3)
    return comps.component, int(comps.count.numel())


def _visibility(xyz, k, level, V, K, H, W, comp, n_obj, max_radius, near=0.01):
    from pagnerf_b200.mapping import object_visibility
    return object_visibility(_t(xyz), samples_per_axis=k, level=level, view=_t(V), intrinsics=_t(K), height=H, width=W,
                             component=comp if isinstance(comp, torch.Tensor) else _t(comp), num_objects=n_obj, max_radius=max_radius,
                             near=near)


def _equal_oracle(vis, xyz, k, level, V, K, H, W, comp, n_obj, max_radius, near=0.01):
    c = comp.cpu().numpy() if isinstance(comp, torch.Tensor) else comp
    wv, ws, wb = ov.visibility(xyz, k, level, V, K, H, W, c, n_obj, max_radius, near)
    assert np.array_equal(vis.visible.cpu().numpy(), wv)
    assert np.array_equal(vis.silhouette.cpu().numpy(), ws)
    assert np.array_equal(vis.bbox.cpu().numpy(), wb)
    return wv, ws


def _equal(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("max_radius", [0, 2, 8])
@pytest.mark.parametrize("k,level,fill", [(1, 5, 0.3), (2, 5, 0.15), (4, 4, 0.2)])
def test_visibility_matches_oracle_and_projection(cuda_lib, max_radius, k, level, fill):
    from pagnerf_b200.mapping import project_map
    xyz = _lattice_map(k * 10 + level, k, level, fill)
    comp, n_obj = _objects(xyz, k, level, seed=k)
    V, K = _pass_cameras((0, 20, 41), 120, 160)
    vis = _visibility(xyz, k, level, V, K, 120, 160, comp, n_obj, max_radius)
    assert vis.visible.shape == (3, n_obj) and vis.visible.dtype == torch.int64 and vis.silhouette.dtype == torch.int64
    assert vis.bbox.shape == (3, n_obj, 4) and vis.bbox.dtype == torch.int32
    wv, ws = _equal_oracle(vis, xyz, k, level, V, K, 120, 160, comp, n_obj, max_radius)
    assert n_obj > 10 and (wv > 0).any() and (wv < ws).any()
    mv = project_map(_t(xyz), samples_per_axis=k, level=level, view=_t(V), intrinsics=_t(K), height=120, width=160,
                     max_radius=max_radius, component=comp)
    for b in range(3):
        o = mv.object[b].reshape(-1)
        assert torch.equal(vis.visible[b], torch.bincount(o[o >= 0], minlength=n_obj))
    assert (vis.visible <= vis.silhouette).all()


def _occluded_scene():
    """The planted nine-ball scene of the projection tests plus a stuff slab (class 2) at lattice z = 32, between the camera and the
    balls, over x in [10, 24] and y in [10, 54]: it hides parts of the three balls at x = 20 and none of the others."""
    s = _planted_scene()
    occ = np.stack(np.meshgrid(np.arange(10, 25), np.arange(10, 55), [32], indexing="ij"), -1).reshape(-1, 3)
    s["j"] = np.concatenate([s["j"], occ])
    s["sem"] = np.concatenate([s["sem"], np.full(len(occ), 2)])
    s["inst"] = np.concatenate([s["inst"], np.zeros(len(occ), np.int64)])
    return s


def test_planted_fruit_with_an_occluder(cuda_lib):
    """Free balls have visible == silhouette; the three balls behind the slab have visible < silhouette; every ball's silhouette
    lies within the analytic bound of its disc.

    The bound, as in tests/test_gpu_projection.py: the camera is 1.13 world units above the balls' centres with f = 112 px, so one
    lattice unit spans about 3.1 px.  The map's ball is the union of the cells of the lattice points with |j - c| <= 4, whose
    outline lies within sqrt(3)/2 units (2.7 px) of the sphere of radius 4.5 units = 14 px; the square footprints cover whole
    pixels (up to 1 px more); the tops, up to 4 units nearer, are magnified by at most 4 %, which the px figures round up.  So the
    silhouette lies between the circles of radius r - w and r + w, r = 14 px, w = 3.7 px: pi (r - w)^2 <= silhouette <= pi (r + w)^2.
    The silhouette ignores occluders, so the bound holds for the hidden balls too."""
    from pagnerf_b200.mapping import PanopticPoints, instance_components, object_visibility, project_map
    s = _occluded_scene()
    P = len(s["j"])
    one = torch.ones(P, device=DEV)
    pts = PanopticPoints(_t(_coords(s["j"], s["D"])), torch.rand(P, 3, device=DEV), one, _t(s["sem"], torch.int64), one,
                         _t(s["inst"], torch.int64), one)
    comps = instance_components(pts, samples_per_axis=s["k"], level=s["level"], num_instances=8, num_classes=3, things={1})
    assert comps.count.numel() == 9
    obj_of_ball = comps.component.cpu().numpy()[s["centre_point"]]
    V, K = _analytic_camera(s)
    res = 160
    vis = object_visibility(pts, samples_per_axis=s["k"], level=s["level"], view=_t(V), intrinsics=_t(K), height=res, width=res,
                            component=comps.component, num_objects=9, max_radius=8)
    _equal_oracle(vis, pts.xyz.cpu().numpy(), s["k"], s["level"], V, K, res, res, comps.component, 9, 8)
    visible, sil = vis.visible[0].cpu().numpy(), vis.silhouette[0].cpu().numpy()
    r, w = 14.0, 3.7
    hidden = s["centres"][:, 0] == 20
    for b in range(9):
        o = obj_of_ball[b]
        assert np.pi * (r - w) ** 2 <= sil[o] <= np.pi * (r + w) ** 2, (b, sil[o])
        if hidden[b]:
            assert visible[o] < sil[o], b
        else:
            assert visible[o] == sil[o], b
    mv = project_map(pts, samples_per_axis=s["k"], level=s["level"], view=_t(V), intrinsics=_t(K), height=res, width=res, max_radius=8,
                     component=comps.component)
    assert int(vis.visible.sum()) == int((mv.object >= 0).sum())
    for o in range(9):           # the box of the visible pixels
        rows, cols = torch.nonzero(mv.object[0] == o, as_tuple=True)
        want = [int(cols.min()), int(rows.min()), int(cols.max()), int(rows.max())] if visible[o] else [-1] * 4
        assert vis.bbox[0, o].tolist() == want


def test_rounds_give_identical_results(cuda_lib, monkeypatch):
    from pagnerf_b200 import ops
    from pagnerf_b200.mapping import panoptic_map
    xyz = _lattice_map(3, 2, 5, 0.2)
    comp, n_obj = _objects(xyz, 2, 5, seed=3)
    V, K = _pass_cameras(range(0, 42, 6), 96, 128)
    ref = _visibility(xyz, 2, 5, V, K, 96, 128, comp, n_obj, 4)
    _, _, _, bad, total = ops.map_visibility(_t(xyz), _t(V), _t(K), 96, 128, float(np.float32(1 / 64)), float(np.float32(0.01)), 4,
                                             comp, n_obj, panoptic_map.VISIBILITY_BITMAP_BYTES)
    cap = 4 * (total // 8 + 96 * 4)                                   # windows of total / 8 words
    words, rounds = ops.silhouette_bitmap_words(total, 96, 128, cap)
    assert bad == 0 and rounds >= 8 and words < total
    monkeypatch.setattr(panoptic_map, "VISIBILITY_BITMAP_BYTES", cap)
    assert _equal(_visibility(xyz, 2, 5, V, K, 96, 128, comp, n_obj, 4), ref)
    cap = 4 * (96 * 4 + max(1, total // 40))                          # about 40 rounds, each wider than a bitmap by a little
    assert ops.silhouette_bitmap_words(total, 96, 128, cap)[1] >= 40
    monkeypatch.setattr(panoptic_map, "VISIBILITY_BITMAP_BYTES", cap)
    assert _equal(_visibility(xyz, 2, 5, V, K, 96, 128, comp, n_obj, 4), ref)


def test_camera_split_invariance_and_determinism(cuda_lib):
    xyz = _lattice_map(4, 2, 5, 0.2)
    comp, n_obj = _objects(xyz, 2, 5, seed=4)
    V, K = _pass_cameras(range(1, 42, 5), 96, 128)
    all_ = _visibility(xyz, 2, 5, V, K, 96, 128, comp, n_obj, 6)
    assert _equal(all_, _visibility(xyz, 2, 5, V, K, 96, 128, comp, n_obj, 6))
    parts = [_visibility(xyz, 2, 5, V[a:a + n], K[a:a + n], 96, 128, comp, n_obj, 6) for a, n in ((0, 1), (1, 3), (4, 5))]
    for field in range(3):
        assert torch.equal(torch.cat([p[field] for p in parts]), all_[field])


def test_empty_map_no_objects_points_behind_and_an_empty_view(cuda_lib):
    V, K = _pass_cameras((0, 1), 32, 48)
    vis = _visibility(np.zeros((0, 3), np.float32), 2, 3, V, K, 32, 48, np.zeros(0, np.int64), 4, 8)
    assert (vis.visible == 0).all() and (vis.silhouette == 0).all() and (vis.bbox == -1).all() and vis.bbox.shape == (2, 4, 4)
    xyz = _lattice_map(5, 2, 4, 0.2)
    vis = _visibility(xyz, 2, 4, V, K, 32, 48, np.full(len(xyz), -1), 0, 8)
    assert vis.visible.shape == (2, 0) and vis.silhouette.shape == (2, 0) and vis.bbox.shape == (2, 0, 4)
    vis = _visibility(xyz, 2, 4, V[:0], K[:0], 32, 48, np.arange(len(xyz)) % 3, 3, 8)
    assert vis.visible.shape == (0, 3) and vis.bbox.shape == (0, 3, 4)
    behind = np.random.default_rng(0).uniform(-1, 1, (1000, 3)).astype(np.float32)
    behind[:, 2] = np.float32(0.95)                                   # cameras at z = 0.9, looking down -z
    vis = _visibility(behind, 2, 3, V, K, 32, 48, np.arange(1000) % 5, 5, 8)
    assert (vis.visible == 0).all() and (vis.silhouette == 0).all() and (vis.bbox == -1).all()
    # view 1 has a negative focal length: it covers nothing, view 0 is unaffected
    comp, n_obj = _objects(xyz, 2, 4, seed=5)
    K2 = K.copy()
    K2[1, 0] = -K2[1, 0]
    vis = _visibility(xyz, 2, 4, V, K2, 32, 48, comp, n_obj, 8)
    _equal_oracle(vis, xyz, 2, 4, V, K2, 32, 48, comp, n_obj, 8)
    assert (vis.visible[1] == 0).all() and (vis.silhouette[1] == 0).all() and (vis.bbox[1] == -1).all() and (vis.visible[0] > 0).any()


def test_out_of_range_components_raise(cuda_lib):
    xyz = _lattice_map(6, 2, 4, 0.2)
    V, K = _pass_cameras((0, 1), 32, 48)
    comp = np.arange(len(xyz)) % 4 - 1
    comp[[3, 50, 700]] = 4
    comp[[10, 11]] = -2
    with pytest.raises(ValueError, match="^5 points carry a component outside \\[-1, 4\\)"):
        _visibility(xyz, 2, 4, V, K, 32, 48, comp, 4, 8)
    with pytest.raises(ValueError, match="^5 points"):                  # counted without cameras too
        _visibility(xyz, 2, 4, V[:0], K[:0], 32, 48, comp, 4, 8)
    with pytest.raises(ValueError, match=f"^{(comp >= 0).sum() + 2} points"):      # no object at all
        _visibility(xyz, 2, 4, V, K, 32, 48, comp, 0, 8)


@pytest.mark.parametrize("name", ["trace_delta_permuto_ray", "trace_nef_tcnn_ray", "trace_dd_permuto_ray"])
def test_golden_field_map_visibility(cuda_lib, name):
    from pagnerf_b200.mapping import extract_panoptic_map, instance_components, object_visibility
    g = load_golden(name)
    nef = build_cuda_nef(g, DEV)
    if "tcnn" in name:
        nef.grid.embedder.round_half = True
    level = int(nef.grid.blas_level)
    pts = extract_panoptic_map(nef, 2, min_density=-1.0)
    comps = instance_components(pts, samples_per_axis=2, level=level, num_instances=nef.num_instances, num_classes=nef.num_classes)
    n_obj = int(comps.count.numel())
    V, K = _pass_cameras((5, 30), 90, 120)
    for R in (1, 8):
        vis = object_visibility(pts, samples_per_axis=2, level=level, view=_t(V), intrinsics=_t(K), height=90, width=120,
                                component=comps.component, num_objects=n_obj, max_radius=R)
        wv, _ = _equal_oracle(vis, pts.xyz.cpu().numpy(), 2, level, V, K, 90, 120, comps.component, n_obj, R)
        assert (wv > 0).any()


def test_memory_bound(cuda_lib):
    from pagnerf_b200 import ops
    from pagnerf_b200.mapping import object_visibility, panoptic_map
    xyz = _t(_lattice_map(6, 4, 5, 0.1))                              # ~ 0.2 M points, overlapping footprints
    comp, n_obj = _objects(xyz.cpu().numpy(), 4, 5, seed=6)
    B, H, W = 4, 256, 320
    V, K = (_t(a) for a in _pass_cameras((0, 10, 20, 30), H, W))
    run = lambda: object_visibility(xyz, samples_per_axis=4, level=5, view=V, intrinsics=K, height=H, width=W, component=comp,
                                    num_objects=n_obj, max_radius=8)
    *_, total = ops.map_visibility(xyz, V, K, H, W, float(np.float32(1 / 128)), float(np.float32(0.01)), 8, comp, n_obj,
                                   panoptic_map.VISIBILITY_BITMAP_BYTES)
    run()
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = run()
    torch.cuda.synchronize()
    growth = torch.cuda.max_memory_allocated() - base
    N = B * n_obj
    bound = 8 * B * H * W + 60 * N + 16 + min(4 * total, panoptic_map.VISIBILITY_BITMAP_BYTES) + 8 * 512
    assert 8 * B * H * W <= growth <= bound, (growth, bound)
    del out
