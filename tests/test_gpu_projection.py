"""GPU: projection of a map into camera views (pagnerf_b200.mapping.project_map; csrc/mapping.cu) against the CPU oracle
(oracle/projection.py), batch invariance, the pixel convention, a planted-fruit frame with a known answer, the golden fields' maps,
edge cases, host reads, CUDA-graph capture, determinism and memory."""
import numpy as np
import pytest
import torch

from oracle import projection as op
from tests.util import load_golden, build_cuda_nef

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _coords(j, D):
    return (2 * np.asarray(j, np.int64) + 1).astype(np.float32) / np.float32(D) - np.float32(1.0)


def _lattice_map(seed, k, level, fill):
    """Points on the (k, level) lattice in the map's order (leaf cell, then sub-point) -> xyz f32 [P, 3]"""
    rng = np.random.default_rng(seed)
    D = k << level
    j = np.argwhere(rng.random((D, D, D)) < fill)
    cell = j // k
    perm = np.lexsort((j[:, 2], j[:, 1], j[:, 0], cell[:, 2], cell[:, 1], cell[:, 0]))
    return _coords(j[perm], D)


def _pass_cameras(idx, H, W):
    """Cameras of the synthetic pass (bench.make_cameras) with bench.make_frame_rays' intrinsics scaled to W: f = 0.9 W, c = centre"""
    import bench
    V = bench.make_cameras()[list(idx)]
    K = np.tile(np.array([0.9 * W, 0.9 * W, W / 2, H / 2], np.float32), (len(idx), 1))
    return V, K


def _t(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    return t if dtype is None else t.to(dtype)


def _project(xyz, k, level, V, K, H, W, max_radius, near=0.01, component=None):
    from pagnerf_b200.mapping import project_map
    return project_map(_t(xyz), samples_per_axis=k, level=level, view=_t(V), intrinsics=_t(K), height=H, width=W,
                       max_radius=max_radius, near=near, component=None if component is None else _t(component))


def _equal_oracle(mv, xyz, k, level, V, K, H, W, max_radius, near=0.01, component=None):
    wp, wd, wo = op.project(xyz, k, level, V, K, H, W, max_radius, near, component)
    assert np.array_equal(mv.point.cpu().numpy(), wp)
    assert np.array_equal(mv.depth.cpu().numpy(), wd)
    if component is not None:
        assert np.array_equal(mv.object.cpu().numpy(), wo)
    return wp


@pytest.mark.parametrize("max_radius", [0, 2, 8])
@pytest.mark.parametrize("k,level,fill", [(1, 5, 0.3), (2, 5, 0.15), (4, 4, 0.2)])
def test_projection_matches_oracle(cuda_lib, max_radius, k, level, fill):
    xyz = _lattice_map(k * 10 + level, k, level, fill)
    comp = np.random.default_rng(k).integers(-1, 40, len(xyz))
    V, K = _pass_cameras((0, 20, 41), 120, 160)
    mv = _project(xyz, k, level, V, K, 120, 160, max_radius, component=comp)
    assert mv.point.shape == (3, 120, 160) and mv.point.dtype == torch.int64 and mv.depth.dtype == torch.float32
    wp = _equal_oracle(mv, xyz, k, level, V, K, 120, 160, max_radius, component=comp)
    assert (wp >= 0).mean() > 0.05 and (wp < 0).any()
    plain = _project(xyz, k, level, V, K, 120, 160, max_radius)
    assert plain.object is None and torch.equal(plain.point, mv.point) and torch.equal(plain.depth, mv.depth)


def test_awkward_points_match_oracle(cuda_lib):
    """Duplicates (ties in z and pixel), points behind the camera and at z == near, far off-screen and non-finite points, clamped
    footprints (a long focal length) and a negative focal length, off the lattice."""
    rng = np.random.default_rng(7)
    P = 5000
    x = rng.uniform(-1, 1, (P, 3)).astype(np.float32)
    x[:, 2] = rng.uniform(-1, 0.5, P).astype(np.float32)
    x[100:200] = x[0:100]
    x[200:300, 2] = np.float32(1.5)
    near = 0.0625
    x[300:310, 2] = np.float32(1.0) - np.float32(near)
    x[310] = [1e30, 0, 0]
    x[311] = [0, -1e30, -0.5]
    x[312, 0], x[313, 1], x[314, 2], x[315] = np.nan, np.inf, -np.inf, np.nan
    V = np.tile(np.eye(4, dtype=np.float32), (4, 1, 1))
    V[:, 2, 3] = -1.0
    V[1:, :3, 3] += rng.uniform(-0.2, 0.2, (3, 3)).astype(np.float32)
    K = np.array([[60, 60, 32, 24], [3000, 2500, 30.5, 20.25], [-60, 60, 32, 24], [55, 70, 40.3, 10.7]], np.float32)
    for R in (0, 1, 32):
        mv = _project(x, 2, 3, V, K, 48, 64, R, near=near, component=np.arange(P) % 7 - 1)
        wp = _equal_oracle(mv, x, 2, 3, V, K, 48, 64, R, near=near, component=np.arange(P) % 7 - 1)
        assert (wp[2] == -1).all() and (wp[0] >= 0).any()
        assert not np.isin(wp, np.r_[100:200, 200:300, 310:316]).any() and not np.isin(wp[0], np.r_[300:310]).any()


def test_batch_invariance(cuda_lib):
    xyz = _lattice_map(3, 2, 5, 0.2)
    V, K = _pass_cameras(range(0, 42, 6), 96, 128)
    comp = np.arange(len(xyz)) % 11 - 1
    all_ = _project(xyz, 2, 5, V, K, 96, 128, 4, component=comp)
    for b in range(len(V)):
        one = _project(xyz, 2, 5, V[b:b + 1], K[b:b + 1], 96, 128, 4, component=comp)
        assert torch.equal(one.point[0], all_.point[b]) and torch.equal(one.depth[0], all_.depth[b])
        assert torch.equal(one.object[0], all_.object[b])


def test_pixel_convention(cuda_lib):
    """With max_radius = 0 each isolated point, kept away from pixel borders, lands on the pixel whose centre ray (the
    bench.make_frame_rays formula) meets the plane at the point's camera depth nearest to the point."""
    res, f = 128, 0.9 * 128
    cam = np.array([0.1, -0.05, 0.9])
    V = np.eye(4, dtype=np.float32)[None].copy()
    V[0, :3, 3] = -cam
    K = np.array([[f, f, res / 2, res / 2]], np.float32)
    rng = np.random.default_rng(11)
    n = 500
    flat = rng.choice(res * res, n, replace=False)
    r, c = flat // res, flat % res
    fu, fv = rng.uniform(0.1, 0.9, n), rng.uniform(0.1, 0.9, n)
    zc = rng.uniform(0.3, 1.5, n)
    d = np.stack([(c + fu - res / 2) / f, (r + fv - res / 2) / f, -np.ones(n)], 1)
    x = (cam + d * zc[:, None]).astype(np.float32)
    mv = _project(x, 2, 7, V, K, res, res, 0)
    point = mv.point[0].cpu().numpy()
    assert (point >= 0).sum() == n
    assert np.array_equal(point[r, c], np.arange(n))
    # the nearest centre ray at the point's depth: pixel centres (c' + 0.5, r' + 0.5) map to cam + ((c' + 0.5 - res/2) / f) zc ...
    cc = np.floor((x[:, 0] - cam[0]) / zc * f + res / 2).astype(int)
    rr = np.floor((x[:, 1] - cam[1]) / zc * f + res / 2).astype(int)
    assert np.array_equal(cc, c) and np.array_equal(rr, r)
    assert np.allclose(mv.depth[0].cpu().numpy()[r, c], zc, rtol=1e-5)


def _planted_scene():
    """Nine lattice balls (radius R = 4, class 1) at one depth, spaced 12 apart, and a ground slab (class 2, stuff) behind them; the
    balls at x = 20 and x = 44 share instance label 0 and mirror each other about the camera axis."""
    k, level = 2, 5
    D = k << level
    R = 4
    cs = [20, 32, 44]
    centres = np.array([(x, y, 24) for y in cs for x in cs])
    labels = np.array([1, 2, 3, 0, 4, 0, 5, 6, 7])
    off = np.stack(np.meshgrid(*[np.arange(-R, R + 1)] * 3, indexing="ij"), -1).reshape(-1, 3)
    ball = off[(off ** 2).sum(1) <= R * R]
    jb = np.concatenate([c + ball for c in centres])
    slab = np.stack(np.meshgrid(np.arange(D), np.arange(D), [2], indexing="ij"), -1).reshape(-1, 3)
    j = np.concatenate([jb, slab])
    sem = np.concatenate([np.ones(len(jb), np.int64), np.full(len(slab), 2)])
    inst = np.concatenate([np.repeat(labels, len(ball)), np.zeros(len(slab), np.int64)])
    perm = np.random.default_rng(0).permutation(len(j))
    centre_point = np.argsort(perm)[np.arange(len(centres)) * len(ball) + np.nonzero((ball == 0).all(1))[0][0]]
    return dict(k=k, level=level, D=D, R=R, centres=centres, labels=labels, j=j[perm], sem=sem[perm], inst=inst[perm],
                centre_point=centre_point)


def _render_analytic(s, rho, res=160):
    """Pinhole frame from above the middle ball, looking down -z: per pixel the first hit of the analytic spheres (radius rho
    lattice units around the ball centres) and of the slab's plane -> origins, dirs, depth, alpha (1 on hits, 0 on misses) and
    the ground-truth (ball id, or -1 slab, or -2 miss)."""
    D = s["D"]
    w = lambda j: (2.0 * np.asarray(j, np.float64) + 1.0) / D - 1.0
    cam = np.array([w(32), w(32), 0.9], np.float32)
    ys, xs = np.meshgrid(np.arange(res) + 0.5, np.arange(res) + 0.5, indexing="ij")
    f = 0.7 * res
    d = np.stack([(xs - res / 2) / f, (ys - res / 2) / f, -np.ones_like(xs)], -1).reshape(-1, 3)
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    o = np.tile(cam, (len(d), 1))
    o64, d64 = o.astype(np.float64), d.astype(np.float64)
    best = np.full(len(d), np.inf)
    gt = np.full(len(d), -2)
    a = (d64 * d64).sum(1)
    for b, c in enumerate(s["centres"]):
        oc = o64 - w(c)
        bb = (d64 * oc).sum(1)
        cc = (oc * oc).sum(1) - (2.0 * rho / D) ** 2
        disc = bb * bb - a * cc
        t = np.where(disc >= 0, (-bb - np.sqrt(np.maximum(disc, 0))) / a, np.inf)
        hit = (t > 0) & (t < best)
        best, gt = np.where(hit, t, best), np.where(hit, b, gt)
    zp = w(2)
    t = (zp - o64[:, 2]) / d64[:, 2]
    p = o64 + d64 * t[:, None]
    on = (t > 0) & (np.abs(p[:, 0]) <= 0.98) & (np.abs(p[:, 1]) <= 0.98) & (t < best)
    best, gt = np.where(on, t, best), np.where(on, -1, gt)
    hit = gt > -2
    depth = np.where(hit, best, 0.0).astype(np.float32)
    return o, d, depth, hit.astype(np.float32), gt


def _analytic_camera(s, res=160):
    """The camera of _render_analytic as view / intrinsics"""
    D = s["D"]
    w = (2.0 * 32 + 1.0) / D - 1.0
    V = np.eye(4, dtype=np.float32)[None].copy()
    V[0, :3, 3] = -np.array([w, w, 0.9], np.float32)
    K = np.array([[0.7 * res, 0.7 * res, res / 2, res / 2]], np.float32)
    return V, K


def test_planted_fruit_projects_to_its_objects(cuda_lib):
    """All nine balls are visible as their own objects, each ball's projected pixels overlap its analytic disc with IoU > 0.3,
    (category, object + 1) scores tp = 9 on the thing class, and on the pixels where both routes see an object the projection agrees
    with lookup_rays on the analytic render.

    Why 0.3: the camera is 1.13 world units above the balls' centres (z = 0.9 against the lattice plane j = 24) with f = 112 px, so
    one lattice unit (2 / D = 1/32) spans about 3.1 px.  The map's ball is the union of the cells (half-size 1/2 unit) of the lattice
    points with |j - c| <= 4, so its outline lies within sqrt(3)/2 units (2.7 px) of the sphere of radius 4.5; the square footprints
    cover whole pixels (up to 1 px more).  Both silhouettes therefore lie within w = 3.7 px of the analytic circle of radius
    r = 4.5 units = 14 px (the balls' tops, up to 4 units nearer, are magnified by at most 4 %, which the px figures round up), and
    IoU >= ((r - w) / (r + w))^2 = (10.3 / 17.7)^2 = 0.34.
    Agreement with lookup_rays: on the rho = 3 render every ball pixel resolves to its ball (tests/test_gpu_lookup.py); those pixels
    lie inside the projected balls, at least 1.5 units from their outline, so the two routes agree on at least 95 % of them (all of
    them in the CPU oracles)."""
    from pagnerf_b200.mapping import PanopticPoints, instance_components, lookup_rays, map_index, project_map
    from pagnerf_b200.metrics import PanopticQuality
    s = _planted_scene()
    P = len(s["j"])
    one = torch.ones(P, device=DEV)
    pts = PanopticPoints(_t(_coords(s["j"], s["D"])), torch.rand(P, 3, device=DEV), one, _t(s["sem"], torch.int64), one,
                         _t(s["inst"], torch.int64), one)
    comps = instance_components(pts, samples_per_axis=s["k"], level=s["level"], num_instances=8, num_classes=3, things={1})
    assert comps.count.numel() == 9
    obj_of_ball = comps.component.cpu().numpy()[s["centre_point"]]
    V, K = _analytic_camera(s)
    res = 160
    mv = project_map(pts, samples_per_axis=s["k"], level=s["level"], view=_t(V), intrinsics=_t(K), height=res, width=res, max_radius=8,
                     component=comps.component)
    _equal_oracle(mv, pts.xyz.cpu().numpy(), s["k"], s["level"], V, K, res, res, 8, component=comps.component.cpu().numpy())
    point, obj = mv.point[0].cpu().numpy().reshape(-1), mv.object[0].cpu().numpy().reshape(-1)
    assert sorted(set(obj[obj >= 0].tolist())) == list(range(9))
    _, _, _, _, gt45 = _render_analytic(s, rho=4.5)
    for b in range(9):
        a, m = obj == obj_of_ball[b], gt45 == b
        assert (a & m).sum() / (a | m).sum() > 0.3, b
    # panoptic quality against the rho = 4.5 analytic frame: background (miss) = stuff 0, slab = stuff 2, balls = thing 1
    sem = pts.semantic.cpu().numpy()
    cat = np.where(point >= 0, sem[np.maximum(point, 0)], 0)
    ball, slab = gt45 >= 0, gt45 == -1
    target = np.stack([np.where(ball, 1, np.where(slab, 2, 0)), np.where(ball, gt45 + 1, 0)], -1).reshape(1, res, res, 2)
    pred = np.stack([cat, obj + 1], -1).reshape(1, res, res, 2)
    m = PanopticQuality(things={1}, stuffs={0, 2}).to(DEV)
    m(_t(pred), _t(target))
    tp = m.stats()[1].cpu().numpy()                   # per category (1, 0, 2)
    assert tp[0] == 9
    # against lookup_rays on the rho = 3 render
    o, d, depth, alpha, gt3 = _render_analytic(s, rho=3.0)
    index = map_index(pts, samples_per_axis=s["k"], level=s["level"])
    hit = lookup_rays(index, _t(o), _t(d), _t(depth), _t(alpha), radius=1, min_alpha=0.5, component=comps.component)
    lo = hit.object.cpu().numpy()
    both = (lo >= 0) & (obj >= 0)
    assert both.sum() > 2000
    assert (lo[both] == obj[both]).mean() >= 0.95


@pytest.mark.parametrize("name", ["trace_delta_permuto_ray", "trace_nef_tcnn_ray", "trace_dd_permuto_ray"])
def test_golden_field_map_projection(cuda_lib, name):
    from pagnerf_b200.mapping import extract_panoptic_map, instance_components, project_map
    g = load_golden(name)
    nef = build_cuda_nef(g, DEV)
    if "tcnn" in name:
        nef.grid.embedder.round_half = True
    level = int(nef.grid.blas_level)
    pts = extract_panoptic_map(nef, 2, min_density=-1.0)
    comps = instance_components(pts, samples_per_axis=2, level=level, num_instances=nef.num_instances, num_classes=nef.num_classes)
    V, K = _pass_cameras((5, 30), 90, 120)
    for R in (1, 8):
        mv = project_map(pts, samples_per_axis=2, level=level, view=_t(V), intrinsics=_t(K), height=90, width=120, max_radius=R,
                         component=comps.component)
        wp = _equal_oracle(mv, pts.xyz.cpu().numpy(), 2, level, V, K, 90, 120, R, component=comps.component.cpu().numpy())
        assert (wp >= 0).any()


def test_empty_map_and_points_behind(cuda_lib):
    V, K = _pass_cameras((0, 1), 32, 48)
    mv = _project(np.zeros((0, 3), np.float32), 2, 3, V, K, 32, 48, 8, component=np.zeros(0, np.int64))
    assert (mv.point == -1).all() and torch.isinf(mv.depth).all() and (mv.object == -1).all()
    behind = np.random.default_rng(0).uniform(-1, 1, (1000, 3)).astype(np.float32)
    behind[:, 2] = np.float32(0.95)                                                    # cameras at z = 0.9, looking down -z
    mv = _project(behind, 2, 3, V, K, 32, 48, 8, component=np.zeros(1000, np.int64))
    assert (mv.point == -1).all() and torch.isinf(mv.depth).all() and (mv.object == -1).all()


def _count_host_reads(monkeypatch):
    reads = []
    for name in ("item", "tolist", "cpu", "numpy", "__bool__", "__int__", "__float__"):
        orig = getattr(torch.Tensor, name)

        def counted(self, *a, _orig=orig, _name=name, **kw):
            if self.is_cuda:
                reads.append(_name)
            return _orig(self, *a, **kw)
        monkeypatch.setattr(torch.Tensor, name, counted)
    return reads


def test_no_host_read_and_graph_replay(cuda_lib, monkeypatch):
    from pagnerf_b200.mapping import project_map
    xyz = _t(_lattice_map(5, 2, 5, 0.2))
    comp = _t(np.arange(xyz.shape[0]) % 9 - 1)
    V, K = (_t(a) for a in _pass_cameras((3, 17, 33), 64, 80))
    run = lambda v: project_map(xyz, samples_per_axis=2, level=5, view=v, intrinsics=K, height=64, width=80, max_radius=4,
                                component=comp)
    run(V)
    torch.cuda.synchronize()
    reads = _count_host_reads(monkeypatch)
    torch.cuda.set_sync_debug_mode("error")
    try:
        run(V)
        project_map(xyz, samples_per_axis=2, level=5, view=V, intrinsics=K, height=64, width=80, max_radius=0)
    finally:
        torch.cuda.set_sync_debug_mode(0)
        monkeypatch.undo()
    assert reads == []
    static_v = V.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run(static_v)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = run(static_v)
    V2 = V.clone()
    V2[:, 0, 3] += 0.1
    static_v.copy_(V2)
    graph.replay()
    torch.cuda.synchronize()
    eager = run(V2)
    assert torch.equal(out.point, eager.point) and torch.equal(out.depth, eager.depth) and torch.equal(out.object, eager.object)
    assert not torch.equal(eager.point, run(V).point)


def test_deterministic_and_memory(cuda_lib):
    from pagnerf_b200.mapping import project_map
    xyz = _t(_lattice_map(6, 4, 5, 0.1))                   # ~ 0.2 M points, overlapping footprints
    comp = _t(np.arange(xyz.shape[0]) % 13 - 1)
    B, H, W = 4, 256, 320
    V, K = (_t(a) for a in _pass_cameras((0, 10, 20, 30), H, W))
    run = lambda c: project_map(xyz, samples_per_axis=4, level=5, view=V, intrinsics=K, height=H, width=W, max_radius=8, component=c)
    a, b = run(comp), run(comp)
    assert torch.equal(a.point, b.point) and torch.equal(a.depth, b.depth) and torch.equal(a.object, b.object)
    for c, per_pixel, n_alloc in ((comp, 28, 4), (None, 20, 3)):
        run(c)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        out = run(c)
        torch.cuda.synchronize()
        growth = torch.cuda.max_memory_allocated() - base
        assert per_pixel * B * H * W <= growth <= per_pixel * B * H * W + n_alloc * 512, (growth, per_pixel * B * H * W)
        del out
