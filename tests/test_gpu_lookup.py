"""GPU: lookups of 3-D points and rendered pixels into a map's objects (pagnerf_b200.mapping.map_index / lookup_points / lookup_rays;
csrc/mapping.cu) against the CPU oracle (oracle/lookup.py), on a planted-fruit frame with a known answer and its panoptic quality,
on the golden fields' renders, and for errors, host reads, CUDA-graph capture, determinism and memory."""
import numpy as np
import pytest
import torch

from oracle import lookup as ol
from tests.util import load_golden, build_cuda_nef

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _coords(j, D):
    return (2 * np.asarray(j, np.int64) + 1).astype(np.float32) / np.float32(D) - np.float32(1.0)


def _pts(xyz, sem, inst):
    from pagnerf_b200.mapping import PanopticPoints
    P = len(xyz)
    t = lambda a, dt: torch.as_tensor(np.asarray(a)).to(dt).to(DEV)
    one = torch.ones(P, device=DEV)
    return PanopticPoints(t(xyz, torch.float32).reshape(P, 3), torch.rand(P, 3, generator=torch.Generator().manual_seed(P)).to(DEV), one,
                          t(sem, torch.int64), one, t(inst, torch.int64), one)


def _synthetic(seed, level=5, k=2, fill=0.3, n_labels=6, Cs=3):
    """A map on the (k, level) lattice in the map's order (leaf cell, then sub-point) with blocky instance labels, and its objects."""
    from pagnerf_b200.mapping import instance_components
    rng = np.random.default_rng(seed)
    D = k << level
    j = np.argwhere(rng.random((D, D, D)) < fill)
    block = rng.integers(0, n_labels, (4, 4, 4))
    inst = block[tuple((j * 4 // D).T)]
    sem = rng.integers(0, Cs, len(j))
    cell = j // k
    perm = np.lexsort((j[:, 2], j[:, 1], j[:, 0], cell[:, 2], cell[:, 1], cell[:, 0]))
    pts = _pts(_coords(j[perm], D), sem[perm], inst[perm])
    comps = instance_components(pts, samples_per_axis=k, level=level, num_instances=n_labels, num_classes=Cs, things={1, 2}, min_points=4)
    return pts, comps, k, level


def _queries(seed, D, n):
    """n queries: lattice centres, sub-cell faces / edges / corners (t = j + 0.5, ties), points just outside the cube, uniform
    points, NaN and inf."""
    rng = np.random.default_rng(seed)
    f32 = np.float32
    m = n // 5
    j = rng.integers(-2, D + 2, (m, 3))
    centre = (2 * j + 1).astype(f32) / f32(D) - f32(1.0)
    face = (2 * (j + 1)).astype(f32) / f32(D) - f32(1.0)
    mixed = np.where(rng.random((m, 3)) < 0.5, centre, face)
    outside = rng.uniform(-1, 1, (m, 3)).astype(f32)
    axis = rng.integers(0, 3, m)
    outside[np.arange(m), axis] = rng.choice([-1, 1], m) * rng.uniform(1.0, 1.0 + 12.0 / D, m).astype(f32)
    rest = rng.uniform(-1.1, 1.1, (n - 4 * m, 3)).astype(f32)
    rest[:64:4, 0], rest[1:64:4, 1], rest[2:64:4, 2], rest[3:64:4] = np.nan, np.inf, -np.inf, np.nan
    q = np.concatenate([centre, face, mixed, outside, rest]).astype(f32)
    return q[rng.permutation(n)]


def _index(pts, k, level):
    from pagnerf_b200.mapping import map_index
    return map_index(pts, samples_per_axis=k, level=level)


@pytest.mark.parametrize("radius,n", [(0, 1 << 20), (1, 1 << 20), (2, 1 << 19), (4, 1 << 16)])
def test_lookups_match_oracle(cuda_lib, radius, n):
    from pagnerf_b200.mapping import lookup_points, lookup_rays
    pts, comps, k, level = _synthetic(radius)
    D = k << level
    index = _index(pts, k, level)
    idx = ol.index(pts.xyz.cpu().numpy(), k, level)
    comp = comps.component.cpu().numpy()
    q = _queries(radius, D, n)
    want_p, want_o = ol.lookup_points(idx, q, radius, comp)
    assert (want_p >= 0).mean() > 0.1 and (want_p < 0).any() and (want_o >= 0).any()
    got = lookup_points(index, torch.from_numpy(q).to(DEV), radius=radius, component=comps.component)
    assert np.array_equal(got.point.cpu().numpy(), want_p)
    assert np.array_equal(got.object.cpu().numpy(), want_o)
    plain = lookup_points(index, torch.from_numpy(q).to(DEV), radius=radius)
    assert plain.object is None and torch.equal(plain.point, got.point)
    # rays whose surface points spread over the map, alpha on both sides of min_alpha, [N, 1] and [N] depth / alpha
    rng = np.random.default_rng(100 + radius)
    N = n // 2
    o = rng.uniform(-1.5, 1.5, (N, 3)).astype(np.float32)
    d = rng.normal(size=(N, 3)).astype(np.float32)
    depth = rng.uniform(0, 2, N).astype(np.float32)
    alpha = rng.uniform(0, 1.2, N).clip(0, 1).astype(np.float32)
    alpha[:1000], alpha[1000:1100], depth[1100:1200] = 0.5, 0.0, np.inf
    for min_alpha in (0.5, 1.0):
        wp, wo = ol.lookup_rays(idx, o, d, depth, alpha, radius, min_alpha, comp)
        assert (wp >= 0).any()
        t = lambda a: torch.from_numpy(a).to(DEV)
        for shape in ((N, 1), (N,)):
            got = lookup_rays(index, t(o), t(d), t(depth).reshape(shape), t(alpha).reshape(shape), radius=radius, min_alpha=min_alpha,
                              component=comps.component)
            assert np.array_equal(got.point.cpu().numpy(), wp)
            assert np.array_equal(got.object.cpu().numpy(), wo)


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


def test_planted_fruit_pixels_resolve_to_their_objects(cuda_lib):
    """Every pixel that sees a ball resolves to that ball's object, the slab's pixels to a slab point (no object), the misses to -1,
    so (category, object + 1) scores PQ = 1 against the analytic ground truth, while the channel-label image, which merges the two
    balls sharing a label, does not.

    Why this follows from the definitions: the analytic sphere has radius rho = 3 lattice units about the centre c of a lattice
    ball of radius R = 4.  A surface point x has |t - c| = rho (up to fp32 rounding, ~1e-5 units), and the window centre j0 rounds
    each axis of t, so |j0 - t| <= sqrt(3)/2 and |j0 - c| <= 3.87 < R: j0 is a point of the ball and a candidate at radius 1.
    Every candidate lies within Chebyshev distance 1.5 of t, while every point of another ball is more than 12 - R - rho = 5 away and
    the slab lies 22 units below: all candidates belong to this ball.  On the slab's plane t_z = 2 and the window only holds slab
    points."""
    from pagnerf_b200.mapping import instance_components, lookup_rays
    from pagnerf_b200.metrics import PanopticQuality
    s = _planted_scene()
    pts = _pts(_coords(s["j"], s["D"]), s["sem"], s["inst"])
    comps = instance_components(pts, samples_per_axis=s["k"], level=s["level"], num_instances=8, num_classes=3, things={1})
    assert comps.count.numel() == 9
    index = _index(pts, s["k"], s["level"])
    obj_of_ball = comps.component.cpu().numpy()[s["centre_point"]]
    assert sorted(obj_of_ball.tolist()) == list(range(9))
    o, d, depth, alpha, gt = _render_analytic(s, rho=3.0)
    t = lambda a: torch.from_numpy(a).to(DEV)
    hit = lookup_rays(index, t(o), t(d), t(depth)[:, None], t(alpha)[:, None], radius=1, min_alpha=0.5, component=comps.component)
    point, obj = hit.point.cpu().numpy(), hit.object.cpu().numpy()
    ball, slab, miss = gt >= 0, gt == -1, gt == -2
    assert ball.sum() > 2000 and slab.sum() > 2000 and miss.sum() > 0
    assert all((gt == b).sum() > 50 for b in range(9))                  # every ball is in the frame
    assert np.array_equal(obj[ball], obj_of_ball[gt[ball]])
    sem = pts.semantic.cpu().numpy()
    assert (point[slab] >= 0).all() and (sem[point[slab]] == 2).all() and (obj[slab] == -1).all()
    assert (point[miss] == -1).all() and (obj[miss] == -1).all()
    assert np.array_equal(hit.point.cpu().numpy(), ol.lookup_rays(ol.index(pts.xyz.cpu().numpy(), s["k"], s["level"]), o, d, depth,
                                                                   alpha, 1, 0.5)[0])
    # panoptic quality: background (miss) = stuff 0, slab = stuff 2, balls = thing 1
    res = 160
    cat = np.where(point >= 0, sem[np.maximum(point, 0)], 0)
    target = np.stack([np.where(ball, 1, np.where(slab, 2, 0)), np.where(ball, gt + 1, 0)], -1).reshape(1, res, res, 2)
    by_object = np.stack([cat, obj + 1], -1).reshape(1, res, res, 2)
    inst_label = pts.instance.cpu().numpy()
    by_channel = np.stack([cat, np.where(obj >= 0, inst_label[np.maximum(point, 0)] + 1, 0)], -1).reshape(1, res, res, 2)

    def pq(pred):
        m = PanopticQuality(things={1}, stuffs={0, 2}).to(DEV)
        value = float(m(t(pred), t(target)))
        return value, [x.cpu().numpy() for x in m.stats()]      # per category (1, 0, 2): iou_sum, tp, fp, fn

    value, (_, tp, fp, fn) = pq(by_object)
    assert value == 1.0 and tp.tolist() == [9, 1, 1] and fp.sum() == 0 and fn.sum() == 0
    # the two balls of label 0 are mirror images: one segment in the channel image, with IoU about 1/2 with each of them, so at
    # least one of the two balls goes unmatched
    assert abs(int((gt == 3).sum()) - int((gt == 5).sum())) <= 2
    value, (_, tp, fp, fn) = pq(by_channel)
    assert value < 1.0 and tp[0] <= 8 and fn[0] >= 1


@pytest.mark.parametrize("name", ["trace_delta_permuto_ray", "trace_nef_tcnn_ray", "trace_dd_permuto_ray"])
def test_golden_field_render_lookup(cuda_lib, name):
    from pagnerf_b200.mapping import extract_panoptic_map, instance_components, lookup_rays
    from pagnerf_b200.tracers import PanopticPackedRFTracer
    from pagnerf_b200.wisp_compat import Rays
    g = load_golden(name)
    nef = build_cuda_nef(g, DEV)
    if "tcnn" in name:
        nef.grid.embedder.round_half = True
    level = int(nef.grid.blas_level)
    pts = extract_panoptic_map(nef, 2, min_density=-1.0)
    comps = instance_components(pts, samples_per_axis=2, level=level, num_instances=nef.num_instances, num_classes=nef.num_classes)
    index = _index(pts, 2, level)
    tracer = PanopticPackedRFTracer(raymarch_type='ray', num_steps=int(g["num_steps"]), bg_color='white')
    o, d = torch.from_numpy(g["o"]).to(DEV), torch.from_numpy(g["d"]).to(DEV)
    with torch.no_grad():
        rb = tracer(nef, channels=['rgb', 'depth', 'semantics', 'inst_embedding'], rays=Rays(origins=o, dirs=d, dist_min=0.0, dist_max=2.0),
                    lod_idx=None, stage='val')
    depth, alpha = rb.depth.float().contiguous(), rb.alpha.float().contiguous()
    assert (alpha > 0).any()
    min_alpha = float(np.clip(alpha[alpha > 0].quantile(0.25).item(), 1e-6, 1.0))
    idx = ol.index(pts.xyz.cpu().numpy(), 2, level)
    comp = comps.component.cpu().numpy()
    for radius in (1, 2):
        got = lookup_rays(index, o, d, depth, alpha, radius=radius, min_alpha=min_alpha, component=comps.component)
        wp, wo = ol.lookup_rays(idx, g["o"], g["d"], depth.cpu().numpy(), alpha.cpu().numpy(), radius, min_alpha, comp)
        assert np.array_equal(got.point.cpu().numpy(), wp)
        assert np.array_equal(got.object.cpu().numpy(), wo)
    assert (wp >= 0).any()


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


def test_index_errors_and_one_host_read(cuda_lib, monkeypatch):
    pts, _, k, level = _synthetic(1)
    xyz = pts.xyz.clone()
    xyz[3, 0] = torch.nextafter(xyz[3, 0], torch.tensor(2.0, device=DEV))
    xyz[10, 2] = 1.5
    with pytest.raises(ValueError, match="2 points are not on the lattice of samples_per_axis=2, level=5"):
        _index(xyz, k, level)
    with pytest.raises(ValueError, match="not on the lattice"):
        _index(pts, k, level - 1)
    with pytest.raises(ValueError, match="4 points repeat the lattice index of another point"):
        _index(torch.cat([pts.xyz, pts.xyz[:4]]), k, level)
    _index(pts, k, level)
    reads = _count_host_reads(monkeypatch)
    index = _index(pts, k, level)
    monkeypatch.undo()
    assert reads == ["tolist"], reads
    assert index.P == pts.xyz.shape[0] and index.keys.numel() == 2 ** int(np.ceil(np.log2(2 * index.P)))
    assert int((index.keys != 0).sum()) == index.P


def test_lookups_make_no_host_read_and_replay_in_a_graph(cuda_lib, monkeypatch):
    from pagnerf_b200.mapping import lookup_points, lookup_rays
    pts, comps, k, level = _synthetic(2)
    index = _index(pts, k, level)
    D = k << level
    q0, q1 = (torch.from_numpy(_queries(s, D, 1 << 16)).to(DEV) for s in (0, 1))
    N = 1 << 15
    g = torch.Generator(device=DEV).manual_seed(0)
    rays = [torch.rand(N, 3, device=DEV, generator=g) * 2 - 1, torch.randn(N, 3, device=DEV, generator=g),
            torch.rand(N, 1, device=DEV, generator=g) * 2, torch.rand(N, 1, device=DEV, generator=g)]
    lookup_points(index, q0, radius=1, component=comps.component)
    lookup_rays(index, *rays, radius=2, component=comps.component)
    torch.cuda.synchronize()
    reads = _count_host_reads(monkeypatch)
    torch.cuda.set_sync_debug_mode("error")
    try:
        for radius in (0, 1, 4):
            lookup_points(index, q0, radius=radius, component=comps.component)
            lookup_points(index, q0, radius=radius)
            lookup_rays(index, *rays, radius=radius, min_alpha=0.3, component=comps.component)
    finally:
        torch.cuda.set_sync_debug_mode(0)
        monkeypatch.undo()
    assert reads == []
    # capture, then replay on new queries
    static_q = q0.clone()
    static_r = [r.clone() for r in rays]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        lookup_points(index, static_q, radius=1, component=comps.component)
        lookup_rays(index, *static_r, radius=1, component=comps.component)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out_p = lookup_points(index, static_q, radius=1, component=comps.component)
        out_r = lookup_rays(index, *static_r, radius=1, component=comps.component)
    static_q.copy_(q1)
    new_rays = [torch.rand_like(rays[0]) * 2 - 1, torch.randn_like(rays[1]), torch.rand_like(rays[2]) * 2, torch.rand_like(rays[3])]
    for dst, src in zip(static_r, new_rays):
        dst.copy_(src)
    graph.replay()
    torch.cuda.synchronize()
    eager_p = lookup_points(index, q1, radius=1, component=comps.component)
    eager_r = lookup_rays(index, *new_rays, radius=1, component=comps.component)
    assert torch.equal(out_p.point, eager_p.point) and torch.equal(out_p.object, eager_p.object)
    assert torch.equal(out_r.point, eager_r.point) and torch.equal(out_r.object, eager_r.object)
    assert not torch.equal(eager_p.point, lookup_points(index, q0, radius=1).point)


def test_deterministic_and_order_free(cuda_lib):
    from pagnerf_b200.mapping import lookup_points
    pts, comps, k, level = _synthetic(3, fill=0.5)
    index = _index(pts, k, level)
    q = torch.from_numpy(_queries(3, k << level, 1 << 18)).to(DEV)
    for radius in (1, 2):
        a = lookup_points(index, q, radius=radius, component=comps.component)
        b = lookup_points(index, q, radius=radius, component=comps.component)
        assert torch.equal(a.point, b.point) and torch.equal(a.object, b.object)
        perm = torch.randperm(q.shape[0], generator=torch.Generator().manual_seed(radius)).to(DEV)
        c = lookup_points(index, q[perm], radius=radius, component=comps.component)
        assert torch.equal(c.point, a.point[perm]) and torch.equal(c.object, a.object[perm])
    # the index of the same map in another point order resolves every query to a point at the same distance (the same point
    # unless several are equally near: ties go to the smallest index of each order)
    perm = torch.randperm(pts.xyz.shape[0], generator=torch.Generator().manual_seed(9)).to(DEV)
    shuffled = _index(pts.xyz[perm], k, level)
    a = lookup_points(index, q, radius=1).point.cpu().numpy()
    c = lookup_points(shuffled, q, radius=1).point.cpu().numpy()
    hit = a >= 0
    assert np.array_equal(hit, c >= 0)
    D = k << level
    t = ol.query_position(q.cpu().numpy(), D, 1)[0][hit]
    dist = lambda xyz: (((t - ol.query_position(xyz, D, 1)[0]) ** 2).sum(1))
    xa, xc = pts.xyz.cpu().numpy()[a[hit]], pts.xyz[perm].cpu().numpy()[c[hit]]
    assert np.array_equal(dist(xa), dist(xc))
    assert (xa != xc).any(axis=1).mean() < 0.5


def test_memory_is_the_table_and_the_outputs(cuda_lib):
    from pagnerf_b200.mapping import lookup_points, lookup_rays
    pts, comps, k, level = _synthetic(4, level=6, fill=0.3)        # ~630 k points
    P = pts.xyz.shape[0]
    C = 2 ** int(np.ceil(np.log2(2 * P)))
    _index(pts, k, level)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    index = _index(pts, k, level)
    torch.cuda.synchronize()
    growth = torch.cuda.max_memory_allocated() - base
    assert growth <= 12 * C + 3 * 512, (growth, 12 * C)               # keys, points and info, each rounded to 512 bytes
    Q = 1 << 20
    q = torch.from_numpy(_queries(4, k << level, Q)).to(DEV)
    rays = [torch.rand(Q, 3, device=DEV) * 2 - 1, torch.randn(Q, 3, device=DEV), torch.rand(Q, 1, device=DEV), torch.rand(Q, 1, device=DEV)]
    for fn in (lambda: lookup_points(index, q, radius=2, component=comps.component),
               lambda: lookup_rays(index, *rays, radius=2, component=comps.component)):
        fn()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        out = fn()
        torch.cuda.synchronize()
        growth = torch.cuda.max_memory_allocated() - base
        assert growth <= 16 * Q + 2 * 512, (growth, 16 * Q)
        del out
