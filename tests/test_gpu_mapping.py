"""GPU: the panoptic point-map export (pagnerf_b200.mapping; csrc/mapping.cu, the label kernel of csrc/decoder_tiled.cu) against the
CPU oracle (oracle/mapping.py) and against the existing route (nef forward + torch.argmax) on the golden fields."""
import math

import numpy as np
import pytest
import torch

from oracle import mapping as om
from tests.util import load_golden, build_cuda_nef, build_oracle_field, assert_close

pytestmark = pytest.mark.gpu
DEV = "cuda"
GOLDENS = ["trace_delta_permuto_ray", "trace_nef_tcnn_ray", "trace_dd_permuto_ray"]
NEAR = 1e-5


def _nef(name):
    g = load_golden(name)
    nef = build_cuda_nef(g, DEV)
    if "tcnn" in name:
        nef.grid.embedder.round_half = True
    return g, nef


def _cells(nef):
    from pagnerf_b200 import spc
    b = nef.grid.blas
    return spc.unbatched_get_level_points(b.points, b.pyramid, nef.grid.blas_level)


def _threshold(nef, k=2):
    """The median density of the field's map points: half the points are kept (the golden fields are denser than prune()'s
    threshold everywhere)."""
    from pagnerf_b200.mapping import extract_panoptic_map
    return float(extract_panoptic_map(nef, k, min_density=-1.0).density.median())


@pytest.mark.parametrize("name", GOLDENS)
@pytest.mark.parametrize("k", [1, 2, 3])
def test_map_matches_oracle(cuda_lib, name, k):
    from pagnerf_b200.mapping import extract_panoptic_map
    g, nef = _nef(name)
    field = build_oracle_field(g)
    thr = _threshold(nef, k)
    pts = extract_panoptic_map(nef, k, min_density=thr)
    cells = _cells(nef).cpu().numpy()
    ref = om.extract(field, cells, int(g["level"]), k, min_density=thr)
    # the kept set: equal except points whose oracle density is within 1e-5 relative of the threshold
    near = np.abs(ref["all_density"] - thr) <= NEAR * abs(thr)
    allx = om.cell_points(cells, int(g["level"]), k)
    got_keys = {tuple(r) for r in pts.xyz.cpu().numpy().view(np.uint32).tolist()}
    want_keep = ref["all_density"] > thr
    for i, key in enumerate(map(tuple, allx.view(np.uint32).tolist())):
        if not near[i]:
            assert (key in got_keys) == bool(want_keep[i]), (i, ref["all_density"][i], thr)
    # compare the points kept by both, in the common (cell, sub-point) order
    ref_keys = [tuple(r) for r in ref["xyz"].view(np.uint32).tolist()]
    both = [key for key in ref_keys if key in got_keys]
    assert len(both) >= 0.4 * len(ref_keys) > 0
    gi = {key: i for i, key in enumerate(map(tuple, pts.xyz.cpu().numpy().view(np.uint32).tolist()))}
    ri = {key: i for i, key in enumerate(ref_keys)}
    a = torch.tensor([gi[key] for key in both])
    b = np.array([ri[key] for key in both])
    assert (np.diff(a.numpy()) > 0).all(), "output order is cell order, then sub-point order"
    xyz = pts.xyz.cpu()[a].numpy()
    assert np.array_equal(xyz.view(np.uint32), ref["xyz"][b].view(np.uint32))          # bit-exact coordinates
    tol = dict(rtol=2e-3, atol_scale=2e-3) if "tcnn" in name else {}                    # fp16-rounded hash features
    assert_close(pts.density.cpu()[a], torch.from_numpy(ref["density"][b]), msg="density", **tol)
    assert_close(pts.rgb.cpu()[a], torch.from_numpy(ref["rgb"][b]), msg="rgb", **tol)
    srel = 1e-5 if "tcnn" not in name else 2e-3
    for head in ("semantic", "instance"):
        lab = getattr(pts, head).cpu()[a].numpy()
        score = getattr(pts, head + "_score").cpu()[a].double().numpy()
        ok = ref[head + "_gap"][b] > srel          # near-ties (top two logits within the tolerance) may go either way
        assert ok.mean() > 0.5
        assert np.array_equal(lab[ok], ref[head][b][ok]), head
        rs = ref[head + "_score"][b][ok]
        assert np.all(np.abs(score[ok] - rs) <= srel * np.abs(rs) + 1e-12), head


@pytest.mark.parametrize("name", GOLDENS)
def test_map_matches_existing_route(cuda_lib, name):
    """On the same kept points: nef(..., channels={'semantics','inst_embedding'}) + torch.argmax gives the same labels (near-ties
    excepted) and the scores are the max probabilities."""
    from pagnerf_b200.mapping import extract_panoptic_map
    _, nef = _nef(name)
    pts = extract_panoptic_map(nef, 2, min_density=_threshold(nef))
    with torch.no_grad():
        out = nef(coords=pts.xyz[:, None], ray_d=torch.tensor([[0.0, 0.0, -1.0]], device=DEV).expand(pts.xyz.shape[0], 3).contiguous(),
                  channels={'semantics', 'inst_embedding'})
    for head, ch in (("semantic", "semantics"), ("instance", "inst_embedding")):
        p = out[ch].double()
        top2 = p.topk(2, dim=1).values
        ok = (top2[:, 0] - top2[:, 1]) > 1e-5 * top2[:, 0]
        assert ok.float().mean() > 0.5
        assert torch.equal(getattr(pts, head)[ok], p.argmax(1)[ok]), head
        assert_close(getattr(pts, head + "_score"), top2[:, 0].float(), rtol=1e-5, atol_scale=0, msg=head)


def _rand_linear(out, inp, gen, scale=1.0):
    bound = 1.0 / math.sqrt(inp)
    w = (torch.rand(out, inp, generator=gen) * 2 - 1) * bound * scale
    b = (torch.rand(out, generator=gen) * 2 - 1) * bound
    return [w.to(DEV), b.to(DEV)]


@pytest.mark.parametrize("M,Cs,Ci,softmax,temp", [
    (1 << 20, 6, 200, True, 0.0), (1 << 20, 6, 200, True, 0.5), (1 << 20, 2, 20, False, 0.0), (1 << 20, 16, 208, True, 0.0),
    (0, 6, 200, True, 0.0), (1, 6, 200, True, 0.0), (1000, 16, 20, True, 2.0), (1000, 2, 208, False, 0.0), (1000, 6, 0, True, 0.0)])
def test_label_kernel_against_decode_pan(cuda_lib, M, Cs, Ci, softmax, temp):
    """pag_pan_labels_fwd_f32 at bench shapes (IN = 48) against pag_decode_pan_fwd (per-sample [M, C] channels) + argmax."""
    from pagnerf_b200 import ops
    IN = 48
    gen = torch.Generator().manual_seed(M + 31 * Cs + Ci)
    w = (_rand_linear(64, IN, gen) + _rand_linear(max(Cs, 1), 64, gen, 4.0)
         + _rand_linear(64, IN, gen) + _rand_linear(64, 64, gen) + _rand_linear(max(Ci, 1), 64, gen, 4.0))
    feats = torch.randn(M, IN, generator=gen).to(DEV)
    dfeats = (torch.randn(M, IN, generator=gen) * 0.3).to(DEV)
    lodw = (torch.rand(IN, generator=gen) + 0.5).to(DEV)
    with torch.no_grad():
        sl, ss, il, is_ = ops.pan_labels_f32(feats, dfeats, lodw, Cs, Ci, softmax, softmax, temp, *w)
        ps, pi = ops.DecodePanFn.apply(feats, dfeats, lodw, Cs, Ci, softmax, softmax, temp, False, *w)
        # raw logits of the same heads (softmax off, temperature off): the ground truth of the argmax
        zs, zi = ops.DecodePanFn.apply(feats, dfeats, lodw, Cs, Ci, False, False, 0.0, False, *w)
    for lab, score, p, z, C in ((sl, ss, ps, zs, Cs), (il, is_, pi, zi, Ci)):
        if C == 0:
            assert lab is None and score is None
            continue
        assert lab.shape == (M,) and lab.dtype == torch.int64 and score.dtype == torch.float32
        if M == 0:
            continue
        assert torch.equal(lab, z.argmax(1))           # logits bit-identical to the per-thread path: exact, ties included
        want = p.gather(1, lab[:, None])[:, 0]
        assert_close(score, want, rtol=1e-5, atol_scale=0, msg=f"score C={C}")
        if not softmax:
            assert torch.equal(score, p.max(1).values)


@pytest.mark.parametrize("name", GOLDENS)
def test_chunk_invariance(cuda_lib, name):
    from pagnerf_b200.mapping import extract_panoptic_map
    _, nef = _nef(name)
    thr = _threshold(nef)
    a = extract_panoptic_map(nef, 3, min_density=thr)
    b = extract_panoptic_map(nef, 3, min_density=thr, chunk_points=1000)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_edge_thresholds(cuda_lib):
    from pagnerf_b200.mapping import extract_panoptic_map
    _, nef = _nef("trace_delta_permuto_ray")
    pts = extract_panoptic_map(nef, 2, min_density=float("inf"))
    shapes = [(0, 3), (0, 3), (0,), (0,), (0,), (0,), (0,)]
    dtypes = [torch.float32, torch.float32, torch.float32, torch.int64, torch.float32, torch.int64, torch.float32]
    for t, s, d in zip(pts, shapes, dtypes):
        assert t.shape == s and t.dtype == d and t.is_cuda
    every = extract_panoptic_map(nef, 2, min_density=-1.0)
    assert every.xyz.shape[0] == _cells(nef).shape[0] * 8
    zero = extract_panoptic_map(nef, 2, min_density=0.0)
    keep = every.density > 0
    assert torch.equal(zero.xyz, every.xyz[keep]) and torch.equal(zero.instance, every.instance[keep])
    default = extract_panoptic_map(nef, 2)
    assert torch.equal(default.xyz, every.xyz[every.density > (0.01 * 512) / math.sqrt(3)])


def test_map_follows_prune(cuda_lib):
    """After prune() the map covers the new octree's cells only."""
    from pagnerf_b200.mapping import extract_panoptic_map
    from bench import nef_kwargs, CONFIGS
    from pagnerf_b200.pc_nerf import PanopticDeltaNeF
    kw = nef_kwargs(CONFIGS[2])
    kw.update(num_lods=6, capacity_log_2=12, delta_capacity_log_2=12, blas_level=5)
    torch.manual_seed(0)
    nef = PanopticDeltaNeF(**kw)
    for gr in (nef.grid, nef.delta_grid):
        gr.init_from_scales()
    nef = nef.to(DEV)
    with torch.no_grad():       # make a third of the space dense: z-dependent features through the density head's bias row
        nef.grid.embedder.lattice_values.normal_(0, 10.0)
    before = extract_panoptic_map(nef, 1, min_density=-1.0)
    assert before.xyz.shape[0] == 8 ** 5
    nef.prune()
    cells = _cells(nef)
    assert 0 < cells.shape[0] < 8 ** 5
    after = extract_panoptic_map(nef, 1, min_density=-1.0)
    want = (cells.double() * 2 + 1) / 32 - 1
    assert torch.equal(after.xyz, want.float())


def test_memory_stays_below_one_probability_chunk(cuda_lib):
    """2^22 points in chunks of 2^20 at bench shapes (IN = 48, Ci = 200), every point kept: the peak allocation growth stays below
    the [chunk, Ci] fp32 instance tensor that the existing route materialises per chunk."""
    from pagnerf_b200.mapping import extract_panoptic_map
    from pagnerf_b200 import spc
    from bench import nef_kwargs, CONFIGS
    from pagnerf_b200.pc_nerf import PanopticDeltaNeF
    kw = nef_kwargs(CONFIGS[2])
    kw.update(capacity_log_2=16, delta_capacity_log_2=16)
    torch.manual_seed(0)
    nef = PanopticDeltaNeF(**kw)
    n = 1 << 7
    ii = np.stack(np.meshgrid(np.arange(n), np.arange(n), np.arange(n // 4), indexing="ij"), -1).reshape(-1, 3).astype(np.int16)
    octree = spc.unbatched_points_to_octree(torch.from_numpy(ii), 7)
    for gr in (nef.grid, nef.delta_grid):
        gr.init_from_scales()
        gr.blas_init(octree)
    nef = nef.to(DEV)
    chunk = 1 << 20
    extract_panoptic_map(nef, 1, min_density=-1.0, chunk_points=chunk)       # warm: kernels loaded, workspaces cached
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    pts = extract_panoptic_map(nef, 2, min_density=-1.0, chunk_points=chunk)
    torch.cuda.synchronize()
    assert pts.xyz.shape[0] == 1 << 22
    growth = torch.cuda.max_memory_allocated() - base
    assert growth < chunk * nef.num_instances * 4, growth


@pytest.mark.parametrize("name", GOLDENS)
@pytest.mark.parametrize("things", [None, {4, 5}])
def test_instance_summary_against_oracle(cuda_lib, name, things):
    from pagnerf_b200.mapping import extract_panoptic_map, instance_summary
    _, nef = _nef(name)
    pts = extract_panoptic_map(nef, 3, min_density=-1.0)
    s = instance_summary(pts, nef.num_instances, nef.num_classes, things)
    ref = om.summary(pts.xyz.cpu().numpy(), pts.rgb.cpu().numpy(), pts.semantic.cpu().numpy(), pts.instance.cpu().numpy(),
                     nef.num_instances, nef.num_classes, things)
    for key in ("count", "votes", "category", "bbox_min", "bbox_max"):
        assert np.array_equal(getattr(s, key).cpu().numpy(), ref[key]), key
    assert s.centroid.dtype == torch.float64 and s.mean_rgb.dtype == torch.float64
    n = ref["count"] > 0
    assert n.any()
    for key in ("centroid", "mean_rgb"):
        got = getattr(s, key).cpu().numpy()
        assert np.allclose(got[n], ref[key][n], rtol=1e-12, atol=1e-15), key
        assert np.isnan(got[~n]).all()


def test_instance_summary_out_of_range_labels(cuda_lib):
    from pagnerf_b200.mapping import PanopticPoints, instance_summary
    P = 5000
    g = torch.Generator().manual_seed(0)
    sem = torch.randint(0, 6, (P,), generator=g)
    inst = torch.randint(0, 200, (P,), generator=g)
    sem[7], inst[11], inst[12] = 6, -1, 200
    pts = PanopticPoints(*(t.to(DEV) for t in (torch.rand(P, 3, generator=g), torch.rand(P, 3, generator=g), torch.rand(P, generator=g),
                                               sem, torch.rand(P, generator=g), inst, torch.rand(P, generator=g))))
    with pytest.raises(ValueError, match="3 points"):
        instance_summary(pts, 200, 6)
