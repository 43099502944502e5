"""GPU: pagnerf_b200.metrics.ScenePanopticQuality (csrc/metrics.cu, pag_scene_pq_*) against the CPU oracle (oracle/scene_metrics.py:
the per-image oracle on all frames concatenated).  tp / fp / fn exact, iou_sum and PQ to 1e-12 relative (float64 sums in another order)."""
import os
import socket
import subprocess
import sys

import pytest
import torch

from oracle import metrics as om
from oracle import scene_metrics as osm

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = (om.SYN_THINGS, om.SYN_STUFFS)


def _assert_pq_close(a, b):
    a, b = float(a), float(b)
    assert (a != a and b != b) or abs(a - b) <= 1e-12 * max(1.0, abs(b)), (a, b)


def _assert_stats_equal(dev_stats, ref_stats):
    iou, tp, fp, fn = (x.cpu() for x in dev_stats)
    r_iou, r_tp, r_fp, r_fn = (x.cpu() for x in ref_stats)
    assert torch.equal(tp, r_tp) and torch.equal(fp, r_fp) and torch.equal(fn, r_fn), ((tp, fp, fn), (r_tp, r_fp, r_fn))
    assert torch.allclose(iou, r_iou, rtol=1e-12, atol=0), (iou, r_iou)


def _scene(things=om.SYN_THINGS, stuffs=om.SYN_STUFFS, **kw):
    from pagnerf_b200.metrics import ScenePanopticQuality
    return ScenePanopticQuality(things, stuffs, **kw).cuda()


def _distinct_keys(p, t, things, stuffs, allow=False):
    """-> distinct keys of the prediction-segment, target-segment and pair tables (host restatement of the device keys)."""
    void = om.void_color(things, stuffs)
    pp = om.preprocess(p.reshape(1, -1, 2), things, stuffs, void, allow)[0]
    tt = om.preprocess(t.reshape(1, -1, 2), things, stuffs, void, True)[0]
    kp, kt = (pp[:, 0] << 32) | pp[:, 1], (tt[:, 0] << 32) | tt[:, 1]
    vp, vt = pp[:, 0] == void[0], tt[:, 0] == void[0]
    pair = ~vp & ~vt & (pp[:, 0] == tt[:, 0])
    n_pair = len(torch.unique(torch.stack([kp[pair], kt[pair]], 1), dim=0))
    return [len(kp[~vp].unique()), len(kt[~vt].unique()), n_pair]


@pytest.mark.parametrize("n,H,W", [(32, 256, 256), (4, 1024, 1024)])
@pytest.mark.parametrize("consistent", [True, False])
def test_scene_equals_oracle(cuda_lib, n, H, W, consistent):
    p, t = osm.synthetic_sequence(n, H, W, seed=n + H, n_inst=150 if H == 1024 else 40, consistent=consistent)
    m = _scene()
    m.update(p.cuda(), t.cuda())
    pq = m.compute()
    assert pq.dtype == torch.float64 and pq.dim() == 0 and pq.is_cuda
    ref = osm.scene_panoptic_quality_stats(p, t, *ARGS)
    _assert_stats_equal(m.stats(), ref)
    _assert_pq_close(pq, om.panoptic_quality_compute(*ref))
    assert m.keys_used().cpu().tolist() == _distinct_keys(p, t, *ARGS)
    per_image = float(om.panoptic_quality(p, t, *ARGS))
    if consistent:
        assert float(pq) > per_image - 0.15
    else:
        assert float(pq) < per_image - 0.3


@pytest.mark.parametrize("kind", ["allow_unknown", "void_heavy"])
def test_scene_void_and_unknown_predictions(cuda_lib, kind):
    allow = kind == "allow_unknown"
    p, t = osm.synthetic_sequence(8, 256, 256, seed=21, n_inst=40, void=0.6 if kind == "void_heavy" else 0.02,
                                 pred_void=0.3 if allow else 0.0)
    m = _scene(allow_unknown_preds_category=allow)
    for f in range(8):
        m.update(p[f:f + 1].cuda(), t[f:f + 1].cuda())
    ref = osm.scene_panoptic_quality_stats(p, t, *ARGS, allow_unknown_preds_category=allow)
    _assert_stats_equal(m.stats(), ref)
    _assert_pq_close(m.compute(), om.panoptic_quality_compute(*ref))


def test_one_frame_equals_panoptic_quality(cuda_lib):
    from pagnerf_b200.metrics import PanopticQuality
    p, t = om.synthetic_frames(1, 720, 1280, seed=3)
    per = PanopticQuality(*ARGS).cuda()
    per.update(p.cuda(), t.cuda())
    m = _scene()
    m.update(p.cuda(), t.cuda())
    _assert_stats_equal(m.stats(), per.stats())
    _assert_pq_close(m.compute(), per.compute())


def test_update_split_and_order_do_not_matter(cuda_lib):
    p, t = osm.synthetic_sequence(12, 200, 300, seed=5, n_inst=40, consistent=False)
    pd, td = p.cuda(), t.cuda()
    a, b, c = _scene(), _scene(), _scene()
    for f in range(12):
        a.update(pd[f:f + 1], td[f:f + 1])
        c.update(pd[11 - f:12 - f], td[11 - f:12 - f])
    b.update(pd, td)
    ref = osm.scene_panoptic_quality_stats(p, t, *ARGS)
    for m in (a, b, c):
        _assert_stats_equal(m.stats(), ref)
    # frames of other sizes: the same pixels as a [1, N] row and as crops
    d = _scene()
    d.update(pd[:4].reshape(1, -1, 2), td[:4].reshape(1, -1, 2))
    d.update(pd[4:, :100], td[4:, :100])
    d.update(pd[4:, 100:], td[4:, 100:])
    _assert_stats_equal(d.stats(), ref)


def test_compute_mid_sequence_is_non_destructive(cuda_lib):
    p, t = osm.synthetic_sequence(10, 256, 256, seed=6, n_inst=40)
    pd, td = p.cuda(), t.cuda()
    m = _scene()
    m.update(pd[:5], td[:5])
    ws = m._workspace.clone()
    mid = m.compute()
    _assert_pq_close(mid, osm.scene_panoptic_quality(p[:5], t[:5], *ARGS))
    m.stats()
    m.keys_used()
    torch.cuda.synchronize()
    assert torch.equal(m._workspace, ws), "stats() / compute() changed the tables"
    m.update(pd[5:], td[5:])
    one = _scene()
    one.update(pd, td)
    _assert_stats_equal(m.stats(), one.stats())
    _assert_pq_close(m.compute(), one.compute())
    _assert_stats_equal(m.stats(), osm.scene_panoptic_quality_stats(p, t, *ARGS))
    m.reset()
    assert int(m._workspace.abs().sum()) == 0 and int(m.keys_used().sum()) == 0


def test_table_overflow_is_an_error_not_a_hang(cuda_lib):
    p, t = osm.synthetic_sequence(6, 128, 128, seed=7, n_inst=40)
    need = _distinct_keys(p, t, *ARGS)
    cap = max(need)
    table = ("prediction segment", "target segment", "pair")[need.index(cap)]
    ok = _scene(capacity=cap)
    ok.update(p.cuda(), t.cuda())
    _assert_stats_equal(ok.stats(), osm.scene_panoptic_quality_stats(p, t, *ARGS))
    ok.compute()
    assert ok.keys_used().cpu().tolist() == need
    small = _scene(capacity=cap - 1)
    small.update(p.cuda(), t.cuda())
    with pytest.raises(ValueError, match=rf"the {table} table refused [1-9]\d* pixels \({cap - 1} of {cap - 1} keys used\)"):
        small.compute()
    assert max(small.keys_used().cpu().tolist()) == cap - 1
    # a tiny capacity: every table full, still an error and no hang
    tiny = _scene(capacity=3)
    tiny.update(p.cuda(), t.cuda())
    with pytest.raises(ValueError, match="suffices"):
        tiny.compute()
    # reset() empties the tables; with the capacity the message names, the same frames pass
    small.reset()
    assert int(small.keys_used().sum()) == 0 and float(small._workspace.abs().sum()) == 0
    with pytest.raises(ValueError) as e:
        tiny.compute()
    suffices = int(str(e.value).split("A capacity of ")[1].split()[0])
    assert suffices >= cap
    big = _scene(capacity=suffices)
    big.update(p.cuda(), t.cuda())
    _assert_pq_close(big.compute(), osm.scene_panoptic_quality(p, t, *ARGS))


def test_areas_are_64_bit(cuda_lib):
    """4097 updates of a 1024x1024 frame: 2^32 + 2^20 pixels.  One predicted thing segment over the whole frame; the target gives
    three quarters of it id 1 and the rest id 2: IoU exactly 0.75 with id 1 (a wrapped u32 area of 2^20 would give 3072.75)."""
    n = 1024 * 1024
    p = torch.stack([torch.ones(n, dtype=torch.int64), torch.full((n,), 5, dtype=torch.int64)], -1).reshape(1, 1024, 1024, 2).cuda()
    t = p.clone()
    t[0, :, :, 1] = 1
    t[0, 768:, :, 1] = 2
    m = _scene(things={1}, stuffs={0})
    for _ in range(4097):
        m.update(p, t)
    iou, tp, fp, fn = (x.cpu() for x in m.stats())
    assert float(iou[0]) == 0.75 and tp.tolist() == [1, 0] and fp.tolist() == [0, 0] and fn.tolist() == [1, 0]
    _assert_pq_close(m.compute(), 0.75 / 1.5)


def test_deferred_errors(cuda_lib):
    p, t = osm.synthetic_sequence(2, 64, 64, seed=8, n_inst=10)
    bad = p.clone()
    bad[0, 0, :3, 0] = 7                      # three prediction pixels of a category in neither set
    m = _scene()
    m.update(bad.cuda(), t.cuda())            # no raise here: the device counts
    with pytest.raises(ValueError, match="Unknown categories found in `preds`: 3 pixels"):
        m.compute()
    m.reset()
    m.update(p.cuda(), t.cuda())
    _assert_pq_close(m.compute(), osm.scene_panoptic_quality(p, t, *ARGS))
    big = p.clone()
    big[1, 5, 5] = torch.tensor([2, 2 ** 31])
    big[1, 6, 6] = torch.tensor([3, -1])
    m = _scene()
    m(big.cuda(), t.cuda())                   # forward is update and returns nothing
    with pytest.raises(ValueError, match=r"2 pixels of a `things` category have an instance id outside"):
        m.compute()


def test_update_makes_no_host_sync(cuda_lib):
    p, t = osm.synthetic_sequence(3, 96, 128, seed=9, n_inst=20)
    p, t = p.cuda(), t.cuda()
    m = _scene()
    m.update(p, t)                            # library load, workspace allocation
    m.reset()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        assert m(p, t) is None
        m.update(p.to(torch.int32), t.to(torch.int32))
    finally:
        torch.cuda.set_sync_debug_mode(0)
    ref = osm.scene_panoptic_quality_stats(torch.cat([p, p]).cpu(), torch.cat([t, t]).cpu(), *ARGS)
    _assert_stats_equal(m.stats(), ref)


def test_update_captured_in_a_cuda_graph(cuda_lib):
    pa, ta = osm.synthetic_sequence(2, 80, 120, seed=10, n_inst=20)
    pb, tb = osm.synthetic_sequence(2, 80, 120, seed=11, n_inst=20, consistent=False)
    sp, st = pa.cuda(), ta.cuda()
    m = _scene()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        m.update(sp, st)                      # warm-up outside the capture (workspace)
    torch.cuda.current_stream().wait_stream(s)
    m.reset()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        m.update(sp, st)
    m.reset()
    g.replay()
    sp.copy_(pb.cuda())
    st.copy_(tb.cuda())
    g.replay()
    torch.cuda.synchronize()
    e = _scene()
    e.update(pa.cuda(), ta.cuda())
    e.update(pb.cuda(), tb.cuda())
    _assert_stats_equal(m.stats(), e.stats())
    _assert_stats_equal(m.stats(), osm.scene_panoptic_quality_stats([pa, pb], [ta, tb], *ARGS))


_WORKER = r'''
import os, sys, torch, torch.distributed as dist
root, port, rank, out = sys.argv[1], sys.argv[2], int(sys.argv[3]), sys.argv[4]
sys.path.insert(0, root)
from oracle import metrics as om
from oracle import scene_metrics as osm
from pagnerf_b200.metrics import ScenePanopticQuality
dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=2)
p, t = osm.synthetic_sequence(6, 128, 160, seed=12, n_inst=30)
m = ScenePanopticQuality(om.SYN_THINGS, om.SYN_STUFFS).to("cuda:0")
m.update(p[rank::2].cuda(), t[rank::2].cuda())          # alternate frames: the same fruit and prediction ids on both ranks
own = [x.cpu() for x in m.stats()]
m.sync()
torch.save({"own": own, "synced": [x.cpu() for x in m.stats()] + [m.compute().cpu(), m.keys_used().cpu()]}, out)
dist.barrier()
dist.destroy_process_group()
print("OK", rank)
'''


def test_two_rank_sync_is_the_union_of_the_tables(cuda_lib, tmp_path):
    """Frames sharded across ranks: after sync() every rank holds one rank's result over all frames.  A fruit seen on both ranks
    is one segment there, so this differs from the sum of the two ranks' scene statistics.  The ranks share cuda:0 over gloo."""
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    outs = [str(tmp_path / f"stats{r}.pt") for r in range(2)]
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, str(port), str(r), outs[r]], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    logs = [p.communicate(timeout=600)[0] for p in procs]
    for r, (p, lg) in enumerate(zip(procs, logs)):
        assert p.returncode == 0 and f"OK {r}" in lg, lg[-3000:]
    p, t = osm.synthetic_sequence(6, 128, 160, seed=12, n_inst=30)
    one = _scene()
    one.update(p.cuda(), t.cuda())
    r0, r1 = torch.load(outs[0]), torch.load(outs[1])
    for a, b in zip(r0["synced"][1:4] + r0["synced"][5:], r1["synced"][1:4] + r1["synced"][5:]):
        assert torch.equal(a, b), "ranks disagree after sync()"
    assert torch.allclose(r0["synced"][0], r1["synced"][0], rtol=1e-12, atol=0)
    _assert_stats_equal(r0["synced"][:4], one.stats())
    _assert_pq_close(r0["synced"][4], one.compute())
    assert r0["synced"][5].tolist() == one.keys_used().cpu().tolist()
    summed = [a + b for a, b in zip(r0["own"], r1["own"])]
    assert not torch.equal(summed[1], r0["synced"][1]), "summing per-rank scene statistics should not equal the scene union"


def test_map_objects_scored_over_a_sequence(cuda_lib):
    """INTEGRATION 6: pixels resolved to the map's objects.  Each frame sees a random subset of the map's points; the target is
    (category, object + 1) from the map's components, the prediction the lookup of those points.  Consistent object ids give scene
    PQ 1; relabelling the objects in every frame keeps every per-frame PQ at 1 and lowers the scene PQ."""
    from pagnerf_b200.mapping import lookup_points
    from pagnerf_b200.metrics import PanopticQuality
    from tests.test_gpu_lookup import _index, _synthetic
    pts, comps, k, level = _synthetic(seed=13)
    index = _index(pts, k, level)
    things, stuffs = {1, 2}, {0}
    n_obj = comps.count.numel()
    assert n_obj > 4
    g = torch.Generator(device="cuda").manual_seed(0)
    good, bad, per = (_scene(things, stuffs), _scene(things, stuffs), PanopticQuality(things, stuffs).cuda())
    for f in range(6):
        sel = torch.randperm(pts.xyz.shape[0], device="cuda", generator=g)[:4096]
        target = torch.stack([pts.semantic[sel], comps.component[sel] + 1], -1)[None]
        hit = lookup_points(index, pts.xyz[sel], radius=0, component=comps.component)
        assert torch.equal(hit.point, sel)
        pred = torch.stack([pts.semantic[hit.point], hit.object + 1], -1)[None]
        relabel = torch.cat([torch.zeros(1, dtype=torch.int64, device="cuda"),
                             1 + torch.randperm(n_obj, device="cuda", generator=g)])
        pred_bad = torch.stack([pred[..., 0], relabel[pred[..., 1]]], -1)
        good.update(pred, target)
        bad.update(pred_bad, target)
        assert float(per(pred_bad, target)) == 1.0
    assert float(good.compute()) == 1.0
    assert float(bad.compute()) < 0.9, float(bad.compute())
