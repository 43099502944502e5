"""GPU: pagnerf_b200.metrics.PanopticQuality (csrc/metrics.cu) against the CPU oracle (oracle/metrics.py).  tp / fp / fn exact,
iou_sum and PQ to 1e-12 relative (float64 sums in another order)."""
import os
import socket
import subprocess
import sys

import pytest
import torch

from oracle import metrics as om

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

KA_PREDS = [[[[6, 0], [0, 0], [6, 0], [6, 0]], [[0, 0], [0, 0], [6, 0], [0, 1]], [[0, 0], [0, 0], [6, 0], [0, 1]],
             [[0, 0], [7, 0], [6, 0], [1, 0]], [[0, 0], [7, 0], [7, 0], [7, 0]]]]
KA_TARGET = [[[[6, 0], [0, 1], [6, 0], [0, 1]], [[0, 1], [0, 1], [6, 0], [0, 1]], [[0, 1], [0, 1], [6, 0], [1, 0]],
              [[0, 1], [7, 0], [1, 0], [1, 0]], [[0, 1], [7, 0], [7, 0], [7, 0]]]]


def _assert_pq_close(a, b):
    a, b = float(a), float(b)
    assert (a != a and b != b) or abs(a - b) <= 1e-12 * max(1.0, abs(b)), (a, b)


def _assert_stats_equal(dev_stats, ref_stats):
    iou, tp, fp, fn = (x.cpu() for x in dev_stats)
    r_iou, r_tp, r_fp, r_fn = ref_stats
    assert torch.equal(tp, r_tp) and torch.equal(fp, r_fp) and torch.equal(fn, r_fn), ((tp, fp, fn), (r_tp, r_fp, r_fn))
    assert torch.allclose(iou, r_iou, rtol=1e-12, atol=0), (iou, r_iou)


def _check(preds, target, things, stuffs, allow=False):
    """device update + compute == oracle; -> the module"""
    from pagnerf_b200.metrics import PanopticQuality
    m = PanopticQuality(things, stuffs, allow_unknown_preds_category=allow).cuda()
    m.update(preds.cuda(), target.cuda())
    pq = m.compute()
    assert pq.dtype == torch.float64 and pq.dim() == 0 and pq.is_cuda
    ref = om.panoptic_quality_stats(preds, target, things, stuffs, allow)
    _assert_stats_equal(m.stats(), ref)
    _assert_pq_close(pq, om.panoptic_quality_compute(*ref))
    return m


def test_known_answer(cuda_lib):
    from pagnerf_b200.metrics import PanopticQuality
    p, t = torch.tensor(KA_PREDS), torch.tensor(KA_TARGET)
    m = _check(p, t, {0, 1}, {6, 7})
    iou, tp, fp, fn = m.stats()
    assert tp.tolist() == [1, 0, 1, 1] and fp.tolist() == [1, 1, 0, 0] and fn.tolist() == [0, 1, 0, 0]
    _assert_pq_close(m.compute(), 59 / 108)
    pq = PanopticQuality(things={0, 1}, stuffs={6, 7}).cuda()
    batch_value = pq(p.cuda(), t.cuda())            # the docstring's usage: __call__ returns the batch PQ
    assert f"{float(batch_value):.4f}" == "0.5463"
    _assert_pq_close(pq.compute(), 59 / 108)        # ... and accumulates it


def test_iou_exactly_half_is_no_match(cuda_lib):
    m = _check(torch.tensor([[[[1, 1], [1, 1]]]]), torch.tensor([[[[1, 1], [0, 0]]]]), {1}, {0})
    assert m.counts[0].tolist() == [0, 0]


def test_void_overlap_exactly_half_still_counts(cuda_lib):
    m = _check(torch.tensor([[[[1, 1], [1, 1]]]]), torch.tensor([[[[9, 0], [0, 0]]]]), {1}, {0})
    assert m.counts[1].tolist() == [1, 0]
    # and on the target side: half of a target segment is void in the prediction -> still a false negative
    m = _check(torch.tensor([[[[9, 0], [0, 0]]]]), torch.tensor([[[[1, 1], [1, 1]]]]), {1}, {0}, allow=True)
    assert m.counts[2].tolist() == [1, 0] and m.counts[1].tolist() == [0, 1]


def test_all_void_images(cuda_lib):
    g = torch.Generator().manual_seed(0)
    p = torch.stack([torch.randint(0, 3, (2, 8, 8), generator=g), torch.randint(0, 4, (2, 8, 8), generator=g)], -1)
    t = torch.full((2, 8, 8, 2), 7)
    m = _check(p, t, {1, 2}, {0})
    assert float(m.compute()) != float(m.compute())      # nothing counted: NaN
    _check(torch.full((2, 8, 8, 2), 7), t, {1, 2}, {0}, allow=True)


def test_category_only_in_prediction(cuda_lib):
    g = torch.Generator().manual_seed(1)
    t = torch.stack([torch.randint(0, 2, (2, 16, 16), generator=g), torch.randint(0, 3, (2, 16, 16), generator=g)], -1)
    p = t.clone()
    p[:, 4:9, 4:12, 0] = 2
    m = _check(p, t, {1, 2}, {0})
    assert m.counts[1, 1] > 0 and m.counts[0, 1] == 0


def test_same_colours_in_different_images(cuda_lib):
    g = torch.Generator().manual_seed(2)
    t = torch.stack([torch.randint(0, 3, (4, 12, 12), generator=g), torch.randint(0, 3, (4, 12, 12), generator=g)], -1)
    p = torch.stack([torch.randint(0, 3, (4, 12, 12), generator=g), torch.randint(0, 3, (4, 12, 12), generator=g)], -1)
    p[1], t[1] = p[0], t[0]
    p[3] = t[3]
    m = _check(p, t, {1, 2}, {0})
    one = [om.panoptic_quality_stats(p[b:b + 1], t[b:b + 1], {1, 2}, {0}) for b in range(4)]
    assert torch.equal(m.counts[0].cpu(), sum(s[1] for s in one))      # segments never merge across images


def test_instance_id_2p31_minus_1(cuda_lib):
    top = 2 ** 31 - 1
    t = torch.tensor([[[[1, top], [1, top], [1, 5]], [[1, top], [0, 0], [1, 5]]]])
    p = torch.tensor([[[[1, top - 1], [1, top - 1], [1, top]], [[1, top - 1], [0, 3], [1, top]]]])
    m = _check(p, t, {1}, {0})
    assert m.counts[0].tolist() == [2, 1]


def test_every_pixel_its_own_segment_256x256(cuda_lib):
    """65 536 segments per map: the worst case of the hash tables (2 slots per pixel)."""
    n = 256 * 256
    g = torch.Generator().manual_seed(3)
    inst_t = torch.randperm(n, generator=g)
    inst_p = inst_t.clone()
    inst_p[: n // 4] = n + torch.arange(n // 4) // 2      # pairs of pixels: IoU 1/2 with each single-pixel target, no match
    cat = torch.ones(n, dtype=torch.int64)
    t = torch.stack([cat, inst_t], -1).reshape(1, 256, 256, 2)
    p = torch.stack([cat, inst_p], -1).reshape(1, 256, 256, 2)
    t = torch.cat([t, t.flip(1)])
    p = torch.cat([p, p.flip(1)])
    m = _check(p, t, {1}, {0})
    assert m.counts[0, 0] == 2 * (n - n // 4)


def test_accumulation_equals_one_concatenated_update(cuda_lib):
    from pagnerf_b200.metrics import PanopticQuality
    p, t = om.synthetic_frames(3, 96, 160, seed=4, n_inst=40)
    p, t = p.cuda(), t.cuda()
    a = PanopticQuality(om.SYN_THINGS, om.SYN_STUFFS).cuda()
    for b in range(3):
        a.update(p[b:b + 1], t[b:b + 1])
    c = PanopticQuality(om.SYN_THINGS, om.SYN_STUFFS).cuda()
    c.update(p, t)
    _assert_stats_equal(a.stats(), [x.cpu() for x in c.stats()])
    _assert_pq_close(a.compute(), c.compute())
    a.reset()
    assert float(a.iou_sum.abs().sum()) == 0 and int(a.counts.abs().sum()) == 0


def test_deferred_errors(cuda_lib):
    from pagnerf_b200.metrics import PanopticQuality
    p, t = torch.tensor(KA_PREDS).cuda(), torch.tensor(KA_TARGET).cuda()
    bad = p.clone()
    bad[0, 0, :2, 0] = 3                      # two prediction pixels of a category in neither set
    m = PanopticQuality(things={0, 1}, stuffs={6, 7}).cuda()
    m.update(bad, t)                          # no raise here: the device counts
    assert m.errors.tolist() == [2, 0]
    with pytest.raises(ValueError, match="Unknown categories found in `preds`: 2 pixels"):
        m.compute()
    _assert_pq_close(m(p, t), 59 / 108)       # __call__ scores its own batch ...
    with pytest.raises(ValueError, match="Unknown categories found in `preds`: 2 pixels"):
        m.compute()                           # ... the error stays in the accumulated state until reset()
    m.reset()
    _assert_pq_close(m(p, t), 59 / 108)
    with pytest.raises(ValueError, match="Unknown categories"):
        m(bad, t)
    # allowed: the unknown pixels are void
    _check(bad.cpu(), t.cpu(), {0, 1}, {6, 7}, allow=True)
    # a thing's instance id outside [0, 2^31)
    big = p.clone()
    big[0, 1, 3, 1] = 2 ** 31
    big[0, 2, 3, 1] = -1
    m = PanopticQuality(things={0, 1}, stuffs={6, 7}).cuda()
    m.update(big, t)
    with pytest.raises(ValueError, match=r"2 pixels of a `things` category have an instance id outside"):
        m.compute()


def test_update_makes_no_host_sync(cuda_lib):
    from pagnerf_b200.metrics import PanopticQuality
    p, t = om.synthetic_frames(2, 64, 96, seed=5, n_inst=20)
    p, t = p.cuda(), t.cuda()
    m = PanopticQuality(om.SYN_THINGS, om.SYN_STUFFS).cuda()
    m.update(p, t)                            # library load, workspace allocation
    m.reset()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        m.update(p, t)
        m.update(p.to(torch.int32), t.to(torch.int32))      # other integer dtypes: converted on the device
    finally:
        torch.cuda.set_sync_debug_mode(0)
    ref = om.panoptic_quality_stats(torch.cat([p, p]).cpu(), torch.cat([t, t]).cpu(), om.SYN_THINGS, om.SYN_STUFFS)
    _assert_stats_equal(m.stats(), ref)


def test_update_captured_in_a_cuda_graph(cuda_lib):
    from pagnerf_b200.metrics import PanopticQuality
    pa, ta = om.synthetic_frames(2, 80, 120, seed=6, n_inst=30)
    pb, tb = om.synthetic_frames(2, 80, 120, seed=7, n_inst=30)
    sp, st = pa.cuda(), ta.cuda()
    m = PanopticQuality(om.SYN_THINGS, om.SYN_STUFFS).cuda()
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
    e = PanopticQuality(om.SYN_THINGS, om.SYN_STUFFS).cuda()
    e.update(pa.cuda(), ta.cuda())
    e.update(pb.cuda(), tb.cuda())
    _assert_stats_equal(m.stats(), [x.cpu() for x in e.stats()])
    ref = om.panoptic_quality_stats(torch.cat([pa, pb]), torch.cat([ta, tb]), om.SYN_THINGS, om.SYN_STUFFS)
    _assert_stats_equal(m.stats(), ref)


@pytest.mark.parametrize("H,W,B", [(1024, 1024, 1), (720, 1280, 3)])
def test_synthetic_frames(cuda_lib, H, W, B):
    """~150 target and prediction instances per frame; three 1280x720 frames take two launches (two images fit the workspace)."""
    p, t = om.synthetic_frames(B, H, W, seed=H + W)
    n_t = [len(t[b, ..., 1].unique()) - 1 for b in range(B)]
    assert min(n_t) > 100
    m = _check(p, t, om.SYN_THINGS, om.SYN_STUFFS)
    assert int(m.counts[0].sum()) > 50 * B


_WORKER = r'''
import os, sys, torch, torch.distributed as dist
root, port, rank, out = sys.argv[1], sys.argv[2], int(sys.argv[3]), sys.argv[4]
sys.path.insert(0, root)
from oracle import metrics as om
from pagnerf_b200.metrics import PanopticQuality
dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=2)
p, t = om.synthetic_frames(2, 200, 300, seed=11, n_inst=60)
m = PanopticQuality(om.SYN_THINGS, om.SYN_STUFFS).to("cuda:0")
m.update(p[rank:rank + 1].cuda(), t[rank:rank + 1].cuda())
m.sync()
torch.save([x.cpu() for x in m.stats()] + [m.compute().cpu()], out)
dist.barrier()
dist.destroy_process_group()
print("OK", rank)
'''


def test_two_rank_sync_equals_one_rank(cuda_lib, tmp_path):
    """Validation frames sharded across ranks as whole images: the summed statistics equal one rank that sees every frame.
    The two ranks share cuda:0 and talk over gloo (NCCL refuses two ranks on one device)."""
    from pagnerf_b200.metrics import PanopticQuality
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    outs = [str(tmp_path / f"stats{r}.pt") for r in range(2)]
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, str(port), str(r), outs[r]], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    logs = [p.communicate(timeout=600)[0] for p in procs]
    for r, (p, lg) in enumerate(zip(procs, logs)):
        assert p.returncode == 0 and f"OK {r}" in lg, lg[-3000:]
    p, t = om.synthetic_frames(2, 200, 300, seed=11, n_inst=60)
    one = PanopticQuality(om.SYN_THINGS, om.SYN_STUFFS).cuda()
    one.update(p.cuda(), t.cuda())
    r0, r1 = torch.load(outs[0]), torch.load(outs[1])
    for a, b in zip(r0, r1):
        assert torch.equal(a, b), "ranks disagree after sync()"
    _assert_stats_equal(r0[:4], [x.cpu() for x in one.stats()])
    _assert_pq_close(r0[4], one.compute())
