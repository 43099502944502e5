"""CPU: the panoptic-quality oracle (oracle/metrics.py) against the known answer of torchmetrics' docstring example and a literal
per-pixel dictionary implementation; argument validation of pagnerf_b200.metrics.PanopticQuality; its ABI entries."""
from collections import Counter
from fractions import Fraction

import pytest
import torch
from hypothesis import given, settings, strategies as st

from oracle import metrics as om

KA_PREDS = [[[[6, 0], [0, 0], [6, 0], [6, 0]], [[0, 0], [0, 0], [6, 0], [0, 1]], [[0, 0], [0, 0], [6, 0], [0, 1]],
             [[0, 0], [7, 0], [6, 0], [1, 0]], [[0, 0], [7, 0], [7, 0], [7, 0]]]]
KA_TARGET = [[[[6, 0], [0, 1], [6, 0], [0, 1]], [[0, 1], [0, 1], [6, 0], [0, 1]], [[0, 1], [0, 1], [6, 0], [1, 0]],
              [[0, 1], [7, 0], [1, 0], [1, 0]], [[0, 1], [7, 0], [7, 0], [7, 0]]]]


def brute_force_pq(preds, target, things, stuffs, allow_unknown_preds_category=False):
    """The rules of torchmetrics' PanopticQuality pixel by pixel with dictionaries and exact fractions -> (pq, iou_sum, tp, fp, fn)."""
    order = sorted(things) + sorted(stuffs)
    cont = {c: i for i, c in enumerate(order)}
    void = (1 + max([0, *things, *stuffs]), 0)
    K = len(order)
    iou_sum, tp, fp, fn = [Fraction(0)] * K, [0] * K, [0] * K, [0] * K

    def color(px, allow):
        c, i = int(px[0]), int(px[1])
        if c in stuffs:
            return (c, 0)
        if c in things:
            return (c, i)
        if not allow:
            raise ValueError("unknown category")
        return void

    P = preds.flatten(1, -2)
    T = target.flatten(1, -2)
    for b in range(P.shape[0]):
        pa, ta, ia = Counter(), Counter(), Counter()
        for pp, tt in zip(P[b].tolist(), T[b].tolist()):
            p, t = color(pp, allow_unknown_preds_category), color(tt, True)
            pa[p] += 1
            ta[t] += 1
            ia[(p, t)] += 1
        pm, tm = set(), set()
        for (p, t), inter in ia.items():
            if t == void or p[0] != t[0]:
                continue
            iou = Fraction(inter, pa[p] - ia.get((p, void), 0) + ta[t] - inter)
            if iou > Fraction(1, 2):
                pm.add(p)
                tm.add(t)
                iou_sum[cont[t[0]]] += iou
                tp[cont[t[0]]] += 1
        for t in set(ta) - tm - {void}:
            if Fraction(ia.get((void, t), 0), ta[t]) <= Fraction(1, 2):
                fn[cont[t[0]]] += 1
        for p in set(pa) - pm - {void}:
            if Fraction(ia.get((p, void), 0), pa[p]) <= Fraction(1, 2):
                fp[cont[p[0]]] += 1
    per = [iou_sum[k] / (tp[k] + Fraction(fp[k], 2) + Fraction(fn[k], 2)) for k in range(K) if tp[k] + fp[k] + fn[k] > 0]
    pq = float(sum(per) / len(per)) if per else float("nan")
    return pq, iou_sum, tp, fp, fn


def test_known_answer_of_the_docstring_example():
    preds, target = torch.tensor(KA_PREDS), torch.tensor(KA_TARGET)
    iou_sum, tp, fp, fn = om.panoptic_quality_stats(preds, target, {0, 1}, {6, 7})
    assert torch.allclose(iou_sum, torch.tensor([7 / 9, 0.0, 2 / 3, 1.0], dtype=torch.float64), rtol=1e-15, atol=0)
    assert tp.tolist() == [1, 0, 1, 1] and fp.tolist() == [1, 1, 0, 0] and fn.tolist() == [0, 1, 0, 0]
    pq = om.panoptic_quality(preds, target, {0, 1}, {6, 7})
    assert pq.dtype == torch.float64 and pq.dim() == 0
    assert abs(float(pq) - 59 / 108) < 1e-15 and f"{float(pq):.4f}" == "0.5463"
    # torchmetrics' float32 IoU: same decisions, iou_sum within float32 rounding
    pq32 = om.panoptic_quality(preds, target, {0, 1}, {6, 7}, iou_dtype=torch.float32)
    assert abs(float(pq32) - 59 / 108) < 1e-7
    bf = brute_force_pq(preds, target, {0, 1}, {6, 7})
    assert bf[1] == [Fraction(7, 9), 0, Fraction(2, 3), 1] and abs(bf[0] - 59 / 108) < 1e-15


@st.composite
def _panoptic_case(draw):
    cats = list(range(6))
    roles = draw(st.lists(st.sampled_from(["thing", "stuff", "none"]), min_size=6, max_size=6))
    things = {c for c, r in zip(cats, roles) if r == "thing"}
    stuffs = {c for c, r in zip(cats, roles) if r == "stuff"}
    if not things and not stuffs:
        things = {0}
    allow = draw(st.booleans())
    B, H, W = draw(st.integers(1, 3)), draw(st.integers(1, 5)), draw(st.integers(1, 6))
    n = B * H * W
    known = sorted(things | stuffs)
    t_cat = draw(st.lists(st.sampled_from(cats + [9]), min_size=n, max_size=n))
    p_cat = draw(st.lists(st.sampled_from((cats + [9]) if allow else known), min_size=n, max_size=n))
    t_ins = draw(st.lists(st.integers(0, 3), min_size=n, max_size=n))
    p_ins = draw(st.lists(st.integers(0, 3), min_size=n, max_size=n))
    mk = lambda c, i: torch.stack([torch.tensor(c), torch.tensor(i)], -1).reshape(B, H, W, 2)
    return mk(p_cat, p_ins), mk(t_cat, t_ins), things, stuffs, allow


@settings(max_examples=300, deadline=None)
@given(_panoptic_case())
def test_oracle_equals_per_pixel_dictionaries(case):
    preds, target, things, stuffs, allow = case
    iou_sum, tp, fp, fn = om.panoptic_quality_stats(preds, target, things, stuffs, allow)
    pq_bf, iou_bf, tp_bf, fp_bf, fn_bf = brute_force_pq(preds, target, things, stuffs, allow)
    assert tp.tolist() == tp_bf and fp.tolist() == fp_bf and fn.tolist() == fn_bf
    assert torch.allclose(iou_sum, torch.tensor([float(x) for x in iou_bf], dtype=torch.float64), rtol=1e-14, atol=0)
    pq = float(om.panoptic_quality_compute(iou_sum, tp, fp, fn))
    assert (pq != pq and pq_bf != pq_bf) or abs(pq - pq_bf) <= 1e-14 * max(1.0, abs(pq_bf))


def test_oracle_boundary_cases():
    # IoU exactly 0.5: no match (|p| = 2, |t| = 1, |p∩t| = 1 -> 1 / 2)
    p = torch.tensor([[[[1, 1], [1, 1]]]])
    t = torch.tensor([[[[1, 1], [0, 0]]]])
    _, tp, fp, fn = om.panoptic_quality_stats(p, t, {1}, {0})
    assert tp.tolist() == [0, 0] and fp.tolist() == [1, 0] and fn.tolist() == [1, 1]
    # void overlap exactly half of the prediction segment: still a false positive
    t = torch.tensor([[[[9, 0], [0, 0]]]])
    _, tp, fp, fn = om.panoptic_quality_stats(p, t, {1}, {0})
    assert tp.tolist() == [0, 0] and fp.tolist() == [1, 0] and fn.tolist() == [0, 1]
    # all-void target: a prediction segment that lies in the void is ignored, no category is counted -> NaN
    pq = om.panoptic_quality(torch.tensor([[[[1, 1]]]]), torch.tensor([[[[9, 0]]]]), {1}, {0})
    assert pq != pq
    pq = om.panoptic_quality(torch.tensor([[[[9, 1]]]]), torch.tensor([[[[9, 0]]]]), {1}, {0}, allow_unknown_preds_category=True)
    assert pq != pq


def test_panoptic_quality_argument_validation():
    from pagnerf_b200.metrics import PanopticQuality
    with pytest.raises(ValueError, match="distinct"):
        PanopticQuality(things={0, 1}, stuffs={1, 2})
    with pytest.raises(ValueError, match="non-empty"):
        PanopticQuality(things=set(), stuffs=set())
    with pytest.raises(TypeError, match="integer"):
        PanopticQuality(things={0.5}, stuffs={1})
    with pytest.raises(ValueError, match="At most 256"):
        PanopticQuality(things=set(range(200)), stuffs=set(range(200, 257)))
    with pytest.raises(ValueError, match=r"\[0, 2\^31\)"):
        PanopticQuality(things={-1}, stuffs={1})
    m = PanopticQuality(things={0, 1}, stuffs={6, 7})
    assert m.cat_id_to_continuous_id == {0: 0, 1: 1, 6: 2, 7: 3}
    z = torch.zeros(1, 4, 4, 2, dtype=torch.int64)
    with pytest.raises(ValueError, match="same shape"):
        m.update(z, torch.zeros(1, 4, 5, 2, dtype=torch.int64))
    with pytest.raises(ValueError, match="last dimension"):
        m.update(torch.zeros(1, 4, 3, dtype=torch.int64), torch.zeros(1, 4, 3, dtype=torch.int64))
    with pytest.raises(ValueError, match="spatial"):
        m.update(torch.zeros(4, 2, dtype=torch.int64), torch.zeros(4, 2, dtype=torch.int64))
    with pytest.raises(TypeError, match="integer"):
        m.update(z.float(), z.float())
    with pytest.raises(TypeError, match="tensors"):
        m.update(z.tolist(), z)
    # the oracle validates the same way
    with pytest.raises(ValueError, match="same shape"):
        om.panoptic_quality(z, torch.zeros(1, 4, 5, 2, dtype=torch.int64), {0}, {6})
    with pytest.raises(ValueError, match="Unknown categories"):
        om.panoptic_quality(torch.full((1, 2, 2, 2), 3), z[:, :2, :2], {0}, {6})


def test_panoptic_quality_refuses_cpu_tensors():
    """No CPU fallback: update() on CPU tensors raises instead of computing anywhere else."""
    from pagnerf_b200.metrics import PanopticQuality
    m = PanopticQuality(things={0, 1}, stuffs={6, 7})
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        m.update(torch.tensor(KA_PREDS), torch.tensor(KA_TARGET))
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        m(torch.tensor(KA_PREDS), torch.tensor(KA_TARGET))


def test_pq_entry_points_in_the_header():
    from pagnerf_b200 import _lib
    protos = _lib.parse_header()
    assert len(protos["pag_pq_update"]) == 14 and len(protos["pag_pq_workspace"]) == 3
    assert _lib.KERNELS_PER_CALL["pag_pq_update"] == 3


def test_synthetic_frames_are_seeded_and_shaped():
    p, t = om.synthetic_frames(1, 72, 128, seed=3, n_inst=20)
    p2, t2 = om.synthetic_frames(1, 72, 128, seed=3, n_inst=20)
    assert torch.equal(p, p2) and torch.equal(t, t2) and p.shape == (1, 72, 128, 2) and p.dtype == torch.int64
    assert set(p[..., 0].unique().tolist()) <= {0, 1, 2, 3, 4, 5}
    assert om.SYN_VOID in t[..., 0].unique().tolist()
    assert int(p[..., 1].max()) < 200
