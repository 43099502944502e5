"""CPU: the scene-level panoptic-quality oracle (oracle/scene_metrics.py: the per-image oracle on all frames concatenated) against the
per-pixel dictionary implementation of test_host_metrics and a hand-computed known answer; its invariances; argument validation of
pagnerf_b200.metrics.ScenePanopticQuality; its ABI entries."""
from fractions import Fraction

import pytest
import torch
from hypothesis import given, settings, strategies as st

from oracle import metrics as om
from oracle import scene_metrics as osm
from tests.test_host_metrics import brute_force_pq


def _concat(frames):
    return torch.cat([f.reshape(-1, 2) for f in frames])[None]


@st.composite
def _scene_case(draw):
    cats = list(range(5))
    roles = draw(st.lists(st.sampled_from(["thing", "stuff", "none"]), min_size=5, max_size=5))
    things = {c for c, r in zip(cats, roles) if r == "thing"}
    stuffs = {c for c, r in zip(cats, roles) if r == "stuff"}
    if not things and not stuffs:
        things = {0}
    allow = draw(st.booleans())
    known = sorted(things | stuffs)
    preds, target = [], []
    for _ in range(draw(st.integers(1, 4))):      # frames of mixed sizes
        B, H, W = draw(st.integers(1, 2)), draw(st.integers(1, 4)), draw(st.integers(1, 5))
        n = B * H * W
        t_cat = draw(st.lists(st.sampled_from(cats + [9]), min_size=n, max_size=n))
        p_cat = draw(st.lists(st.sampled_from((cats + [9]) if allow else known), min_size=n, max_size=n))
        t_ins = draw(st.lists(st.integers(0, 3), min_size=n, max_size=n))
        p_ins = draw(st.lists(st.integers(0, 3), min_size=n, max_size=n))
        mk = lambda c, i: torch.stack([torch.tensor(c), torch.tensor(i)], -1).reshape(B, H, W, 2)
        preds.append(mk(p_cat, p_ins))
        target.append(mk(t_cat, t_ins))
    return preds, target, things, stuffs, allow


@settings(max_examples=200, deadline=None)
@given(_scene_case())
def test_scene_oracle_equals_per_pixel_dictionaries_on_the_concatenated_frames(case):
    preds, target, things, stuffs, allow = case
    iou_sum, tp, fp, fn = osm.scene_panoptic_quality_stats(preds, target, things, stuffs, allow)
    pq_bf, iou_bf, tp_bf, fp_bf, fn_bf = brute_force_pq(_concat(preds), _concat(target), things, stuffs, allow)
    assert tp.tolist() == tp_bf and fp.tolist() == fp_bf and fn.tolist() == fn_bf
    assert torch.allclose(iou_sum, torch.tensor([float(x) for x in iou_bf], dtype=torch.float64), rtol=1e-14, atol=0)
    pq = float(om.panoptic_quality_compute(iou_sum, tp, fp, fn))
    assert (pq != pq and pq_bf != pq_bf) or abs(pq - pq_bf) <= 1e-14 * max(1.0, abs(pq_bf))


# Two frames of one row, thing category 1, stuff 0.  Frame 1 (8 px): fruit A (target id 1) 6 px, fruit B (id 2) 2 px.  Frame 2
# (4 px): A 2 px, B 2 px; the prediction swaps the ids of A and B.
KA_SCENE_TARGET = [torch.tensor([[[1, 1]] * 6 + [[1, 2]] * 2]), torch.tensor([[[1, 1]] * 2 + [[1, 2]] * 2])]
KA_SCENE_PREDS = [torch.tensor([[[1, 1]] * 6 + [[1, 2]] * 2]), torch.tensor([[[1, 2]] * 2 + [[1, 1]] * 2])]


def test_known_answer_ids_swapped_in_frame_two():
    # per image: every segment of both frames matches with IoU 1 -> PQ 1
    per = [om.panoptic_quality_stats(p, t, {1}, {0}) for p, t in zip(KA_SCENE_PREDS, KA_SCENE_TARGET)]
    assert sum(s[1][0] for s in per) == 4 and sum(s[2][0] + s[3][0] for s in per) == 0
    per_pq = om.panoptic_quality_compute(*(sum(s[i] for s in per) for i in range(4)))
    assert float(per_pq) == 1.0
    # scene: prediction id 1 = A in frame 1 (6) + B in frame 2 (2) = 8 px, target A = 6 + 2 = 8 px, |p∩t| = 6: IoU 6 / 10 = 3/5 > 1/2.
    # prediction id 2 = B (2) + A (2) = 4 px against B (4 px): |p∩t| = 2, IoU 2 / 6; against A: 2 / 10.  -> tp 1, fp 1, fn 1.
    iou_sum, tp, fp, fn = osm.scene_panoptic_quality_stats(KA_SCENE_PREDS, KA_SCENE_TARGET, {1}, {0})
    assert tp.tolist() == [1, 0] and fp.tolist() == [1, 0] and fn.tolist() == [1, 0]
    assert float(iou_sum[0]) == float(Fraction(3, 5))
    scene_pq = osm.scene_panoptic_quality(KA_SCENE_PREDS, KA_SCENE_TARGET, {1}, {0})
    assert float(scene_pq) == float(Fraction(3, 10)) and float(scene_pq) != float(per_pq)
    bf = brute_force_pq(_concat(KA_SCENE_PREDS), _concat(KA_SCENE_TARGET), {1}, {0})
    assert bf[1] == [Fraction(3, 5), 0] and bf[2:] == ([1, 0], [1, 0], [1, 0])


def test_scene_oracle_is_invariant_to_frame_order_and_splitting():
    p, t = osm.synthetic_sequence(6, 48, 64, seed=3, n_inst=12, consistent=False)
    ref = osm.scene_panoptic_quality_stats(p, t, om.SYN_THINGS, om.SYN_STUFFS)
    orders = [list(range(6))[::-1], [3, 0, 5, 1, 4, 2]]
    for order in orders:
        got = osm.scene_panoptic_quality_stats([p[i:i + 1] for i in order], [t[i:i + 1] for i in order], om.SYN_THINGS, om.SYN_STUFFS)
        assert [x.tolist() for x in got[1:]] == [x.tolist() for x in ref[1:]]
        assert torch.allclose(got[0], ref[0], rtol=1e-14, atol=0)
    # one frame split into two pieces of other shapes, and frames grouped into batches
    pieces_p = [p[:2], p[2, :20].reshape(1, 20 * 64, 2), p[2, 20:][None], p[3:]]
    pieces_t = [t[:2], t[2, :20].reshape(1, 20 * 64, 2), t[2, 20:][None], t[3:]]
    got = osm.scene_panoptic_quality_stats(pieces_p, pieces_t, om.SYN_THINGS, om.SYN_STUFFS)
    assert [x.tolist() for x in got[1:]] == [x.tolist() for x in ref[1:]]
    assert torch.allclose(got[0], ref[0], rtol=1e-14, atol=0)


def test_synthetic_sequence_consistent_and_permuted_ids():
    p, t = osm.synthetic_sequence(6, 96, 128, seed=4, n_inst=20)
    p2, t2 = osm.synthetic_sequence(6, 96, 128, seed=4, n_inst=20)
    assert torch.equal(p, p2) and torch.equal(t, t2) and p.shape == (6, 96, 128, 2) and p.dtype == torch.int64
    assert set(t[..., 1].unique().tolist()) <= set(range(21))
    assert om.SYN_VOID in t[..., 0].unique().tolist() and om.SYN_VOID not in p[..., 0].unique().tolist()
    pq, tq = osm.synthetic_sequence(6, 96, 128, seed=4, n_inst=20, consistent=False)
    assert torch.equal(tq, t)                                          # same scene
    assert torch.equal(pq[..., 0], p[..., 0]) and not torch.equal(pq[..., 1], p[..., 1])
    args = (om.SYN_THINGS, om.SYN_STUFFS)
    per_c, per_p = float(om.panoptic_quality(p, t, *args)), float(om.panoptic_quality(pq, tq, *args))
    scene_c, scene_p = float(osm.scene_panoptic_quality(p, t, *args)), float(osm.scene_panoptic_quality(pq, tq, *args))
    assert per_c == per_p and scene_c > per_c - 0.15 and scene_p < scene_c - 0.15, (per_c, per_p, scene_c, scene_p)
    pv, _ = osm.synthetic_sequence(2, 64, 64, seed=5, pred_void=0.3)
    assert 0.2 < float((pv[..., 0] == om.SYN_VOID).double().mean()) < 0.4


def test_scene_panoptic_quality_argument_validation():
    from pagnerf_b200.metrics import ScenePanopticQuality
    for bad in (0, -1, (1 << 26) + 1):
        with pytest.raises(ValueError, match="capacity"):
            ScenePanopticQuality({1}, {0}, capacity=bad)
    for bad in (2.0, "8", True, None):
        with pytest.raises(TypeError, match="capacity"):
            ScenePanopticQuality({1}, {0}, capacity=bad)
    assert ScenePanopticQuality({1}, {0}, capacity=1).capacity == 1
    assert ScenePanopticQuality({1}, {0}, capacity=1 << 26).capacity == 1 << 26
    with pytest.raises(ValueError, match="distinct"):
        ScenePanopticQuality(things={0, 1}, stuffs={1, 2})
    with pytest.raises(ValueError, match="non-empty"):
        ScenePanopticQuality(things=set(), stuffs=set())
    with pytest.raises(TypeError, match="integer"):
        ScenePanopticQuality(things={0.5}, stuffs={1})
    with pytest.raises(ValueError, match="At most 256"):
        ScenePanopticQuality(things=set(range(200)), stuffs=set(range(200, 257)))
    with pytest.raises(ValueError, match=r"\[0, 2\^31\)"):
        ScenePanopticQuality(things={-1}, stuffs={1})
    m = ScenePanopticQuality(things={0, 1}, stuffs={6, 7})
    assert m.cat_id_to_continuous_id == {0: 0, 1: 1, 6: 2, 7: 3} and m.capacity == 1 << 18
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
    with pytest.raises(ValueError, match="same, non-zero number"):
        osm.scene_panoptic_quality_stats([z, z], [z], {0}, {6})


def test_scene_panoptic_quality_refuses_cpu_tensors():
    from pagnerf_b200.metrics import ScenePanopticQuality
    m = ScenePanopticQuality(things={1}, stuffs={0})
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        m.update(KA_SCENE_PREDS[0], KA_SCENE_TARGET[0])
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        m(KA_SCENE_PREDS[0], KA_SCENE_TARGET[0])


def test_scene_pq_entry_points_in_the_header_and_the_library():
    from pagnerf_b200 import _lib
    protos = _lib.parse_header()
    assert len(protos["pag_scene_pq_workspace"]) == 2 and len(protos["pag_scene_pq_update"]) == 12
    assert len(protos["pag_scene_pq_stats"]) == 7 and len(protos["pag_scene_pq_merge"]) == 5
    assert _lib.KERNELS_PER_CALL["pag_scene_pq_stats"] == 2 and _lib.KERNELS_PER_CALL["pag_scene_pq_merge"] == 2
    syms = _lib.exported_symbols()
    assert {"pag_scene_pq_workspace", "pag_scene_pq_update", "pag_scene_pq_stats", "pag_scene_pq_merge"} <= set(syms)
    # 64 B per slot of C = the smallest power of two >= 2 * capacity, plus the counters
    assert _lib.query_i64("pag_scene_pq_workspace", 1 << 18) == 64 * (1 << 19) + 128
    assert _lib.query_i64("pag_scene_pq_workspace", 3) == 64 * 8 + 128
    with pytest.raises(RuntimeError):
        _lib.query_i64("pag_scene_pq_workspace", (1 << 26) + 1)
