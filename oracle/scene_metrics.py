"""CPU oracle of scene-level panoptic quality (pagnerf_b200.metrics.ScenePanopticQuality) -- TEST INFRASTRUCTURE ONLY.

Scene PQ is DEFINED as the per-image statistics of one image made of all pixels of all frames, so ``scene_panoptic_quality_stats``
concatenates the frames and calls ``oracle.metrics.panoptic_quality_stats``: no second implementation.  ``synthetic_sequence``
makes seeded sequences in which the target's fruit keep their ids while they move, with prediction ids kept or permuted per frame
(tools/scene_pq_bench.py, tests/test_host_scene_metrics.py, tests/test_gpu_scene_metrics.py)."""
import numpy as np
import torch

from .metrics import SYN_VOID, _paint_disc, panoptic_quality_compute, panoptic_quality_stats, validate_inputs


def scene_panoptic_quality_stats(frames_preds, frames_target, things, stuffs, allow_unknown_preds_category=False,
                                 iou_dtype=torch.float64):
    """Scene PQ statistics of a sequence: the per-image statistics of ONE image made of all pixels of all frames.

    frames_preds / frames_target: a [B, *spatial, 2] tensor, or a list of them of any sizes (frame i of preds and of target have
    the same shape).  -> iou_sum f64[K], tp, fp, fn i64[K] in continuous-id order."""
    if isinstance(frames_preds, torch.Tensor):
        frames_preds, frames_target = [frames_preds], [frames_target]
    if len(frames_preds) != len(frames_target) or not frames_preds:
        raise ValueError("Expected the same, non-zero number of prediction and target frames")
    for p, t in zip(frames_preds, frames_target):
        validate_inputs(p, t)
    p = torch.cat([x.detach().cpu().to(torch.int64).reshape(-1, 2) for x in frames_preds])[None]
    t = torch.cat([x.detach().cpu().to(torch.int64).reshape(-1, 2) for x in frames_target])[None]
    return panoptic_quality_stats(p, t, things, stuffs, allow_unknown_preds_category, iou_dtype)


def scene_panoptic_quality(frames_preds, frames_target, things, stuffs, allow_unknown_preds_category=False):
    return panoptic_quality_compute(*scene_panoptic_quality_stats(frames_preds, frames_target, things, stuffs, allow_unknown_preds_category))


def synthetic_sequence(n, H, W, seed=0, n_inst=40, consistent=True, void=0.02, pred_void=0.0):
    """-> preds, target int64 [n, H, W, 2]: n frames of one scene, things = SYN_THINGS, stuffs = SYN_STUFFS.

    Target: stuff bands {0, 1} whose wavy border drifts from frame to frame, n_inst thing discs (categories 2-5) that keep their
    ids 1..n_inst while they move across the frames (wrapping at the borders; later discs occlude earlier ones), a `void`
    fraction of the pixels void (category SYN_VOID).  Prediction: the target's discs with radius and centre jittered by up to
    1 px (2 px from 512 px frames on), 10 % of them dropped per frame, 3 spurious discs per frame, a `pred_void` fraction of the
    pixels of category SYN_VOID (unknown: score with allow_unknown_preds_category=True).  consistent=True gives every fruit one
    prediction id over the whole sequence (ids permuted once into [1, 200)); consistent=False permutes the ids anew in every
    frame, which leaves the scene and each frame's per-image PQ exactly as they are and makes the scene PQ collapse."""
    if n_inst + 10 >= 200:
        raise ValueError("n_inst must be below 190")
    rng = np.random.default_rng(seed)
    S = min(H, W)
    r_lo, r_hi = max(3, S // 128), max(6, S // 25)
    jit = 2 if S >= 512 else 1
    cy0, cx0 = rng.uniform(0, H, n_inst), rng.uniform(0, W, n_inst)
    vy, vx = rng.uniform(-1, 1, n_inst) * S / 64, rng.uniform(-1, 1, n_inst) * S / 64
    r = rng.integers(r_lo, r_hi + 1, n_inst)
    c = rng.integers(2, 6, n_inst)
    perm = np.concatenate([[0], rng.permutation(np.arange(1, 200))])
    id_rng = np.random.default_rng([seed, 1])      # the per-frame permutations: both variants draw the same scene from rng
    preds = np.zeros((n, H, W, 2), dtype=np.int64)
    target = np.zeros((n, H, W, 2), dtype=np.int64)
    yy, xx = np.mgrid[0:H, 0:W]
    for f in range(n):
        band = ((yy + 12.0 * np.sin(xx / 37.0 + 0.2 * f)) // (H / 6.0)).astype(np.int64) % 2
        tc, ti = band.copy(), np.zeros((H, W), np.int64)
        pc, pi = band.copy(), np.zeros((H, W), np.int64)
        cy, cx = (cy0 + vy * f).astype(np.int64) % H, (cx0 + vx * f).astype(np.int64) % W
        keep = rng.random(n_inst) >= 0.10
        for k in range(n_inst):
            _paint_disc(tc, ti, cy[k], cx[k], r[k], c[k], k + 1)
            if keep[k]:
                dr = int(rng.integers(-jit, jit + 1))
                dy, dx = rng.integers(-jit, jit + 1, 2)
                _paint_disc(pc, pi, cy[k] + dy, cx[k] + dx, max(2, r[k] + dr), c[k], k + 1)
        for j in range(3):      # spurious instances
            _paint_disc(pc, pi, int(rng.integers(0, H)), int(rng.integers(0, W)), int(rng.integers(r_lo, r_hi + 1)),
                        int(rng.integers(2, 6)), n_inst + 1 + j)
        if not consistent:
            perm = np.concatenate([[0], id_rng.permutation(np.arange(1, 200))])
        pi = perm[pi]
        tv = rng.random((H, W)) < void
        tc[tv], ti[tv] = SYN_VOID, 0
        pv = rng.random((H, W)) < pred_void
        pc[pv], pi[pv] = SYN_VOID, 0
        preds[f, :, :, 0], preds[f, :, :, 1] = pc, pi
        target[f, :, :, 0], target[f, :, :, 1] = tc, ti
    return torch.from_numpy(preds), torch.from_numpy(target)
