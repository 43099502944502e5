"""Panoptic quality (PQ) on the device: drop-in for the vendored torchmetrics PanopticQuality (utils/metrics/panoptic_quality.py),
which evaluate_metrics (pc_nerf/trainer.py:651-941) uses to score the argmax label maps of a validation render.

    pq = PanopticQuality(things={0, 1}, stuffs={6, 7}).to(device)
    pq(preds, target)            # [B, *spatial, 2] (category, instance) integer maps: this batch's PQ, accumulated as well
    pq.update(preds, target)     # accumulate only: three kernels (csrc/metrics.cu), no host synchronisation, graph capturable
    pq.compute()                 # float64 0-dim PQ of everything accumulated since reset(): one device-to-host read
    iou_sum, tp, fp, fn = pq.stats()     # per category, continuous-id order: sorted(things) then sorted(stuffs)
    pq.sync()                    # sum the statistics over torch.distributed ranks (images sharded across ranks)

Semantics are torchmetrics', applied per image (segments never cross images): stuff pixels get instance 0, pixels of a category in
neither set are void (always allowed in the target, in the prediction only with allow_unknown_preds_category); a prediction
segment p and a target segment t of the same category, t not void, match when
IoU = |p∩t| / (|p| - |p ∩ void_target| + |t| - |p∩t|) > 0.5; an unmatched target segment is a false negative unless more than
half of it is void in the prediction, an unmatched prediction segment a false positive unless more than half of it is void in the
target; PQ = mean over the categories with tp + fp + fn > 0 of iou_sum / (tp + fp/2 + fn/2), NaN when there are none.

Parity: the vendored file is not available in this tree; the restatement in oracle/metrics.py follows torchmetrics' functions and
reproduces the docstring example (PQ 0.5463).  Each IoU is computed here in float64 from the exact integer areas, and the match
decision is taken on the integers.  torchmetrics divides two int64 area tensors, which gives torch's default float32: that moves
iou_sum by at most ~6e-8 relative per match, and changes no match decision for images under 2^23 pixels (there an IoU above 0.5 is at
least 2^-24 above it).  Beyond the docstring example, parity with torchmetrics is unpinned.

One documented difference: errors that only the device can see -- a prediction pixel of an unknown category while
allow_unknown_preds_category=False, a thing pixel whose instance id lies outside [0, 2^31) -- are counted on the device and raised
as ValueError by compute() / __call__ (torchmetrics raises inside update).  The count stays in the state until reset().
"""
import math

import torch
import torch.distributed as dist
from torch import nn

from .._lib import call, ptr, query_i64

MAX_CATEGORIES = 256                 # len(things) + len(stuffs); the category table lives in shared memory
MAX_PIXELS_PER_IMAGE = 1 << 30
WORKSPACE_BUDGET = 256 << 20         # hash tables of several images per launch up to this size; always at least one image


def _parse_categories(things, stuffs):
    things, stuffs = set(things), set(stuffs)
    if not all(isinstance(v, int) and not isinstance(v, bool) for v in things | stuffs):
        raise TypeError("Expected arguments `things` and `stuffs` to contain integer category ids")
    if things & stuffs:
        raise ValueError(f"Expected arguments `things` and `stuffs` to have distinct keys, but got {things} and {stuffs}")
    if not (things or stuffs):
        raise ValueError("At least one of `things` and `stuffs` must be non-empty.")
    if not all(0 <= v < 2 ** 31 for v in things | stuffs):
        raise ValueError("Expected category ids in [0, 2^31)")
    if len(things) + len(stuffs) > MAX_CATEGORIES:
        raise ValueError(f"At most {MAX_CATEGORIES} categories are supported, got {len(things) + len(stuffs)}")
    return things, stuffs


def _validate_inputs(preds, target):
    if not isinstance(preds, torch.Tensor) or not isinstance(target, torch.Tensor):
        raise TypeError("Expected arguments `preds` and `target` to be tensors")
    if preds.shape != target.shape:
        raise ValueError(f"Expected arguments `preds` and `target` to have the same shape, but got {preds.shape} and {target.shape}")
    if preds.dim() < 3:
        raise ValueError("Expected arguments `preds` and `target` to have at least one spatial dimension (B, *spatial, 2)")
    if preds.shape[-1] != 2:
        raise ValueError("Expected arguments `preds` and `target` to have the last dimension of size 2 (category, instance)")
    for t in (preds, target):
        if t.is_floating_point() or t.is_complex() or t.dtype == torch.bool:
            raise TypeError(f"Expected integer category / instance ids, but got dtype {t.dtype}")
    if not (preds.is_cuda and target.is_cuda):
        raise RuntimeError("pagnerf_b200 metrics run on CUDA tensors only (no CPU fallback)")
    if preds.device != target.device:
        raise ValueError(f"Expected `preds` and `target` on the same device, got {preds.device} and {target.device}")


def _as_i64_rows(x, B, P):
    """[B, *spatial, 2] integer -> contiguous, 16-byte aligned int64 [B, P, 2] (a copy only when needed)."""
    x = x.to(torch.int64).reshape(B, P, 2)
    if not x.is_contiguous() or x.data_ptr() % 16:
        x = x.clone(memory_format=torch.contiguous_format)
    return x


class PanopticQuality(nn.Module):
    def __init__(self, things, stuffs, allow_unknown_preds_category=False):
        super().__init__()
        things, stuffs = _parse_categories(things, stuffs)
        self.things, self.stuffs = things, stuffs
        self.allow_unknown_preds_category = bool(allow_unknown_preds_category)
        order = sorted(things) + sorted(stuffs)
        self.cat_id_to_continuous_id = {c: i for i, c in enumerate(order)}
        K = self.num_categories = len(order)
        by_id = sorted(order)
        code = [self.cat_id_to_continuous_id[c] | (0x100 if c in things else 0) for c in by_id]
        self.register_buffer("cat_ids", torch.tensor(by_id, dtype=torch.int32), persistent=False)
        self.register_buffer("cat_code", torch.tensor(code, dtype=torch.int32), persistent=False)
        self.register_buffer("iou_sum", torch.zeros(K, dtype=torch.float64), persistent=False)
        self.register_buffer("counts", torch.zeros(3, K, dtype=torch.int64), persistent=False)      # tp | fp | fn
        self.register_buffer("errors", torch.zeros(2, dtype=torch.int64), persistent=False)         # unknown preds | bad instance ids
        self._workspace = None      # zero-filled; every update leaves it zeroed

    def extra_repr(self):
        return f"things={sorted(self.things)}, stuffs={sorted(self.stuffs)}, allow_unknown_preds_category={self.allow_unknown_preds_category}"

    def reset(self):
        self.iou_sum.zero_()
        self.counts.zero_()
        self.errors.zero_()

    def _workspace_for(self, B, P, device):
        per_image = query_i64("pag_pq_workspace", 1, P)
        G = int(max(1, min(B, 65535, WORKSPACE_BUDGET // per_image)))
        need = query_i64("pag_pq_workspace", G, P)
        ws = self._workspace
        if ws is None or ws.device != device or ws.numel() < need:
            ws = self._workspace = torch.zeros(need, dtype=torch.uint8, device=device)
        return ws, G

    @torch.no_grad()
    def update(self, preds, target):
        """Accumulate the statistics of a batch of [B, *spatial, 2] CUDA integer maps; no host synchronisation."""
        _validate_inputs(preds, target)
        B, P = preds.shape[0], math.prod(preds.shape[1:-1])
        if B == 0 or P == 0:
            return
        if P > MAX_PIXELS_PER_IMAGE:
            raise ValueError(f"At most 2^30 pixels per image are supported, got {P}")
        dev = preds.device
        if self.iou_sum.device != dev:
            self.to(dev)
        p, t = _as_i64_rows(preds, B, P), _as_i64_rows(target, B, P)
        ws, G = self._workspace_for(B, P, dev)
        for b0 in range(0, B, G):
            b1 = min(B, b0 + G)
            call("pag_pq_update", ptr(p[b0:b1]), ptr(t[b0:b1]), b1 - b0, P, ptr(self.cat_ids), ptr(self.cat_code), self.num_categories,
                 int(self.allow_unknown_preds_category), ptr(ws), ws.numel(), ptr(self.iou_sum), ptr(self.counts), ptr(self.errors))

    def stats(self):
        """-> iou_sum f64[K], tp, fp, fn i64[K] (device tensors, copies) in continuous-id order: sorted(things), sorted(stuffs)."""
        return self.iou_sum.clone(), self.counts[0].clone(), self.counts[1].clone(), self.counts[2].clone()

    @torch.no_grad()
    def compute(self):
        """float64 0-dim PQ over everything accumulated since reset(); raises ValueError for errors counted on the device."""
        tp, fp, fn = self.counts.double()
        den = tp + 0.5 * fp + 0.5 * fn
        valid = den > 0
        pq = torch.where(valid, self.iou_sum / den, 0.0).sum() / valid.sum()      # 0 / 0 = NaN: no category
        unknown, bad = self.errors.cpu().tolist()
        if unknown:
            raise ValueError(f"Unknown categories found in `preds`: {unknown} pixels of a category in neither `things` nor `stuffs` "
                             "(pass allow_unknown_preds_category=True to treat them as void)")
        if bad:
            raise ValueError(f"{bad} pixels of a `things` category have an instance id outside [0, 2^31)")
        return pq

    def forward(self, preds, target):
        """Accumulate the batch and return the PQ of this batch alone (torchmetrics' forward)."""
        if isinstance(preds, torch.Tensor) and preds.is_cuda and self.iou_sum.device != preds.device:
            self.to(preds.device)
        saved = (self.iou_sum.clone(), self.counts.clone(), self.errors.clone())
        self.reset()
        try:
            self.update(preds, target)
            return self.compute()
        finally:
            for s, x in zip((self.iou_sum, self.counts, self.errors), saved):
                s += x.to(s.device)

    @torch.no_grad()
    def sync(self, group=None):
        """Sum iou_sum, tp, fp, fn (and the error counts) over the ranks of `group`; a no-op without an initialised process group."""
        if not (dist.is_available() and dist.is_initialized()):
            return
        for x in (self.iou_sum, self.counts, self.errors):
            dist.all_reduce(x, op=dist.ReduceOp.SUM, group=group)
