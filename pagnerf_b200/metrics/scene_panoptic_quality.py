"""Scene-level panoptic quality on the device: every (category, instance) id is ONE segment over all frames of a sequence.

    spq = ScenePanopticQuality(things={0, 1}, stuffs={6, 7}).to(device)
    for pred, target in frames:
        spq.update(pred, target)     # [B, *spatial, 2] (category, instance) integer maps: one kernel, no host synchronisation
    spq.sync()                       # frames sharded across ranks: every rank then holds the union of all ranks' tables
    spq.compute()                    # float64 0-dim PQ of the scene so far: one device-to-host read; updates may continue after it
    iou_sum, tp, fp, fn = spq.stats()        # per category, continuous-id order: sorted(things) then sorted(stuffs)

Definition: after updates with frames F1..Fn, ScenePanopticQuality returns what PanopticQuality returns for ONE image made of all
pixels of F1..Fn concatenated.  Every rule is the one PanopticQuality's docstring states: stuff pixels get instance 0; pixels of a
category in neither set are void (in the prediction only with allow_unknown_preds_category, otherwise an error); a prediction and a
target segment of the same category match when IoU = |p∩t| / (|p| - |p ∩ void_t| + |t| - |p∩t|) > 0.5, decided on the exact
integers; the void-overlap rule decides FP and FN; PQ is the mean over the categories with tp + fp + fn > 0.  So a (category,
instance) pair is one segment wherever it appears, each stuff category is one segment per scene, and the result depends neither on
frame order, frame sizes nor on how the frames are split into update calls.  Areas are 64-bit (a long sequence exceeds 2^32
pixels); each IoU is float64 from the exact integer areas.  This is the idea of Panoptic Lifting's scene-level PQ; parity with
its evaluation code is not claimed.

Per-image PQ cannot see whether ids are consistent across frames: a prediction that calls a fruit 3 in one frame and 17 in the
next scores like one that keeps its id.  Here the two ids are two segments of the scene, and at most one of them can match.

Tables: three open-addressing tables (prediction segments, target segments, same-category pairs) of C = pag_hash_slots(capacity)
slots, 64 B per slot in all: 32 MiB at the default capacity 2^18.  Each table admits at most `capacity` distinct keys; the pixels
of a key beyond that are refused and counted, and compute() raises ValueError naming the table, the refused pixels and a capacity
that suffices.  keys_used() says how full the tables are.  Errors only the device sees (unknown prediction categories, thing
instance ids outside [0, 2^31)) are counted there and raised by compute(), as in PanopticQuality.
"""
import math

import torch
import torch.distributed as dist
from torch import nn

from .._lib import call, ptr, query_i64
from .panoptic_quality import _as_i64_rows, _parse_categories, _validate_inputs

MAX_CAPACITY = 1 << 26
TABLES = ("prediction segment", "target segment", "pair")
_COUNTERS = 16      # u64 counters at the end of the workspace: reserved[3] | used[3] | refused[3] | padding


class ScenePanopticQuality(nn.Module):
    def __init__(self, things, stuffs, allow_unknown_preds_category=False, capacity=1 << 18):
        super().__init__()
        things, stuffs = _parse_categories(things, stuffs)
        if not isinstance(capacity, int) or isinstance(capacity, bool):
            raise TypeError(f"Expected `capacity` to be an integer, got {type(capacity).__name__}")
        if not 1 <= capacity <= MAX_CAPACITY:
            raise ValueError(f"Expected `capacity` in [1, 2^26], got {capacity}")
        self.things, self.stuffs = things, stuffs
        self.allow_unknown_preds_category = bool(allow_unknown_preds_category)
        self.capacity = capacity
        order = sorted(things) + sorted(stuffs)
        self.cat_id_to_continuous_id = {c: i for i, c in enumerate(order)}
        self.num_categories = len(order)
        by_id = sorted(order)
        code = [self.cat_id_to_continuous_id[c] | (0x100 if c in things else 0) for c in by_id]
        self.register_buffer("cat_ids", torch.tensor(by_id, dtype=torch.int32), persistent=False)
        self.register_buffer("cat_code", torch.tensor(code, dtype=torch.int32), persistent=False)
        self.register_buffer("errors", torch.zeros(2, dtype=torch.int64), persistent=False)      # unknown preds | bad instance ids
        self._workspace = None      # the scene's tables, zero-filled once; they persist across updates

    def extra_repr(self):
        return (f"things={sorted(self.things)}, stuffs={sorted(self.stuffs)}, "
                f"allow_unknown_preds_category={self.allow_unknown_preds_category}, capacity={self.capacity}")

    def _device(self):
        return self.errors.device if self.errors.is_cuda else torch.device("cuda", torch.cuda.current_device())

    def _tables(self, device=None):
        device = device or self._device()
        ws = self._workspace
        if ws is None or ws.device != device:
            ws = self._workspace = torch.zeros(query_i64("pag_scene_pq_workspace", self.capacity), dtype=torch.uint8, device=device)
        return ws

    def _counters(self):
        """-> i64[3, 3] view of the workspace's counters (reserved | used | refused, each in TABLES order)."""
        return self._tables()[-8 * _COUNTERS:].view(torch.int64)[:9].view(3, 3)

    def reset(self):
        """Empty the tables and the error counts."""
        self.errors.zero_()
        if self._workspace is not None:
            self._workspace.zero_()

    @torch.no_grad()
    def update(self, preds, target):
        """Add a batch of [B, *spatial, 2] CUDA integer maps to the scene: one launch, no host synchronisation."""
        _validate_inputs(preds, target)
        B, P = preds.shape[0], math.prod(preds.shape[1:-1])
        if B == 0 or P == 0:
            return
        dev = preds.device
        if self.errors.device != dev:
            self.to(dev)
        p, t = _as_i64_rows(preds, B, P), _as_i64_rows(target, B, P)
        ws = self._tables(dev)
        call("pag_scene_pq_update", ptr(p), ptr(t), B * P, ptr(self.cat_ids), ptr(self.cat_code), self.num_categories,
             int(self.allow_unknown_preds_category), ptr(ws), self.capacity, ws.numel(), ptr(self.errors))

    def forward(self, preds, target):
        """update(); a scene has no per-batch PQ, so nothing is returned."""
        self.update(preds, target)

    @torch.no_grad()
    def stats(self):
        """-> iou_sum f64[K], tp, fp, fn i64[K] of the scene so far (device tensors) in continuous-id order: sorted(things), sorted(stuffs).
        Leaves the tables as they were; errors are raised by compute()."""
        dev = self._device()
        K = self.num_categories
        iou_sum = torch.zeros(K, dtype=torch.float64, device=dev)
        counts = torch.zeros(3, K, dtype=torch.int64, device=dev)
        ws = self._tables(dev)
        call("pag_scene_pq_stats", ptr(ws), self.capacity, ws.numel(), K, ptr(iou_sum), ptr(counts))
        return iou_sum, counts[0], counts[1], counts[2]

    def keys_used(self):
        """-> i64[3] distinct keys in the prediction-segment, target-segment and pair tables (device tensor); each is at most capacity."""
        return self._counters()[1].clone()

    @torch.no_grad()
    def compute(self):
        """float64 0-dim PQ of the scene so far (one device-to-host read); raises ValueError for errors counted on the device."""
        iou_sum, tp, fp, fn = self.stats()
        tp, fp, fn = tp.double(), fp.double(), fn.double()
        den = tp + 0.5 * fp + 0.5 * fn
        valid = den > 0
        pq = torch.where(valid, iou_sum / den, 0.0).sum() / valid.sum()      # 0 / 0 = NaN: no category
        host = torch.cat([self.errors, self._counters()[1:].flatten()]).cpu().tolist()
        unknown, bad, used, refused = host[0], host[1], host[2:5], host[5:8]
        if unknown:
            raise ValueError(f"Unknown categories found in `preds`: {unknown} pixels of a category in neither `things` nor `stuffs` "
                             "(pass allow_unknown_preds_category=True to treat them as void)")
        if bad:
            raise ValueError(f"{bad} pixels of a `things` category have an instance id outside [0, 2^31)")
        if any(refused):
            # each refused pixel adds at most one key; refused segments also withheld their pairs
            need = max(used[0] + refused[0], used[1] + refused[1], used[2] + refused[2] + refused[0] + refused[1])
            full = [f"the {TABLES[i]} table refused {refused[i]} pixels ({used[i]} of {self.capacity} keys used)"
                    for i in range(3) if refused[i]]
            raise ValueError(f"ScenePanopticQuality tables full: {'; '.join(full)}. "
                             f"A capacity of {min(need, MAX_CAPACITY)} suffices; reset() and update with a larger `capacity`")
        return pq

    @torch.no_grad()
    def sync(self, group=None):
        """Union of the tables of all ranks of `group` on every rank (a segment seen on two ranks becomes one segment with the
        summed area), and the summed error counts.  Call once before compute(); a no-op without an initialised process group."""
        if not (dist.is_available() and dist.is_initialized()):
            return
        ws = self._tables()
        gathered = [torch.empty_like(ws) for _ in range(dist.get_world_size(group))]
        dist.all_gather(gathered, ws, group=group)
        me = dist.get_rank(group)
        for r, other in enumerate(gathered):
            if r != me:
                call("pag_scene_pq_merge", ptr(ws), ptr(other), self.capacity, ws.numel())
        dist.all_reduce(self.errors, op=dist.ReduceOp.SUM, group=group)
