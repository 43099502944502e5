"""CPU restatement of torchmetrics' PanopticQuality (the vendored utils/metrics/panoptic_quality.py of the reference, SURVEY 2.1)
-- TEST INFRASTRUCTURE ONLY.

It follows torchmetrics' functional steps: validate the inputs, parse the category sets, map category ids to continuous ids
(sorted things, then sorted stuffs), preprocess each map (stuff -> instance 0, unknown category -> the void colour
(1 + max category, 0)), then per image the colour areas of the prediction, of the target and of the (prediction, target) pairs
with torch.unique(..., return_counts=True), the IoU of every same-category pair with a non-void target, and the FP / FN counts
of the unmatched segments.  The per-colour dictionaries become arrays indexed by the colour's rank in torch.unique, which scores
a 1 MP frame in a fraction of a second.

Two choices, shared with the device path: the match and void-overlap decisions are taken on the exact integer areas
(2 |p∩t| > union, 2 |void ∩ s| <= |s|), and the IoU is computed in ``iou_dtype`` (float64 by default; float32 reproduces the
torchmetrics division of two int64 tensors).  For images under 2^23 pixels both choices give torchmetrics' decisions.

``synthetic_frames`` makes the seeded panoptic frames of tools/pq_bench.py and tests/test_gpu_metrics.py."""
import numpy as np
import torch


def parse_categories(things, stuffs):
    things, stuffs = set(things), set(stuffs)
    if not all(isinstance(v, int) and not isinstance(v, bool) for v in things | stuffs):
        raise TypeError("Expected arguments `things` and `stuffs` to contain integer category ids")
    if things & stuffs:
        raise ValueError(f"Expected arguments `things` and `stuffs` to have distinct keys, but got {things} and {stuffs}")
    if not (things or stuffs):
        raise ValueError("At least one of `things` and `stuffs` must be non-empty.")
    return things, stuffs


def validate_inputs(preds, target):
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


def continuous_ids(things, stuffs):
    return {c: i for i, c in enumerate(sorted(things) + sorted(stuffs))}


def void_color(things, stuffs):
    return (1 + max([0, *things, *stuffs]), 0)


def preprocess(x, things, stuffs, void, allow_unknown_category):
    """[B, *spatial, 2] -> [B, P, 2] int64 with stuff instances zeroed and unknown categories set to the void colour."""
    out = x.detach().to(torch.int64).clone().flatten(1, -2)
    cat = out[:, :, 0]
    is_stuff = torch.isin(cat, torch.tensor(sorted(stuffs), dtype=torch.int64))
    is_thing = torch.isin(cat, torch.tensor(sorted(things), dtype=torch.int64))
    out[:, :, 1][is_stuff] = 0
    known = is_stuff | is_thing
    if not allow_unknown_category and not bool(known.all()):
        raise ValueError(f"Unknown categories found: {sorted(set(cat[~known].tolist()))}")
    out[~known] = torch.tensor(void, dtype=torch.int64)
    return out


def _unique_colors(x):
    """torch.unique(x, dim=0, return_inverse=True, return_counts=True) for [P, 2] colours with category and instance in [0, 2^31),
    through one int64 key per colour (same order, several times faster than the row-wise unique)."""
    key, inv, cnt = torch.unique((x[:, 0] << 32) | x[:, 1], return_inverse=True, return_counts=True)
    return torch.stack([key >> 32, key & 0xFFFFFFFF], 1), inv, cnt


def update_sample(pred, tgt, cat_to_cont, void, iou_dtype=torch.float64):
    """One image: pred / tgt [P, 2] preprocessed -> iou_sum f64[K], tp, fp, fn i64[K]."""
    K = len(cat_to_cont)
    iou_sum = torch.zeros(K, dtype=torch.float64)
    tp, fp, fn = (torch.zeros(K, dtype=torch.int64) for _ in range(3))
    up, p_inv, p_area = _unique_colors(pred)
    ut, t_inv, t_area = _unique_colors(tgt)
    nt = ut.shape[0]
    code, inter = torch.unique(p_inv * nt + t_inv, return_counts=True)      # intersection areas of the colour pairs
    pi, ti = code // nt, code % nt
    vt = torch.nonzero((ut == torch.tensor(void)).all(1)).flatten()
    vp = torch.nonzero((up == torch.tensor(void)).all(1)).flatten()
    p_void = torch.zeros(up.shape[0], dtype=torch.int64)      # |p ∩ void_target|
    t_void = torch.zeros(nt, dtype=torch.int64)               # |void_pred ∩ t|
    if vt.numel():
        sel = ti == vt[0]
        p_void[pi[sel]] = inter[sel]
    if vp.numel():
        sel = pi == vp[0]
        t_void[ti[sel]] = inter[sel]
    cats = torch.tensor(sorted(cat_to_cont), dtype=torch.int64)
    conts = torch.tensor([cat_to_cont[c] for c in sorted(cat_to_cont)], dtype=torch.int64)

    def lut(c):      # category id -> continuous id (c known)
        return conts[torch.searchsorted(cats, c)]

    t_is_void = torch.zeros(nt, dtype=torch.bool)
    t_is_void[vt] = True
    p_is_void = torch.zeros(up.shape[0], dtype=torch.bool)
    p_is_void[vp] = True
    cand = ~t_is_void[ti] & (up[pi, 0] == ut[ti, 0])
    pi, ti, inter = pi[cand], ti[cand], inter[cand]
    union = p_area[pi] - p_void[pi] + t_area[ti] - inter
    matched = 2 * inter > union
    iou = inter.to(iou_dtype) / union.to(iou_dtype)
    cont = lut(ut[ti, 0])
    iou_sum.index_add_(0, cont[matched], iou[matched].to(torch.float64))
    tp.index_add_(0, cont[matched], torch.ones_like(cont[matched]))
    t_matched = torch.zeros(nt, dtype=torch.bool)
    t_matched[ti[matched]] = True
    p_matched = torch.zeros(up.shape[0], dtype=torch.bool)
    p_matched[pi[matched]] = True
    fn_sel = ~t_matched & ~t_is_void & (2 * t_void <= t_area)
    fn.index_add_(0, lut(ut[fn_sel, 0]), torch.ones(int(fn_sel.sum()), dtype=torch.int64))
    fp_sel = ~p_matched & ~p_is_void & (2 * p_void <= p_area)
    fp.index_add_(0, lut(up[fp_sel, 0]), torch.ones(int(fp_sel.sum()), dtype=torch.int64))
    return iou_sum, tp, fp, fn


def panoptic_quality_stats(preds, target, things, stuffs, allow_unknown_preds_category=False, iou_dtype=torch.float64):
    """-> iou_sum f64[K], tp, fp, fn i64[K] in continuous-id order (sorted things, then sorted stuffs), summed over the batch."""
    things, stuffs = parse_categories(things, stuffs)
    validate_inputs(preds, target)
    cat_to_cont = continuous_ids(things, stuffs)
    void = void_color(things, stuffs)
    p = preprocess(preds.cpu(), things, stuffs, void, allow_unknown_preds_category)
    t = preprocess(target.cpu(), things, stuffs, void, True)
    K = len(cat_to_cont)
    acc = [torch.zeros(K, dtype=torch.float64)] + [torch.zeros(K, dtype=torch.int64) for _ in range(3)]
    for b in range(p.shape[0]):
        for a, x in zip(acc, update_sample(p[b], t[b], cat_to_cont, void, iou_dtype)):
            a += x
    return tuple(acc)


def panoptic_quality_compute(iou_sum, tp, fp, fn):
    denominator = (tp + 0.5 * fp + 0.5 * fn).double()
    pq = torch.where(denominator > 0.0, iou_sum / denominator, 0.0)
    return torch.mean(pq[denominator > 0])


def panoptic_quality(preds, target, things, stuffs, allow_unknown_preds_category=False, iou_dtype=torch.float64):
    return panoptic_quality_compute(*panoptic_quality_stats(preds, target, things, stuffs, allow_unknown_preds_category, iou_dtype))


# ---------------------------------------------------------------------------------------------------------------------------
# seeded synthetic panoptic frames
# ---------------------------------------------------------------------------------------------------------------------------
SYN_STUFFS = (0, 1)
SYN_THINGS = (2, 3, 4, 5)
SYN_VOID = 9          # in neither set: void in the target


def _paint_disc(cat, inst, cy, cx, r, c, i, split_id=None):
    H, W = cat.shape
    y0, y1, x0, x1 = max(0, cy - r), min(H, cy + r + 1), max(0, cx - r), min(W, cx + r + 1)
    if y0 >= y1 or x0 >= x1:
        return
    yy, xx = np.mgrid[y0:y1, x0:x1]
    m = (yy - cy) ** 2 + (xx - cx) ** 2 <= r * r
    cat[y0:y1, x0:x1][m] = c
    ids = np.full(m.shape, i)
    if split_id is not None:
        ids[xx >= cx] = split_id
    inst[y0:y1, x0:x1][m] = ids[m]


def synthetic_frames(n, H, W, seed=0, n_inst=150):
    """-> preds, target int64 [n, H, W, 2] (category, instance), things = SYN_THINGS, stuffs = SYN_STUFFS.

    Target: stuff bands {0, 1} with wavy borders, ~n_inst thing discs of radius 8-40 px (categories 2-5, ids 1..n_inst),
    ~2 % of the pixels void (category SYN_VOID).  Prediction: the target's discs with radius and centre jittered by 1-3 px,
    10 % of them dropped, 5 % split in two down the middle, ~10 spurious discs, instance ids permuted into [1, 200); no void."""
    rng = np.random.default_rng(seed)
    preds = np.zeros((n, H, W, 2), dtype=np.int64)
    target = np.zeros((n, H, W, 2), dtype=np.int64)
    yy, xx = np.mgrid[0:H, 0:W]
    for f in range(n):
        band = ((yy + 12.0 * np.sin(xx / 37.0 + rng.uniform(0, 6.3))) // (H / 6.0)).astype(np.int64) % 2
        tc, ti = band.copy(), np.zeros((H, W), np.int64)
        pc, pi = band.copy(), np.zeros((H, W), np.int64)
        cy, cx = rng.integers(0, H, n_inst), rng.integers(0, W, n_inst)
        r = rng.integers(8, 41, n_inst)
        c = rng.integers(2, 6, n_inst)
        keep = rng.random(n_inst) >= 0.10
        split = rng.random(n_inst) < 0.05
        next_id = n_inst + 1
        for k in range(n_inst):
            _paint_disc(tc, ti, cy[k], cx[k], r[k], c[k], k + 1)
            if keep[k]:
                dr = int(rng.integers(1, 4)) * (1 if rng.random() < 0.5 else -1)
                dy, dx = rng.integers(-3, 4, 2)
                sid = None
                if split[k]:
                    sid, next_id = next_id, next_id + 1
                _paint_disc(pc, pi, cy[k] + dy, cx[k] + dx, max(2, r[k] + dr), c[k], k + 1, sid)
        for _ in range(10):      # spurious instances
            _paint_disc(pc, pi, int(rng.integers(0, H)), int(rng.integers(0, W)), int(rng.integers(8, 41)), int(rng.integers(2, 6)), next_id)
            next_id += 1
        perm = np.concatenate([[0], rng.permutation(np.arange(1, 200))])
        assert next_id <= 200
        pi = perm[pi]
        void = rng.random((H, W)) < 0.02
        tc[void], ti[void] = SYN_VOID, 0
        preds[f, :, :, 0], preds[f, :, :, 1] = pc, pi
        target[f, :, :, 0], target[f, :, :, 1] = tc, ti
    return torch.from_numpy(preds), torch.from_numpy(target)
