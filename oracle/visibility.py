"""Oracle: per-object visibility of a map in camera views (pagnerf_b200.mapping.object_visibility) on the CPU.  TEST INFRASTRUCTURE
ONLY.

Built on oracle/projection.py, whose footprints are the device's bit for bit: `visible` and `bbox` come from the object image of
`project`, `silhouette` from the (pixel, key) pairs of `pixel_pairs` mapped to (object, pixel) and reduced with np.unique.
"""
import numpy as np

from . import projection as op


def visibility(xyz, k, level, view, intrinsics, H, W, component, K, max_radius=8, near=0.01):
    """-> (visible i64 [B, K], silhouette i64 [B, K], bbox i32 [B, K, 4]) by the definitions"""
    x = np.asarray(xyz, np.float32).reshape(-1, 3)
    comp = np.asarray(component, np.int64).reshape(-1)
    V = np.asarray(view, np.float32).reshape(-1, 4, 4)
    Kc = np.asarray(intrinsics, np.float32).reshape(-1, 4)
    B = V.shape[0]
    visible = np.zeros((B, K), np.int64)
    silhouette = np.zeros((B, K), np.int64)
    bbox = np.full((B, K, 4), -1, np.int32)
    _, _, obj = op.project(x, k, level, V, Kc, H, W, max_radius, near, comp)
    h = op.half_size(k, level)
    for b in range(B):
        rows, cols = np.nonzero(obj[b] >= 0)
        o = obj[b][rows, cols]
        visible[b] = np.bincount(o, minlength=K)
        for a, v, red in ((0, cols, np.minimum), (1, rows, np.minimum), (2, cols, np.maximum), (3, rows, np.maximum)):
            col = np.full(K, np.iinfo(np.int32).max if red is np.minimum else -1, np.int64)
            red.at(col, o, v)
            bbox[b, :, a] = np.where(visible[b] > 0, col, -1)
        pix, key = op.pixel_pairs(x, V[b], Kc[b], H, W, h, near, max_radius)
        po = comp[(key & np.uint64(0xFFFFFFFF)).astype(np.int64)] if pix.size else np.zeros(0, np.int64)
        own = po >= 0
        pairs = np.unique(po[own] * (H * W) + pix[own])
        silhouette[b] = np.bincount(pairs // (H * W), minlength=K)
    return visible, silhouette, bbox
