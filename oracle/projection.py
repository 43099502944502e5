"""Oracle: z-buffered splatting of a map into camera views (pagnerf_b200.mapping.project_map) on the CPU.  TEST INFRASTRUCTURE ONLY.

Restates the definitions of pagnerf_b200/mapping/panoptic_map.py in float32 numpy.  numpy evaluates every float32 operation
separately rounded, in the order written, so the transform, the pixel positions and the footprints are the device's bit for bit.
`project` expands each point's rectangle to (pixel, key) pairs and reduces them with np.minimum.at on a u64 buffer, the device's
depth buffer; `brute_force` tests every point against every pixel with scalar arithmetic, for tiny inputs.
"""
import numpy as np

EMPTY = np.uint64(0xFFFFFFFFFFFFFFFF)


def half_size(k, level):
    """h = fl(1 / D), D = k << level"""
    return np.float32(1.0) / np.float32(int(k) << int(level))


def footprints(xyz, view, intrinsics, h, near, max_radius):
    """One camera (view [4, 4], intrinsics (fx, fy, cx, cy)) -> z, u, v, su, sv (f32 [P]) and ok (bool [P]: the point is projected)."""
    f32 = np.float32
    x = np.asarray(xyz, f32).reshape(-1, 3)
    V = np.asarray(view, f32).reshape(4, 4)
    fx, fy, cx, cy = (f32(c) for c in np.asarray(intrinsics, f32).reshape(4))
    with np.errstate(all="ignore"):
        p = [((V[q, 0] * x[:, 0] + V[q, 1] * x[:, 1]) + V[q, 2] * x[:, 2]) + V[q, 3] for q in range(3)]
        z = -p[2]
        u = fx * (p[0] / z) + cx
        v = fy * (p[1] / z) + cy
        R = f32(max_radius)
        su = np.minimum((fx * f32(h)) / z, R)
        sv = np.minimum((fy * f32(h)) / z, R)
        ok = (z > f32(near)) & np.isfinite(u) & np.isfinite(v) & (su >= 0) & (sv >= 0)
    return z, u, v, su, sv, ok


def keys(z, n):
    """(z bits << 32) | point index, u64"""
    return (np.asarray(z, np.float32).view(np.uint32).astype(np.uint64) << np.uint64(32)) | np.arange(n, dtype=np.uint64)


def rectangles(u, v, su, sv, H, W, ok):
    """-> c0, c1, r0, r1 (i64) and nonempty (bool): the covered columns / rows of the projected points (ok), clamped to the image in
    float and tested for emptiness before the conversion to integers"""
    with np.errstate(all="ignore"):
        c0 = np.maximum(np.floor(u - su), np.float32(0))
        c1 = np.minimum(np.floor(u + su), np.float32(W - 1))
        r0 = np.maximum(np.floor(v - sv), np.float32(0))
        r1 = np.minimum(np.floor(v + sv), np.float32(H - 1))
        nonempty = ok & (c0 <= c1) & (r0 <= r1)
    i = lambda a: np.where(nonempty, a, 0).astype(np.int64)
    return i(c0), i(c1), i(r0), i(r1), nonempty


def pixel_pairs(xyz, view, intrinsics, H, W, h, near, max_radius):
    """One camera -> (pixel i64 [M], key u64 [M]): every (covered pixel, point key) pair"""
    x = np.asarray(xyz, np.float32).reshape(-1, 3)
    z, u, v, su, sv, ok = footprints(x, view, intrinsics, h, near, max_radius)
    c0, c1, r0, r1, nonempty = rectangles(u, v, su, sv, H, W, ok)
    idx = np.nonzero(nonempty)[0]
    nc, nr = (c1 - c0 + 1)[idx], (r1 - r0 + 1)[idx]
    n = nc * nr
    rep = np.repeat(np.arange(idx.size), n)
    off = np.arange(int(n.sum()), dtype=np.int64) - np.repeat(np.cumsum(n) - n, n)
    col = c0[idx][rep] + off % nc[rep]
    row = r0[idx][rep] + off // nc[rep]
    return row * W + col, keys(z, x.shape[0])[idx][rep]


def project(xyz, k, level, view, intrinsics, H, W, max_radius=8, near=0.01, component=None):
    """-> (point i64 [B,H,W], depth f32 [B,H,W], object i64 [B,H,W] or None) by the definitions"""
    h = half_size(k, level)
    V = np.asarray(view, np.float32).reshape(-1, 4, 4)
    K = np.asarray(intrinsics, np.float32).reshape(-1, 4)
    B = V.shape[0]
    buf = np.full((B, H * W), EMPTY, np.uint64)
    for b in range(B):
        pix, key = pixel_pairs(xyz, V[b], K[b], H, W, h, near, max_radius)
        np.minimum.at(buf[b], pix, key)
    return decode(buf.reshape(B, H, W), component)


def decode(buf, component=None):
    hit = buf != EMPTY
    point = np.where(hit, (buf & np.uint64(0xFFFFFFFF)).astype(np.int64), -1)
    depth = np.where(hit, (buf >> np.uint64(32)).astype(np.uint32).view(np.float32), np.float32(np.inf)).astype(np.float32)
    obj = None
    if component is not None:
        component = np.asarray(component, np.int64)
        obj = np.where(hit, component[np.maximum(point, 0)] if component.size else -1, -1)
    return point, depth, obj


def brute_force(xyz, k, level, view, intrinsics, H, W, max_radius=8, near=0.01):
    """Every point against every pixel, scalar float32 arithmetic: point i64 [B,H,W] (tiny inputs only)"""
    f32 = np.float32
    h = half_size(k, level)
    x = np.asarray(xyz, f32).reshape(-1, 3)
    V = np.asarray(view, f32).reshape(-1, 4, 4)
    K = np.asarray(intrinsics, f32).reshape(-1, 4)
    out = np.full((V.shape[0], H, W), -1, np.int64)
    with np.errstate(all="ignore"):
        for b in range(V.shape[0]):
            fx, fy, cx, cy = K[b]
            best = {}
            for i in range(x.shape[0]):
                p = []
                for q in range(3):
                    s = V[b, q, 0] * x[i, 0]
                    s = s + V[b, q, 1] * x[i, 1]
                    s = s + V[b, q, 2] * x[i, 2]
                    p.append(s + V[b, q, 3])
                z = -p[2]
                u, v = fx * (p[0] / z) + cx, fy * (p[1] / z) + cy
                ru, rv = (fx * h) / z, (fy * h) / z
                if not (z > f32(near) and np.isfinite(u) and np.isfinite(v) and ru >= 0 and rv >= 0):
                    continue
                su, sv = min(ru, f32(max_radius)), min(rv, f32(max_radius))
                lo_c, hi_c, lo_r, hi_r = np.floor(u - su), np.floor(u + su), np.floor(v - sv), np.floor(v + sv)
                for r in range(H):
                    for c in range(W):
                        covers = lo_c <= c <= hi_c and lo_r <= r <= hi_r
                        if covers and ((r, c) not in best or (z, i) < best[(r, c)]):
                            best[(r, c)] = (z, i)
            for (r, c), (_, i) in best.items():
                out[b, r, c] = i
    return out
