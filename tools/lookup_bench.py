"""Map-lookup benchmark: pagnerf_b200.mapping.map_index on the maps tools/components_bench.py builds, and lookup_rays / lookup_points
on a rendered 1 MP frame and on synthetic surface queries.

    python tools/lookup_bench.py [--ks 2,4] [--reps 20] [--check-k 2] [--out FILE]

Inputs:
  * index build: the map of bench.py's BASELINE config-2 field at each k (half of the points kept, as components_bench.py), and a
    planted-fruit map of the same size (components_bench.fruit_map).
  * lookup_rays: one 1024 x 1024 frame of bench.py's config-5 camera (make_frame_rays), rendered once in exact fp32 with depth, looked
    up in the index of the config-5 field's map at each k (half of the points kept), at radius 0, 1 and 2, with min_alpha = 0.5 and
    with min_alpha = 1e-6 (every ray the field touches is looked up).
  * lookup_points: 2^20 synthetic surface queries, map points moved by up to one lattice step per axis.
Prints one JSON line (and writes it to --out): CUDA-event ms (median of --reps warm runs), the table's bytes against the 126 MB L2, peak
memory growth, the fraction of rays resolved, and at --check-k the equality of lookup_rays with the CPU oracle (oracle/lookup.py).  The
card's name and power limit are read in the same process.
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.map_bench import card, timed, peak_growth      # noqa: E402
from tools.components_bench import fruit_map              # noqa: E402

L2_BYTES = 126 * 10 ** 6


def render_frame(wl, res=1024, chunk=131072):
    """-> origins, dirs [res^2, 3], depth, alpha [res^2, 1] of one exact-fp32 validation frame, and its ms (one warm run)."""
    from bench import make_frame_rays, NEAR, FAR
    from pagnerf_b200.wisp_compat import Rays
    o_np, d_np = make_frame_rays(res)
    dev = torch.device("cuda")
    o, d = torch.from_numpy(o_np).to(dev), torch.from_numpy(d_np).to(dev)
    wl.nef.decoder_precision = 'fp32'
    chans = ['rgb', 'depth', 'semantics', 'inst_embedding']

    def run():
        depth, alpha = [], []
        with torch.no_grad():
            for c0 in range(0, res * res, chunk):
                rb = wl.tracer(wl.nef, channels=chans, rays=Rays(origins=o[c0:c0 + chunk], dirs=d[c0:c0 + chunk], dist_min=NEAR,
                                                                  dist_max=FAR), lod_idx=None, stage='val')
                depth.append(rb.depth.float())
                alpha.append(rb.alpha.float())
        return torch.cat(depth).contiguous(), torch.cat(alpha).contiguous()

    ms, (depth, alpha) = timed(run, 3)
    return o, d, depth, alpha, ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="2,4")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--check-k", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lookup_bench needs a CUDA device")
    import bench
    from pagnerf_b200 import build
    from pagnerf_b200.mapping import extract_panoptic_map, instance_components, map_index, lookup_points, lookup_rays
    build.build()
    dev = torch.device("cuda:0")
    name, power = card()
    res = {"tool": "tools/lookup_bench.py", "gpu": name, "power_limit": power, "l2_bytes": L2_BYTES, "index": [], "rays": [],
           "points": []}
    ks = [int(x) for x in args.ks.split(",")]
    # index builds
    nef = bench.Workload(dev, n_rays=4096, seed=0, n_batches=1, config=2).nef
    level = int(nef.grid.blas_level)
    Ci, Cs = int(nef.num_instances), int(nef.num_classes)
    thr = float(torch.quantile(extract_panoptic_map(nef, 1, min_density=-1.0).density, 0.5))
    for k in ks:
        field = extract_panoptic_map(nef, k, min_density=thr)
        fruit, n_balls = fruit_map(field.xyz.shape[0], k, level)
        for kind, pts in (("field", field), ("fruit", fruit)):
            run = lambda: map_index(pts, samples_per_axis=k, level=level)
            ms, index = timed(run, args.reps)
            mem, _ = peak_growth(run)
            C = index.keys.numel()
            res["index"].append({"input": kind, "k": k, "points": int(pts.xyz.shape[0]), "slots": C, "ms": round(ms, 3),
                                 "points_per_s": round(pts.xyz.shape[0] / (ms * 1e-3), 1), "table_mb": round(12 * C / 2 ** 20, 1),
                                 "key_bytes_exceed_l2": 8 * C > L2_BYTES, "peak_mem_growth_mb": round(mem / 2 ** 20, 1)})
            print(json.dumps(res["index"][-1]), file=sys.stderr)
        del field, fruit
    del nef
    # a rendered frame of config 5, looked up in its field's maps
    wl = bench.Workload(dev, n_rays=4096, seed=0, n_batches=1, config=5)
    o, d, depth, alpha, render_ms = render_frame(wl)
    res["frame"] = {"rays": int(o.shape[0]), "render_fp32_ms": round(render_ms, 3), "alpha_ge_0.5": float((alpha >= 0.5).float().mean()),
                    "alpha_gt_0": float((alpha > 0).float().mean())}
    level = int(wl.nef.grid.blas_level)
    thr5 = float(torch.quantile(extract_panoptic_map(wl.nef, 1, min_density=-1.0).density, 0.5))
    for k in ks:
        pts = extract_panoptic_map(wl.nef, k, min_density=thr5)
        comps = instance_components(pts, samples_per_axis=k, level=level, num_instances=Ci, num_classes=Cs)
        index = map_index(pts, samples_per_axis=k, level=level)
        C = index.keys.numel()
        for radius in (0, 1, 2):
            for min_alpha in (0.5, 1e-6):
                run = lambda: lookup_rays(index, o, d, depth, alpha, radius=radius, min_alpha=min_alpha, component=comps.component)
                ms, hit = timed(run, args.reps)
                mem, _ = peak_growth(run)
                row = {"k": k, "map_points": int(pts.xyz.shape[0]), "slots": C, "key_bytes_exceed_l2": 8 * C > L2_BYTES,
                       "radius": radius, "min_alpha": min_alpha, "ms": round(ms, 4), "share_of_frame": round(ms / render_ms, 5),
                       "resolved_point": float((hit.point >= 0).float().mean()), "resolved_object": float((hit.object >= 0).float().mean()),
                       "peak_mem_growth_mb": round(mem / 2 ** 20, 2)}
                if k == args.check_k and radius == 1:
                    from oracle import lookup as ol
                    idx = ol.index(pts.xyz.cpu().numpy(), k, level)
                    wp, wo = ol.lookup_rays(idx, o.cpu().numpy(), d.cpu().numpy(), depth.cpu().numpy(), alpha.cpu().numpy(), radius,
                                            min_alpha, comps.component.cpu().numpy())
                    row["oracle_equal"] = bool(np.array_equal(hit.point.cpu().numpy(), wp) and np.array_equal(hit.object.cpu().numpy(), wo))
                res["rays"].append(row)
                print(json.dumps(row), file=sys.stderr)
        # 2^20 synthetic surface queries: map points moved by up to one lattice step per axis
        g = torch.Generator(device=dev).manual_seed(k)
        Q = 1 << 20
        pick = torch.randint(0, pts.xyz.shape[0], (Q,), generator=g, device=dev)
        D = k << level
        q = (pts.xyz[pick] + (torch.rand(Q, 3, generator=g, device=dev) * 2 - 1) * (2.0 / D)).contiguous()
        for radius in (0, 1, 2):
            ms, hit = timed(lambda: lookup_points(index, q, radius=radius, component=comps.component), args.reps)
            res["points"].append({"k": k, "queries": Q, "radius": radius, "ms": round(ms, 4),
                                  "resolved_point": float((hit.point >= 0).float().mean())})
            print(json.dumps(res["points"][-1]), file=sys.stderr)
        del pts, comps, index
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
