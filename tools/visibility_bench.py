"""Per-object visibility benchmark: pagnerf_b200.mapping.object_visibility against project_map on the same inputs, on the maps and
views of tools/project_bench.py.

    python tools/visibility_bench.py [--ks 2,4] [--reps 10] [--check-k 2] [--out FILE]

Inputs (as project_bench.py): the map of bench.py's BASELINE config-2 field at each k (half of the points kept) split into
objects by instance_components, and a planted-fruit map of the same size (components_bench.fruit_map, one object per ball);
config 5's 1024 x 1024 camera (B = 1) and the 42 cameras of bench.make_cameras (B = 42), max_radius 8.
Prints one JSON line (and writes it to --out): per input and view count the median CUDA-event ms of object_visibility and of
project_map (with component) over --reps warm runs in the same process and their ratio, the kernels' time from a separate
torch.profiler run, the silhouette rounds and bitmap bytes, peak memory growth, and at --check-k the integer equality with the
CPU oracle (oracle/visibility.py) on a 256 x 256 view.  The card's name and power limit are read in the same process.
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
from tools.project_bench import MAX_RADIUS, frame_camera  # noqa: E402

KERNELS = {"map_project_splat_kernel": "splat", "map_vis_visible_kernel": "visible", "map_vis_box_kernel": "box",
           "map_vis_init_kernel": "pairs", "map_vis_pairs_kernel": "pairs", "exclusive_scan_kernel": "scan",
           "map_vis_or_kernel": "silhouette_or", "map_vis_popc_kernel": "silhouette_popcount", "Memset": "fills"}


def stage_ms(run, reps):
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            run()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        name = next((s for key, s in KERNELS.items() if key in ev.key), None)
        if name is not None:
            out[name] = out.get(name, 0.0) + ev.device_time_total / 1e3 / reps
    return {key: round(v, 4) for key, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="2,4")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--check-k", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("visibility_bench needs a CUDA device")
    import bench
    from pagnerf_b200 import build, ops
    from pagnerf_b200.mapping import extract_panoptic_map, instance_components, object_visibility, project_map, panoptic_map
    build.build()
    dev = torch.device("cuda:0")
    name, power = card()
    res = {"tool": "tools/visibility_bench.py", "gpu": name, "power_limit": power, "max_radius": MAX_RADIUS, "near": 0.01,
           "bitmap_cap_bytes": panoptic_map.VISIBILITY_BITMAP_BYTES, "results": []}
    V1, K1 = (torch.from_numpy(a).to(dev) for a in frame_camera())
    V42 = torch.from_numpy(bench.make_cameras()).to(dev)
    K42 = K1.expand(42, 4).contiguous()
    nef = bench.Workload(dev, n_rays=4096, seed=0, n_batches=1, config=2).nef
    level = int(nef.grid.blas_level)
    thr = float(torch.quantile(extract_panoptic_map(nef, 1, min_density=-1.0).density, 0.5))
    for k in [int(x) for x in args.ks.split(",")]:
        field = extract_panoptic_map(nef, k, min_density=thr)
        fruit, _ = fruit_map(field.xyz.shape[0], k, level)
        h = float(np.float32(1.0) / np.float32(k << level))
        for kind, pts, Ci, Cs in (("field", field, nef.num_instances, nef.num_classes), ("fruit", fruit, 200, 6)):
            comps = instance_components(pts, samples_per_axis=k, level=level, num_instances=Ci, num_classes=Cs)
            comp, K = comps.component, int(comps.count.numel())
            for B, V, Kc in ((1, V1, K1), (42, V42, K42)):
                vis_run = lambda: object_visibility(pts, samples_per_axis=k, level=level, view=V, intrinsics=Kc, height=1024, width=1024,
                                                    component=comp, num_objects=K, max_radius=MAX_RADIUS)
                proj_run = lambda: project_map(pts, samples_per_axis=k, level=level, view=V, intrinsics=Kc, height=1024, width=1024,
                                               max_radius=MAX_RADIUS, component=comp)
                ms, vis = timed(vis_run, args.reps)
                pms, _ = timed(proj_run, args.reps)
                ms2, _ = timed(vis_run, args.reps)                     # alternate: a second visibility pass after the projection
                mem, _ = peak_growth(vis_run)
                *_, total = ops.map_visibility(pts.xyz, V, Kc, 1024, 1024, h, float(np.float32(0.01)), MAX_RADIUS, comp, K,
                                               panoptic_map.VISIBILITY_BITMAP_BYTES)
                words, rounds = ops.silhouette_bitmap_words(total, 1024, 1024, panoptic_map.VISIBILITY_BITMAP_BYTES)
                seen = vis.visible > 0
                row = {"input": kind, "k": k, "points": int(pts.xyz.shape[0]), "objects": K, "views": B,
                       "ms": round(min(ms, ms2), 4), "ms_runs": [round(ms, 4), round(ms2, 4)], "project_map_ms": round(pms, 4),
                       "ratio_to_project_map": round(min(ms, ms2) / pms, 3), "ms_stages": stage_ms(vis_run, min(args.reps, 3)),
                       "rounds": rounds, "bitmap_words_total": int(total), "bitmap_bytes_allocated": 4 * int(words),
                       "peak_mem_growth_mb": round(mem / 2 ** 20, 2),
                       "object_views_seen": int(seen.sum()),
                       "mean_visible_over_silhouette": round(float((vis.visible[seen].double() / vis.silhouette[seen]).mean()), 5)
                       if bool(seen.any()) else None}
                res["results"].append(row)
                print(json.dumps(row), file=sys.stderr)
                del vis
            if kind == "field" and k == args.check_k:
                from oracle import visibility as ov
                Vs, Ks = V1.clone(), torch.tensor([[0.9 * 256, 0.9 * 256, 128.0, 128.0]], device=dev)
                vis = object_visibility(pts, samples_per_axis=k, level=level, view=Vs, intrinsics=Ks, height=256, width=256,
                                        component=comp, num_objects=K, max_radius=MAX_RADIUS)
                wv, ws, wb = ov.visibility(pts.xyz.cpu().numpy(), k, level, Vs.cpu().numpy(), Ks.cpu().numpy(), 256, 256,
                                           comp.cpu().numpy(), K, MAX_RADIUS, 0.01)
                res["oracle_check"] = {"k": k, "view": "256 x 256, config-5 camera", "points": int(pts.xyz.shape[0]), "objects": K,
                                       "equal": bool(np.array_equal(vis.visible.cpu().numpy(), wv)
                                                     and np.array_equal(vis.silhouette.cpu().numpy(), ws)
                                                     and np.array_equal(vis.bbox.cpu().numpy(), wb))}
                print(json.dumps(res["oracle_check"]), file=sys.stderr)
            del comps, comp
        del field, fruit
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
