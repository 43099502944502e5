"""Map-object benchmark: pagnerf_b200.mapping.instance_components on the maps tools/map_bench.py exports, and on planted-fruit maps
of the same sizes.

    python tools/components_bench.py [--ks 2,4] [--reps 5] [--check-k 2] [--out FILE]

Inputs per k (samples per cell axis):
  * field: the map of bench.py's BASELINE config-2 field (PanopticDeltaNeF, pruned level-7 synthetic scene) at k, half of the points
    kept (threshold = the median density of the k=1 map, as map_bench.py).  The random-init field gives every kept point the same
    instance label, so the map is one giant component: the worst case of the union step.
  * fruit: a map of the same size of separate lattice balls (radius 4, 257 points) with labels drawn from 200, thousands of
    objects, points in leaf-cell order like an exported map.
Prints one JSON line (and writes it to --out): points, objects, CUDA-event ms of the call (median of --reps warm runs), the stages
from a separate torch.profiler run (kernel time summed per stage: keys / insert, union, flatten / renumber, statistics), peak
memory growth against the documented bound, and at --check-k the comparison with the CPU oracle (oracle/components.py) with its CPU
time -- a CPU restatement, not a reference figure.  The card's name and power limit are read in the same process.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.map_bench import card, timed, peak_growth      # noqa: E402

STAGES = {"map_cc_keys_kernel": "keys_insert", "map_cc_union_kernel": "union", "map_cc_flatten_kernel": "flatten_renumber",
          "map_cc_flags_kernel": "flatten_renumber", "exclusive_scan_kernel": "flatten_renumber", "map_cc_rank_kernel": "flatten_renumber",
          "map_cc_label_kernel": "flatten_renumber", "map_instance_stats_kernel": "statistics",
          "map_instance_stats_global_kernel": "statistics"}


def fruit_map(n_points, k, level, seed=0):
    """Balls of radius 4 on a grid of spacing 12 (never adjacent), as many as make about n_points points -> PanopticPoints."""
    from pagnerf_b200.mapping import PanopticPoints
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(seed)
    D = k << level
    r = 4
    off = torch.stack(torch.meshgrid(*[torch.arange(-r, r + 1, device=dev)] * 3, indexing="ij"), -1).reshape(-1, 3)
    ball = off[(off ** 2).sum(1) <= r * r]
    slots = torch.arange(r, D - r, 12, device=dev)
    grid = torch.stack(torch.meshgrid(slots, slots, slots, indexing="ij"), -1).reshape(-1, 3)
    n_balls = min(grid.shape[0], max(1, n_points // ball.shape[0]))
    centres = grid[torch.randperm(grid.shape[0], generator=g, device=dev)[:n_balls]]
    j = (centres[:, None] + ball[None]).reshape(-1, 3)
    inst = torch.randint(0, 200, (n_balls,), generator=g, device=dev).repeat_interleave(ball.shape[0])
    cell, sub = j // k, j % k
    n = D // k
    order = torch.argsort(((cell[:, 0] * n + cell[:, 1]) * n + cell[:, 2]) * k ** 3 + (sub[:, 0] * k + sub[:, 1]) * k + sub[:, 2])
    j, inst = j[order], inst[order]
    P = j.shape[0]
    xyz = ((2 * j + 1).float() / float(D) - 1.0).contiguous()      # exact: integer numerator and power-of-two denominator
    rgb = torch.rand(P, 3, generator=g, device=dev)
    sem = torch.randint(0, 6, (P,), generator=g, device=dev)
    one = torch.ones(P, device=dev)
    return PanopticPoints(xyz, rgb, one, sem, one, inst, one), n_balls


def stage_ms(run, reps):
    """kernel time per stage (ms per call) from torch.profiler over `reps` calls"""
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            run()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        name = next((s for key, s in STAGES.items() if key in ev.key), None)
        if name is not None:
            out[name] = out.get(name, 0.0) + ev.device_time_total / 1e3 / reps
    return {key: round(v, 3) for key, v in out.items()}


def bound_bytes(P, K, Cs):
    C = 2
    while C < 2 * P:
        C *= 2
    return 12 * C + 24 * P + 12 * (P // 1024 + 1) + 8 + (160 + 8 * Cs) * K


def check(pts, got, k, level, Ci, Cs):
    from oracle import components as oc
    t0 = time.perf_counter()
    ref = oc.components(pts.xyz.cpu().numpy(), pts.semantic.cpu().numpy(), pts.instance.cpu().numpy(), k, level, None, 26, 1,
                        pts.rgb.cpu().numpy(), Ci, Cs)
    cpu_s = time.perf_counter() - t0
    exact = all(np.array_equal(getattr(got, key).cpu().numpy(), ref[key])
                for key in ("component", "count", "instance", "category", "votes", "bbox_min", "bbox_max"))
    close = all(np.allclose(getattr(got, key).cpu().numpy(), ref[key], rtol=1e-12, atol=1e-15) for key in ("centroid", "mean_rgb"))
    return {"oracle_equal": bool(exact and close), "oracle_cpu_s": round(cpu_s, 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="2,4")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--check-k", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("components_bench needs a CUDA device")
    import bench
    from pagnerf_b200 import build
    from pagnerf_b200.mapping import extract_panoptic_map, instance_components
    build.build()
    dev = torch.device("cuda:0")
    name, power = card()
    res = {"tool": "tools/components_bench.py", "gpu": name, "power_limit": power, "connectivity": 26, "min_points": 1, "results": []}
    nef = bench.Workload(dev, n_rays=4096, seed=0, n_batches=1, config=2).nef
    level = int(nef.grid.blas_level)
    Ci, Cs = int(nef.num_instances), int(nef.num_classes)
    thr = float(torch.quantile(extract_panoptic_map(nef, 1, min_density=-1.0).density, 0.5))
    for k in [int(x) for x in args.ks.split(",")]:
        field = extract_panoptic_map(nef, k, min_density=thr)
        fruit, n_balls = fruit_map(field.xyz.shape[0], k, level)
        for kind, pts in (("field", field), ("fruit", fruit)):
            run = lambda: instance_components(pts, samples_per_axis=k, level=level, num_instances=Ci, num_classes=Cs)
            ms, got = timed(run, args.reps)
            mem, _ = peak_growth(run)
            P, K = int(pts.xyz.shape[0]), int(got.count.numel())
            row = {"input": kind, "k": k, "points": P, "objects": K, "largest_object": int(got.count.max()) if K else 0,
                   "ms": round(ms, 3), "ms_stages": stage_ms(run, args.reps), "points_per_s": round(P / (ms * 1e-3), 1),
                   "peak_mem_growth_mb": round(mem / 2 ** 20, 1), "documented_bound_mb": round(bound_bytes(P, K, Cs) / 2 ** 20, 1)}
            if kind == "fruit":
                row["planted_balls"] = n_balls
            if k == args.check_k:
                row.update(check(pts, got, k, level, Ci, Cs))
            res["results"].append(row)
            print(json.dumps(row), file=sys.stderr)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
