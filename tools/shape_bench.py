"""Object-shape benchmark: pagnerf_b200.mapping.object_shape against the torch route (index_add_ of per-point outer products,
torch.linalg.eigh, scatter_reduce for the extents) in the same process, on the maps of tools/components_bench.py.

    python tools/shape_bench.py [--ks 2,4] [--reps 20] [--check-k 2] [--out FILE]

Inputs per k (samples per cell axis): the map of bench.py's BASELINE config-2 field at k (half of the points kept) split into
objects by instance_components, and the planted-fruit map of the same size (components_bench.fruit_map, one object per ball).  The
random-init field's map is one giant component: every point of it lands on the same object's accumulators, the worst case of the
moments and extents passes.
Prints one JSON line (and writes it to --out): per input the points, objects and largest object, the median CUDA-event ms of
object_shape and of the torch route over --reps warm runs (alternated: object_shape, torch, object_shape), the kernels' time from a
separate torch.profiler run, the peak memory growth of each route, the documented bound of object_shape's, and at --check-k the
bit-for-bit covariance comparison with the CPU oracle (oracle/shape.py).  The card's name and power limit are read in the same
process.  The torch route's f64 sums are not exact (S_ab reaches 2^66), so it is a timing and memory comparison, not a reference.
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

KERNELS = {"map_shape_moments_kernel": "moments", "map_shape_axes_kernel": "axes", "map_shape_extent_kernel": "extents",
           "map_shape_box_kernel": "box", "Memset": "fills"}
PAIRS = [0, 1, 2, 4, 5, 8]       # xx, xy, xz, yy, yz, zz of a row-major 3x3
EIGH_BACKEND = {"name": "default"}


def torch_route(xyz, component, K, D):
    """The same quantities with stock torch ops: f64 lattice indices, index_add_ of counts, sums and per-point outer products (a
    [P, 6] f64 temporary), covariance, torch.linalg.eigh (descending, no sign rule), projections and scatter_reduce amin / amax."""
    sel = component >= 0
    j = torch.round(((xyz[sel].double() + 1.0) * D) * 0.5 - 0.5)
    c = component[sel]
    n = torch.zeros(K, dtype=torch.float64, device=xyz.device).index_add_(0, c, torch.ones_like(j[:, 0]))
    s1 = torch.zeros(K, 3, dtype=torch.float64, device=xyz.device).index_add_(0, c, j)
    s2 = torch.zeros(K, 6, dtype=torch.float64, device=xyz.device).index_add_(0, c, (j[:, :, None] * j[:, None, :]).reshape(-1, 9)[:, PAIRS])
    mean = s1 / n[:, None]
    full = s2[:, [0, 1, 2, 1, 3, 4, 2, 4, 5]].reshape(K, 3, 3)
    cov = (full / n[:, None, None] - mean[:, :, None] * mean[:, None, :]) * (4.0 / D / D)
    try:
        var, vec = torch.linalg.eigh(cov)
    except torch.linalg.LinAlgError:      # cuSOLVER's batched solver refuses some batches (CUSOLVER_STATUS_INVALID_VALUE)
        EIGH_BACKEND["name"] = "magma"
        torch.backends.cuda.preferred_linalg_library("magma")
        var, vec = torch.linalg.eigh(cov)
    axes = vec.flip(-1).transpose(-1, -2)
    p = torch.einsum("pc,pac->pa", j, axes[c])
    idx = c[:, None].expand(-1, 3)
    lo = torch.full((K, 3), float("inf"), dtype=torch.float64, device=xyz.device).scatter_reduce_(0, idx, p, "amin")
    hi = torch.full((K, 3), float("-inf"), dtype=torch.float64, device=xyz.device).scatter_reduce_(0, idx, p, "amax")
    extent = ((hi - lo) + 1.0) * 2.0 / D
    centre = (2.0 * torch.einsum("ka,kac->kc", (lo + hi) / 2.0, axes) + 1.0) / D - 1.0
    return cov, var.flip(-1), axes, centre, extent


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
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--check-k", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("shape_bench needs a CUDA device")
    import bench
    from pagnerf_b200 import build
    from pagnerf_b200.mapping import extract_panoptic_map, instance_components, object_shape, panoptic_map
    build.build()
    dev = torch.device("cuda:0")
    name, power = card()
    res = {"tool": "tools/shape_bench.py", "gpu": name, "power_limit": power, "results": []}
    nef = bench.Workload(dev, n_rays=4096, seed=0, n_batches=1, config=2).nef
    level = int(nef.grid.blas_level)
    thr = float(torch.quantile(extract_panoptic_map(nef, 1, min_density=-1.0).density, 0.5))
    for k in [int(x) for x in args.ks.split(",")]:
        D = k << level
        field = extract_panoptic_map(nef, k, min_density=thr)
        fruit, _ = fruit_map(field.xyz.shape[0], k, level)
        for kind, pts, Ci, Cs in (("field", field, nef.num_instances, nef.num_classes), ("fruit", fruit, 200, 6)):
            comps = instance_components(pts, samples_per_axis=k, level=level, num_instances=Ci, num_classes=Cs)
            comp, K = comps.component, int(comps.count.numel())
            run = lambda: object_shape(pts, samples_per_axis=k, level=level, component=comp, num_objects=K)
            ref = lambda: torch_route(pts.xyz, comp, K, D)
            ms, got = timed(run, args.reps)
            tms, tr = timed(ref, args.reps)
            ms2, _ = timed(run, args.reps)
            mem, _ = peak_growth(run)
            tmem, _ = peak_growth(ref)
            P = int(pts.xyz.shape[0])
            row = {"input": kind, "k": k, "points": P, "objects": K, "largest_object": int(comps.count.max()) if K else 0,
                   "ms": round(min(ms, ms2), 4), "ms_runs": [round(ms, 4), round(ms2, 4)], "ms_stages": stage_ms(run, 5),
                   "torch_route_ms": round(tms, 4), "torch_route_eigh_backend": EIGH_BACKEND["name"], "speedup_over_torch_route": round(tms / min(ms, ms2), 2),
                   "peak_mem_growth_mb": round(mem / 2 ** 20, 3),
                   "documented_bound_mb": round(((216 + panoptic_map.SHAPE_WORKSPACE_BYTES) * K + 16) / 2 ** 20, 3),
                   "torch_route_peak_mem_growth_mb": round(tmem / 2 ** 20, 1),
                   "torch_route_max_abs_extent_diff": float((tr[4] - got.extent).abs().max()),
                   "median_extent_world": [round(float(x), 5) for x in got.extent.median(0).values]}
            if k == args.check_k:
                from oracle import shape as osh
                from oracle.components import lattice_index
                j, on = lattice_index(pts.xyz.cpu().numpy(), k, level)
                n, S, SS = osh.moments(j, comp.cpu().numpy(), K)
                want = osh.covariance(n, S, SS, D)
                row["oracle_covariance_bit_equal"] = bool(on.all() and np.array_equal(got.covariance.cpu().numpy().view(np.uint64),
                                                                                       want.view(np.uint64)))
            res["results"].append(row)
            print(json.dumps(row), file=sys.stderr)
            del comps, comp, got, tr
        del field, fruit
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
