"""Map-projection benchmark: pagnerf_b200.mapping.project_map on the maps tools/components_bench.py builds, into bench.py's config-5
camera and into the whole synthetic pass.

    python tools/project_bench.py [--ks 2,4] [--reps 20] [--check-k 2] [--out FILE]

Inputs:
  * maps: the map of bench.py's BASELINE config-2 field at each k (half of the points kept, as components_bench.py) and a
    planted-fruit map of the same size (components_bench.fruit_map).
  * views: config 5's 1024 x 1024 camera (the view and intrinsics that reproduce bench.make_frame_rays: identity rotation,
    f = 0.9 res, c = res / 2), B = 1, and the 42 cameras of bench.make_cameras with the same intrinsics, B = 42.
Prints one JSON line (and writes it to --out): CUDA-event ms (median of --reps warm runs; the depth buffer of one view is 8 MB and
stays in the 126 MB L2, the maps' 17 / 134 MB of coordinates are streamed), pixel tests per view (computed on the device from the
footprints by this script), the covered-pixel fraction, peak memory growth, the kernels' time from a separate torch.profiler run,
the config-5 fp32 render plus lookup_rays of the same frame with the fraction of pixels where the two routes give the same object,
and at --check-k the equality with the CPU oracle (oracle/projection.py) on a 256 x 256 view.  The card's name and power limit are
read in the same process.
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
from tools.lookup_bench import render_frame               # noqa: E402

MAX_RADIUS = 8
MIN_ALPHA = 1e-6          # the random-init config-5 field has alpha < 0.5 on almost every ray (lookup_bench.py): look up every ray it touches
KERNELS = {"map_project_splat_kernel": "splat", "map_project_resolve_kernel": "resolve", "Memset": "fill"}


def frame_camera(res=1024, seed=0):
    """view [1, 4, 4] and intrinsics [1, 4] of bench.make_frame_rays' camera"""
    rng = np.random.default_rng(seed * 100003 + 77)            # make_frame_rays' draw of the camera position
    cam = np.array([rng.uniform(-0.8, 0.8), rng.uniform(-0.05, 0.05), 0.9])
    V = np.eye(4, dtype=np.float32)[None].copy()
    V[0, :3, 3] = -cam
    return V, np.array([[0.9 * res, 0.9 * res, res / 2, res / 2]], np.float32)


def pixel_tests(xyz, V, K, H, W, h, near=0.01):
    """Pixels tested per view: the clamped footprint areas of the projected points (torch on the device, not bit-exact)"""
    tot = torch.zeros((), dtype=torch.float64, device=xyz.device)
    for b in range(V.shape[0]):
        p = xyz @ V[b, :3, :3].T + V[b, :3, 3]
        z = -p[:, 2]
        fx, fy, cx, cy = K[b]
        u, v = fx * (p[:, 0] / z) + cx, fy * (p[:, 1] / z) + cy
        su, sv = (fx * h / z).clamp(max=MAX_RADIUS), (fy * h / z).clamp(max=MAX_RADIUS)
        ok = (z > near) & torch.isfinite(u) & torch.isfinite(v)
        nc = (torch.floor(u + su).clamp(max=W - 1) - torch.floor(u - su).clamp(min=0) + 1).clamp(min=0)
        nr = (torch.floor(v + sv).clamp(max=H - 1) - torch.floor(v - sv).clamp(min=0) + 1).clamp(min=0)
        tot += torch.where(ok, nc * nr, torch.zeros_like(nc)).double().sum()
    return float(tot) / V.shape[0]


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
        raise SystemExit("project_bench needs a CUDA device")
    import bench
    from pagnerf_b200 import build
    from pagnerf_b200.mapping import extract_panoptic_map, instance_components, map_index, lookup_rays, project_map
    build.build()
    dev = torch.device("cuda:0")
    name, power = card()
    res = {"tool": "tools/project_bench.py", "gpu": name, "power_limit": power, "max_radius": MAX_RADIUS, "near": 0.01, "results": []}
    ks = [int(x) for x in args.ks.split(",")]
    V1, K1 = (torch.from_numpy(a).to(dev) for a in frame_camera())
    V42 = torch.from_numpy(bench.make_cameras()).to(dev)
    K42 = K1.expand(42, 4).contiguous()
    nef = bench.Workload(dev, n_rays=4096, seed=0, n_batches=1, config=2).nef
    level = int(nef.grid.blas_level)
    thr = float(torch.quantile(extract_panoptic_map(nef, 1, min_density=-1.0).density, 0.5))
    for k in ks:
        field = extract_panoptic_map(nef, k, min_density=thr)
        fruit, _ = fruit_map(field.xyz.shape[0], k, level)
        h = 1.0 / (k << level)
        for kind, pts in (("field", field), ("fruit", fruit)):
            for B, V, K in ((1, V1, K1), (42, V42, K42)):
                run = lambda: project_map(pts, samples_per_axis=k, level=level, view=V, intrinsics=K, height=1024, width=1024,
                                          max_radius=MAX_RADIUS)
                ms, mv = timed(run, args.reps)
                mem, _ = peak_growth(run)
                row = {"input": kind, "k": k, "points": int(pts.xyz.shape[0]), "views": B, "ms": round(ms, 4),
                       "ms_per_view": round(ms / B, 4), "ms_stages": stage_ms(run, min(args.reps, 5)),
                       "pixel_tests_per_view": round(pixel_tests(pts.xyz, V, K, 1024, 1024, h), 1),
                       "covered_pixel_fraction": round(float((mv.point >= 0).float().mean()), 5),
                       "peak_mem_growth_mb": round(mem / 2 ** 20, 2)}
                res["results"].append(row)
                print(json.dumps(row), file=sys.stderr)
                del mv
        if k == args.check_k:
            from oracle import projection as op
            Vs, Ks = V1.clone(), torch.tensor([[0.9 * 256, 0.9 * 256, 128.0, 128.0]], device=dev)
            comps = instance_components(field, samples_per_axis=k, level=level, num_instances=nef.num_instances,
                                        num_classes=nef.num_classes)
            mv = project_map(field, samples_per_axis=k, level=level, view=Vs, intrinsics=Ks, height=256, width=256,
                             max_radius=MAX_RADIUS, component=comps.component)
            wp, wd, wo = op.project(field.xyz.cpu().numpy(), k, level, Vs.cpu().numpy(), Ks.cpu().numpy(), 256, 256, MAX_RADIUS, 0.01,
                                    comps.component.cpu().numpy())
            res["oracle_check"] = {"k": k, "view": "256 x 256, config-5 camera", "points": int(field.xyz.shape[0]),
                                   "equal": bool(np.array_equal(mv.point.cpu().numpy(), wp) and np.array_equal(mv.depth.cpu().numpy(), wd)
                                                 and np.array_equal(mv.object.cpu().numpy(), wo))}
            print(json.dumps(res["oracle_check"]), file=sys.stderr)
        del field, fruit
    del nef
    # the config-5 route: fp32 render of the frame + lookup_rays, against the projection of the config-5 field's map
    wl = bench.Workload(dev, n_rays=4096, seed=0, n_batches=1, config=5)
    o, d, depth, alpha, render_ms = render_frame(wl)
    level = int(wl.nef.grid.blas_level)
    thr5 = float(torch.quantile(extract_panoptic_map(wl.nef, 1, min_density=-1.0).density, 0.5))
    res["render_vs_projection"] = []
    for k in ks:
        pts = extract_panoptic_map(wl.nef, k, min_density=thr5)
        comps = instance_components(pts, samples_per_axis=k, level=level, num_instances=wl.nef.num_instances,
                                    num_classes=wl.nef.num_classes)
        index = map_index(pts, samples_per_axis=k, level=level)
        lms, hit = timed(lambda: lookup_rays(index, o, d, depth, alpha, radius=1, min_alpha=MIN_ALPHA, component=comps.component), args.reps)
        pms, mv = timed(lambda: project_map(pts, samples_per_axis=k, level=level, view=V1, intrinsics=K1, height=1024, width=1024,
                                            max_radius=MAX_RADIUS, component=comps.component), args.reps)
        lo, po = hit.object, mv.object.reshape(-1)
        both = (lo >= 0) & (po >= 0)
        row = {"k": k, "min_alpha": MIN_ALPHA, "lookup_radius": 1, "map_points": int(pts.xyz.shape[0]), "objects": int(comps.count.numel()), "render_fp32_ms": round(render_ms, 3),
               "lookup_rays_ms": round(lms, 4), "project_ms": round(pms, 4), "project_share_of_render": round(pms / render_ms, 5),
               "same_object_fraction": round(float((lo == po).float().mean()), 5),
               "same_object_fraction_where_both_see_one": round(float((lo[both] == po[both]).float().mean()), 5) if bool(both.any()) else None,
               "lookup_object_fraction": round(float((lo >= 0).float().mean()), 5),
               "project_object_fraction": round(float((po >= 0).float().mean()), 5)}
        res["render_vs_projection"].append(row)
        print(json.dumps(row), file=sys.stderr)
        del pts, comps, index, mv, hit
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
