"""Point-map export benchmark: pagnerf_b200.mapping.extract_panoptic_map + instance_summary against the existing route (nef forward
with every channel + torch.argmax + threshold, what utils/render_map.py does through this package) on the fields of bench.py's
BASELINE configs 2 and 5 (PanopticDeltaNeF, permutohedral grids L=24 T=2^18, pruned level-7 synthetic scene).

    python tools/map_bench.py [--configs 2,5] [--ks 1,2,4] [--chunk 2097152] [--reps 3] [--out FILE]

Prints one JSON line (and writes it to --out): occupied cells, points and kept points per k, CUDA-event ms per stage (points, encode,
density + colour, compaction + delta encode, labels, summary) of a staged run -- plus, on the same rows, the existing route's heads
(per-thread decoder.cu [K, C] channels + torch.argmax) --, the end-to-end ms of the public call, points per
second, peak memory growth, the existing route's ms / peak memory on the same points and chunking, the label agreement of the two
routes, and the card's name and power limit read in the same process.  Every shape is run once before it is timed; the chunks'
working sets (2^21 x 48 fp32 features = 400 MB) are larger than the 126 MB L2.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [s.strip() for s in q.strip().splitlines()[torch.cuda.current_device()].split(",")]
    except (OSError, subprocess.CalledProcessError, ValueError, IndexError):
        name, power = torch.cuda.get_device_name(), "unknown"
    return name, power


class Stages:
    """CUDA-event timer of named stages (summed over chunks)."""

    def __init__(self):
        self.ev = []

    def mark(self, name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.ev.append((name, e))

    def report(self):
        torch.cuda.synchronize()
        out = {}
        for (name, e0), (_, e1) in zip(self.ev, self.ev[1:]):
            if name is not None:
                out[name] = out.get(name, 0.0) + e0.elapsed_time(e1)
        return out


def staged_extract(nef, k, chunk, thr, vd, t):
    """extract_panoptic_map's steps with a stage mark between them (same calls, same order) -> (kept count, instance labels)."""
    from pagnerf_b200 import ops, spc
    from pagnerf_b200.pc_nerf.panoptic_nef import _decoder_tensors
    grid = nef.grid
    level = grid.blas_level
    cells = spc.unbatched_get_level_points(grid.blas.points, grid.blas.pyramid, level)
    per = max(1, chunk // k ** 3)
    lod_idx = nef.num_lods - 1
    w_dc = _decoder_tensors(nef.decoder_density, 1) + _decoder_tensors(nef.decoder_color, 2)
    w_pan = _decoder_tensors(nef.decoder_semantics, 1) + _decoder_tensors(nef.decoder_inst, 2)
    lodw = nef._lodw(vd.device)
    kept, labels = 0, []
    with torch.no_grad():
        for c0 in range(0, cells.shape[0], per):
            t.mark("points")
            xyz = ops.map_cell_points(cells[c0:c0 + per], level, k)
            t.mark("encode")
            coords = xyz[:, None]
            feats = nef._encode(grid, coords, lod_idx)
            t.mark("density_colour")
            sigma, rgb = ops.DecodeDCFn.apply(feats, lodw, vd, xyz.shape[0], True, 'tiled', *w_dc)
            t.mark("compaction_delta_encode")
            rows = torch.nonzero(sigma > thr).reshape(-1)
            a, b = nef._panoptic_inputs(feats, coords, lod_idx, rows)
            parts = (xyz.index_select(0, rows), rgb.index_select(0, rows), sigma.index_select(0, rows))
            del feats
            t.mark("labels")
            out = ops.pan_labels_f32(a, b, lodw, nef.num_classes, nef.num_instances, bool(nef.sem_softmax), bool(nef.inst_softmax),
                                     float(getattr(nef, 'inst_soft_temperature', 0.0)), *w_pan)
            t.mark("existing_heads")
            # the existing route's heads on the same rows: per-sample [K, C] channels (csrc/decoder.cu) + torch.argmax
            ps, pi = ops.DecodePanFn.apply(a, b, lodw, nef.num_classes, nef.num_instances, bool(nef.sem_softmax),
                                           bool(nef.inst_softmax), float(getattr(nef, 'inst_soft_temperature', 0.0)), False, *w_pan)
            ps.argmax(1), pi.argmax(1)
            t.mark(None)
            del ps, pi
            kept += rows.numel()
            labels.append(out[2])
            del a, b, parts
    return kept, torch.cat(labels)


def existing_route(nef, k, chunk, thr, vd):
    """nef(coords, ray_d, channels={'density','rgb','semantics','inst_embedding'}) per chunk, then threshold + torch.argmax."""
    from pagnerf_b200 import ops, spc
    grid = nef.grid
    cells = spc.unbatched_get_level_points(grid.blas.points, grid.blas.pyramid, grid.blas_level)
    per = max(1, chunk // k ** 3)
    labels = []
    with torch.no_grad():
        for c0 in range(0, cells.shape[0], per):
            xyz = ops.map_cell_points(cells[c0:c0 + per], grid.blas_level, k)
            n = xyz.shape[0]
            out = nef(coords=xyz[:, None], ray_d=vd.expand(n, 3).contiguous(), channels={'density', 'rgb', 'semantics', 'inst_embedding'})
            keep = out['density'].reshape(-1) > thr
            out['semantics'][keep].argmax(1)
            labels.append(out['inst_embedding'][keep].argmax(1))
    return torch.cat(labels)


def timed(fn, reps):
    fn()                                  # warm this shape
    ms = []
    for _ in range(reps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return sorted(ms)[len(ms) // 2], r


def peak_growth(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    r = fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="2,5")
    ap.add_argument("--ks", default="1,2,4")
    ap.add_argument("--chunk", type=int, default=1 << 21)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--keep", type=float, default=0.5,
                    help="threshold = this quantile of the density of the field's k=1 map (a random-init field is below prune()'s "
                         "threshold everywhere, so the default threshold would keep nothing); <= 0: prune()'s threshold")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("map_bench needs a CUDA device")
    import bench
    from pagnerf_b200 import build
    from pagnerf_b200.mapping import extract_panoptic_map, instance_summary
    from pagnerf_b200.mapping.panoptic_map import PRUNE_MIN_DENSITY
    build.build()
    dev = torch.device("cuda:0")
    name, power = card()
    res = {"tool": "tools/map_bench.py", "gpu": name, "power_limit": power, "chunk_points": args.chunk, "view_dir": [0.0, 0.0, -1.0],
           "threshold_rule": (f"{1 - args.keep:g} quantile of the k=1 map's density" if args.keep > 0 else "prune() threshold"),
           "results": []}
    vd = torch.tensor([[0.0, 0.0, -1.0]], device=dev)
    for cfg in [int(c) for c in args.configs.split(",")]:
        wl = bench.Workload(dev, n_rays=4096, seed=0, n_batches=1, config=cfg)
        nef = wl.nef
        from pagnerf_b200 import spc
        cells = spc.unbatched_get_level_points(nef.grid.blas.points, nef.grid.blas.pyramid, nef.grid.blas_level).shape[0]
        kept_at_prune_threshold = int(extract_panoptic_map(nef, 1).xyz.shape[0])
        thr = PRUNE_MIN_DENSITY
        if args.keep > 0:
            thr = float(torch.quantile(extract_panoptic_map(nef, 1, min_density=-1.0).density, 1.0 - args.keep))
        for k in [int(x) for x in args.ks.split(",")]:
            P = cells * k ** 3
            run = lambda: extract_panoptic_map(nef, k, min_density=thr, chunk_points=args.chunk)
            ms_e2e, pts = timed(run, args.reps)
            mem_ours, _ = peak_growth(run)
            ms_sum, summ = timed(lambda: instance_summary(pts, nef.num_instances, nef.num_classes), args.reps)
            staged_extract(nef, k, args.chunk, thr, vd, Stages())          # warm
            st = []
            for _ in range(args.reps):
                t = Stages()
                kept_s, lab_s = staged_extract(nef, k, args.chunk, thr, vd, t)
                st.append(t.report())
            stages = {key: sorted(s[key] for s in st)[len(st) // 2] for key in st[0]}
            stages["summary"] = ms_sum
            ms_old, lab_old = timed(lambda: existing_route(nef, k, args.chunk, thr, vd), args.reps)
            mem_old, _ = peak_growth(lambda: existing_route(nef, k, args.chunk, thr, vd))
            same = lab_old.shape == pts.instance.shape
            agree = float((lab_old == pts.instance).double().mean()) if same and pts.instance.numel() else None
            res["results"].append({
                "config": cfg, "k": k, "threshold": thr, "kept_points_k1_at_prune_threshold": kept_at_prune_threshold,
                "occupied_cells": cells, "level_cells": 8 ** nef.grid.blas_level, "points": P,
                "kept_points": int(pts.xyz.shape[0]), "staged_kept_equal": kept_s == int(pts.xyz.shape[0]) and torch.equal(lab_s, pts.instance),
                "ms_end_to_end": round(ms_e2e, 3), "ms_stages": {key: round(v, 3) for key, v in stages.items()},
                "points_per_s": round(P / (ms_e2e * 1e-3), 1), "peak_mem_growth_mb": round(mem_ours / 2 ** 20, 1),
                "existing_route": {"ms": round(ms_old, 3), "peak_mem_growth_mb": round(mem_old / 2 ** 20, 1),
                                   "kept_points": int(lab_old.shape[0]), "instance_label_agreement": agree},
                "labels_vs_existing_heads_speedup": round(stages["existing_heads"] / stages["labels"], 2),
                "instances_with_points": int((summ.count > 0).sum()),
            })
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
