"""Scene-level panoptic quality on the device: update ms per frame, compute() and sync-merge ms, table bytes and keys used, the CPU
oracle's seconds, and the device result against the oracle.

    python tools/scene_pq_bench.py [--updates 300] [--out profiles/scene_pq_bench.json]

Prints one JSON line (and writes it to --out):
  update       ScenePanopticQuality.update of one frame of a 100-frame oracle.scene_metrics.synthetic_sequence (~150 fruit that keep
               their ids, consistent prediction ids) at 1024x1024 and 1280x720: CUDA events around --updates warm updates, the
               frames cycled, after 200 warm-up updates; the tables' keys used after all of them
  compute      compute() at the default capacity (2^18) on those tables: host clock around the call, which ends in its one
               device-to-host read; stats() alone (its two kernels) with CUDA events
  sync_merge   pag_scene_pq_merge of one such table into another on the same device (what sync() runs per other rank), CUDA events
  oracle       the first 20 frames at 1024x1024, consistent and permuted ids: the CPU oracle's seconds (kind "port": a
               restatement, not Panoptic Lifting's code) and whether the device result equals it (counts exact, iou_sum to 1e-12)"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import metrics as om                               # noqa: E402
from oracle import scene_metrics as osm                        # noqa: E402
from pagnerf_b200._lib import call, ptr                        # noqa: E402
from pagnerf_b200.metrics import ScenePanopticQuality          # noqa: E402

ARGS = (om.SYN_THINGS, om.SYN_STUFFS)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], text=True, timeout=30)
        power = out.strip().splitlines()[0]
    except Exception as e:      # noqa: BLE001
        power = f"unknown ({type(e).__name__})"
    return name, power


def events(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(reps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def time_updates(H, W, updates, dev, n_frames=100):
    p, t = osm.synthetic_sequence(n_frames, H, W, seed=H + W, n_inst=150)
    pd, td = p.to(dev), t.to(dev)
    del p, t
    m = ScenePanopticQuality(*ARGS).to(dev)
    for i in range(200):
        m.update(pd[i % n_frames:i % n_frames + 1], td[i % n_frames:i % n_frames + 1])
    ms = events(lambda i: m.update(pd[i % n_frames:i % n_frames + 1], td[i % n_frames:i % n_frames + 1]), updates)
    res = {"H": H, "W": W, "ms_per_frame": round(ms, 4), "updates_timed": updates, "frames_in_sequence": n_frames,
           "keys_used": m.keys_used().cpu().tolist(), "pq": float(m.compute())}
    return res, m


def time_compute(m, reps=50):
    m.compute()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        m.compute()
    host_ms = (time.perf_counter() - t0) / reps * 1e3
    stats_ms = events(lambda i: m.stats(), reps)
    return {"capacity": m.capacity, "compute_ms": round(host_ms, 4), "stats_kernels_ms": round(stats_ms, 4), "reps": reps,
            "table_bytes": m._workspace.numel()}


def time_merge(a, b, reps=50):
    wa, wb = a._workspace.clone(), b._workspace
    ms = events(lambda i: call("pag_scene_pq_merge", ptr(wa), ptr(wb), a.capacity, wa.numel()), reps)
    return {"merge_ms": round(ms, 4), "reps": reps, "what": "one 1024x1024-sequence table into a 1280x720-sequence table, same device"}


def check_oracle(dev, n=20):
    out = []
    for consistent in (True, False):
        p, t = osm.synthetic_sequence(n, 1024, 1024, seed=7, n_inst=150, consistent=consistent)
        torch.set_num_threads(os.cpu_count())
        t0 = time.perf_counter()
        ref = osm.scene_panoptic_quality_stats(p, t, *ARGS)
        cpu_s = time.perf_counter() - t0
        m = ScenePanopticQuality(*ARGS).to(dev)
        for f in range(n):
            m.update(p[f:f + 1].to(dev), t[f:f + 1].to(dev))
        iou, tp, fp, fn = (x.cpu() for x in m.stats())
        exact = torch.equal(tp, ref[1]) and torch.equal(fp, ref[2]) and torch.equal(fn, ref[3])
        rel = float(((iou - ref[0]).abs() / ref[0].abs().clamp_min(1e-300)).max())
        out.append({"consistent_ids": consistent, "frames": n, "H": 1024, "W": 1024, "kind": "port", "threads": torch.get_num_threads(),
                    "cpu_oracle_s": round(cpu_s, 3), "counts_exact_vs_oracle": exact, "iou_sum_max_rel_diff_vs_oracle": rel,
                    "equal": exact and rel <= 1e-12, "scene_pq": float(m.compute()),
                    "per_image_pq": float(om.panoptic_quality(p, t, *ARGS))})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--updates", type=int, default=300)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("scene_pq_bench needs a CUDA device (no CPU fallback)")
    dev = torch.device("cuda:0")
    name, power = card()
    u1, m1 = time_updates(1024, 1024, args.updates, dev)
    u2, m2 = time_updates(720, 1280, args.updates, dev)
    res = {"tool": "scene_pq_bench", "gpu": name, "power_limit": power, "update": [u1, u2], "compute": time_compute(m1),
           "sync_merge": time_merge(m2, m1), "oracle": check_oracle(dev),
           "targets_not_measured": {"update_ms_per_1mp_frame": 0.05, "compute_ms_at_capacity_2p18": 0.2}}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
