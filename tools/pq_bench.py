"""Panoptic-quality update on the device: ms per frame, the CPU oracle's s per frame, and PQ's share of a validation frame.

    python tools/pq_bench.py [--frames 200] [--out profiles/pq_bench.json]

Prints one JSON line (and writes it to --out):
  update           device PanopticQuality.update of one synthetic frame (oracle.metrics.synthetic_frames: ~150 target and
                   ~150 prediction instances, 2 % void) at 1024x1024 and 1280x720: CUDA events around --frames warm updates, four
                   distinct frames cycled; the statistics of one update are checked against the CPU oracle in the same run
  cpu_oracle       oracle.metrics on all host threads, s per 1 MP frame (kind "port": a restatement, not the reference's code)
  validation_frame bench config 5's render (fp32 decoders, bench.Workload / make_frame_rays), the argmax label maps as
                   evaluate_metrics forms them, [1, H, W, 2] int64 maps and one update; ms of each and PQ's share
The byte count is a lower bound from the shapes (the int64 maps are read once), not a measurement."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import metrics as om                          # noqa: E402
from pagnerf_b200.metrics import PanopticQuality          # noqa: E402

HBM_DATASHEET_GBS = 7700.0


def card():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], text=True, timeout=30)
        power = out.strip().splitlines()[0]
    except Exception as e:      # noqa: BLE001
        power = f"unknown ({type(e).__name__})"
    return name, power


def time_updates(H, W, frames, dev):
    p, t = om.synthetic_frames(4, H, W, seed=H * W)
    m = PanopticQuality(om.SYN_THINGS, om.SYN_STUFFS).to(dev)
    pd, td = p.to(dev), t.to(dev)
    m.update(pd[:1], td[:1])
    ref = om.panoptic_quality_stats(p[:1], t[:1], om.SYN_THINGS, om.SYN_STUFFS)
    iou, tp, fp, fn = (x.cpu() for x in m.stats())
    exact = torch.equal(tp, ref[1]) and torch.equal(fp, ref[2]) and torch.equal(fn, ref[3])
    iou_rel = float(((iou - ref[0]).abs() / ref[0].abs().clamp_min(1e-300)).max())
    for i in range(20):
        m.update(pd[i % 4:i % 4 + 1], td[i % 4:i % 4 + 1])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(frames):
        m.update(pd[i % 4:i % 4 + 1], td[i % 4:i % 4 + 1])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / frames
    nbytes = 2 * H * W * 2 * 8
    return {"H": H, "W": W, "ms_per_frame": round(ms, 4), "frames_timed": frames, "counts_exact_vs_oracle": exact,
            "iou_sum_max_rel_diff_vs_oracle": iou_rel, "target_instances": len(t[0, ..., 1].unique()) - 1,
            "pred_instances": len(p[0, ..., 1].unique()) - 1, "map_bytes": nbytes,
            "map_bytes_at_datasheet_hbm_us": round(nbytes / HBM_DATASHEET_GBS / 1e3, 2)}


def time_oracle(n=3):
    torch.set_num_threads(os.cpu_count())
    p, t = om.synthetic_frames(n, 1024, 1024, seed=1)
    t0 = time.perf_counter()
    for b in range(n):
        om.panoptic_quality_stats(p[b:b + 1], t[b:b + 1], om.SYN_THINGS, om.SYN_STUFFS)
    return {"kind": "port", "what": "oracle.metrics (torch CPU) per 1024x1024 frame", "threads": torch.get_num_threads(),
            "s_per_frame": round((time.perf_counter() - t0) / n, 4)}


def time_validation_frame(dev, reps=5):
    from bench import Workload, make_frame_rays, NEAR, FAR
    from pagnerf_b200.wisp_compat import Rays
    res = 1024
    wl = Workload(dev, n_rays=4096, seed=0, n_batches=1, config=5)
    wl.nef.decoder_precision = 'fp32'
    o_np, d_np = make_frame_rays(res)
    o, d = torch.from_numpy(o_np).to(dev), torch.from_numpy(d_np).to(dev)
    chans = ['rgb', 'depth', 'semantics', 'inst_embedding']
    chunk = 131072
    # stuffs {0}, things {1..5} of the 6 semantic classes (an assumption of this tool: the split only moves the segment count)
    m = PanopticQuality(things=set(range(1, 6)), stuffs={0}).to(dev)

    def render():
        sem, inst = [], []
        with torch.no_grad():
            for c0 in range(0, res * res, chunk):
                rb = wl.tracer(wl.nef, channels=chans, rays=Rays(origins=o[c0:c0 + chunk], dirs=d[c0:c0 + chunk], dist_min=NEAR, dist_max=FAR),
                               lod_idx=None, stage='val')
                sem.append(rb.semantics)
                inst.append(rb.inst_embedding)
        return torch.cat(sem), torch.cat(inst)

    def label_maps(sem, inst):
        return torch.stack([sem.argmax(-1), inst.argmax(-1)], -1).reshape(1, res, res, 2)

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    tot = [0.0, 0.0, 0.0]
    target = None
    for r in range(reps + 2):
        ev[0].record()
        sem, inst = render()
        ev[1].record()
        maps = label_maps(sem, inst)
        ev[2].record()
        m.update(maps, maps if target is None else target)      # scored against the previous frame's maps
        ev[3].record()
        torch.cuda.synchronize()
        target = maps
        if r >= 2:
            for i in range(3):
                tot[i] += ev[i].elapsed_time(ev[i + 1]) / reps
    pq = float(m.compute())
    frame = sum(tot)
    return {"render_fp32_ms": round(tot[0], 3), "argmax_maps_ms": round(tot[1], 4), "pq_update_ms": round(tot[2], 4),
            "pq_share_of_frame": round(tot[2] / frame, 6), "segments_pred": int(len((maps[0, ..., 0] * 256 + maps[0, ..., 1]).unique())),
            "pq": pq, "frames": reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pq_bench needs a CUDA device (no CPU fallback)")
    dev = torch.device("cuda:0")
    name, power = card()
    res = {"tool": "pq_bench", "gpu": name, "power_limit": power,
           "update": [time_updates(1024, 1024, args.frames, dev), time_updates(720, 1280, args.frames, dev)],
           "cpu_oracle": time_oracle(), "validation_frame": time_validation_frame(dev)}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
