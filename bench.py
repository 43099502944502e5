#!/usr/bin/env python
"""bench.py -- PAg-NeRF hot path on B200.  Default = BASELINE.json config[1] ("config 2" in BASELINE.md's 1-based table):
rays/s of a training step (march + encode + decode + composite + backward) of
  PanopticDeltaNeF + permutohedral grid (L=24, F=2, T=2^18, colour + delta grid), BUP20-shaped 1 MP
  camera, 16 384 rays / step / GPU, occupancy-octree 'ray' march with 128 steps on a pruned level-7 octree.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 1|2|3|4|5] [--march ray|voxel]
                  [--dump-outputs DIR]
Prints ONE JSON line (rank 0).  The other BASELINE configs (1-based, BASELINE.md section 3):
  1  PanopticDeltaNeF + hash_grid_torch (L=16, T=2^19), 4 096 rays x 64 samples (the reference's CPU-runnable case)
  3  PanopticNeF + tcnn-style hash grid (L=14, T=2^19, base 16), 65 536 rays x 128 samples dense
  4  config 2's model + pose gradients (BAPipeline) + Adam + gradient all-reduce, 65 536 rays / GPU
  5  inference: one 1 048 576-ray frame, rgb + depth + semantics(6) + instances(200), forward only -> frames/s
`--impl reference` times the reference's own torch CPU path (north_star: grids/hash_grid_torch.py + torch MLPs + torch
compositing; restated in oracle/, pinned to the verbatim reference file by tests/golden/hash_torch.npz) on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_RAYS = 16384
NUM_STEPS = 128
LEVEL = 7
L, F, CAP_LOG2 = 24, 2, 18
C_SEM, C_INST = 6, 200
RAYS_PER_IMG = 4096
NEAR, FAR = 0.0, 2.0

# BASELINE.json configs (1-based like BASELINE.md).  scene: 'pruned' = slab + blobs (a few % of the level-7 cells), 'dense' =
# the pre-prune 128^3 occupancy (grids/occtree.py:60) with rays confined to the cube so that every ray keeps all S samples
CONFIGS = {
    1: dict(field='delta', grid='hashtorch', levels=16, rays=4096, S=64, scene='dense', mode='train', far=1.7,
            workload="PanopticDeltaNeF + hash_grid_torch (L=16,F=2,T=2^19 x2, 16..2048), 4096 rays x 64 samples dense packing"),
    2: dict(field='delta', grid='permuto', levels=24, rays=16384, S=128, scene='pruned', mode='train', far=FAR,
            workload="PanopticDeltaNeF + permutohedral grid (L=24,F=2,T=2^18 x2), BUP20-shaped 1MP frame, 16384 rays/step/GPU, "
                     "occtree 'ray' march 128 steps, level-7 pruned octree"),
    3: dict(field='nef', grid='tcnn', levels=14, rays=65536, S=128, scene='dense', mode='train', far=1.7,
            workload="PanopticNeF (no delta grid) + tcnn-style hash grid (L=14,F=2,T=2^19, base 16 x2/level), 65536 rays x 128 samples dense"),
    4: dict(field='delta', grid='permuto', levels=24, rays=65536, S=128, scene='pruned', mode='train', far=FAR, pose=True, adam=True,
            workload="config 2 model + pose optimisation (6-DoF per image) + Adam + gradient all-reduce, 65536 rays/GPU"),
    5: dict(field='delta', grid='permuto', levels=24, rays=1048576, S=128, scene='pruned', mode='infer', far=FAR,
            workload="inference render of one 1024x1024 frame (1 048 576 rays): rgb+depth+semantics(6)+inst(200), forward only, "
                     "random-init PanopticDeltaNeF + permutohedral grid, level-7 pruned octree, 128 march steps"),
}


# ------------------------------------------------------------------------------------------------
# synthetic BUP20-shaped workload (SURVEY 8d): scene, cameras, rays, targets
# ------------------------------------------------------------------------------------------------
def make_scene(level=LEVEL, seed=0):
    """Pruned occupancy: slab |z| < 0.15 plus 200 blobs r = 0.05 (a few % of the level-7 cells)."""
    rng = np.random.default_rng(seed)
    n = 1 << level
    ax = (np.arange(n) + 0.5) / n * 2 - 1
    occ = np.zeros((n, n, n), dtype=bool)
    occ[:, :, np.abs(ax) < 0.15] = True
    ctr = rng.uniform(-0.9, 0.9, (200, 3))
    r = 0.05
    for c in ctr:
        lo = np.clip(((c - r + 1) / 2 * n).astype(int), 0, n - 1)
        hi = np.clip(((c + r + 1) / 2 * n).astype(int) + 1, 1, n)
        sub = np.stack(np.meshgrid(ax[lo[0]:hi[0]], ax[lo[1]:hi[1]], ax[lo[2]:hi[2]], indexing="ij"), -1)
        occ[lo[0]:hi[0], lo[1]:hi[1], lo[2]:hi[2]] |= np.linalg.norm(sub - c, axis=-1) < r
    return np.argwhere(occ).astype(np.int16)


def make_rays(n_rays, step, seed=0, res=1024, confined=False):
    """`n_rays/4096` images x 4096 random pixels; pinhole res x res, focal 0.9*res; cameras on the line
    x in [-0.8, 0.8] at z = +0.9 looking down -z with 2 degrees of seeded jitter.
    confined: narrower frustum (focal 2*res) from x, y in [-0.4, 0.4] so that every sample up to t = 1.7 stays inside
    the unit cube -- the dense N x S packing of BASELINE configs 1 and 3 (every ray keeps all its samples)."""
    rng = np.random.default_rng(seed * 100003 + step)
    n_img = max(1, n_rays // RAYS_PER_IMG)
    per = n_rays // n_img
    os_, ds_ = [], []
    for _ in range(n_img):
        cam = np.array([rng.uniform(-0.8, 0.8), rng.uniform(-0.05, 0.05), 0.9])
        focal = 0.9 * res
        if confined:
            cam = np.array([rng.uniform(-0.4, 0.4), rng.uniform(-0.4, 0.4), 0.9])
            focal = 2.0 * res
        pix = rng.integers(0, res, size=(per, 2)).astype(np.float64) + 0.5
        d = np.stack([(pix[:, 0] - res / 2) / focal, (pix[:, 1] - res / 2) / focal, -np.ones(per)], 1)
        ang = np.deg2rad(rng.normal(0, 2.0, 2))
        if confined:
            ang = np.clip(ang, -np.deg2rad(3.0), np.deg2rad(3.0))
        cx, sx, cy, sy = np.cos(ang[0]), np.sin(ang[0]), np.cos(ang[1]), np.sin(ang[1])
        Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
        Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
        d = d @ (Ry @ Rx).T
        d /= np.linalg.norm(d, axis=1, keepdims=True)
        os_.append(np.tile(cam, (per, 1)))
        ds_.append(d)
    return np.concatenate(os_).astype(np.float32), np.concatenate(ds_).astype(np.float32)


def make_cameras(seed=0, n_cam=42):
    """The synthetic robot pass as view matrices [n_cam, 4, 4] (world -> camera): 42 poses on the line x in [-0.8, 0.8] at z = +0.9
    looking down -z with 2 degrees of seeded jitter (agrobot_base.py:110-113: 42 train frames)."""
    rng = np.random.default_rng(seed * 100003 + 4242)
    V = np.tile(np.eye(4), (n_cam, 1, 1))
    for i in range(n_cam):
        cam = np.array([-0.8 + 1.6 * i / (n_cam - 1), rng.uniform(-0.05, 0.05), 0.9])
        ang = np.deg2rad(rng.normal(0, 2.0, 2))
        cx, sx, cy, sy = np.cos(ang[0]), np.sin(ang[0]), np.cos(ang[1]), np.sin(ang[1])
        Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
        Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
        Rcw = Ry @ Rx                      # camera -> world
        V[i, :3, :3] = Rcw.T
        V[i, :3, 3] = -Rcw.T @ cam
    return V.astype(np.float32)


def make_base_rays(n_rays, step, seed=0, res=1024, n_cam=42):
    """Camera-space base rays (origin 0, unit pixel directions) of n_rays/4096 images + the camera index of each image: what
    BAPipeline.transform_rays consumes (data['base_rays'], pc_nerf/trainer.py:421)."""
    rng = np.random.default_rng(seed * 100003 + step + 99)
    n_img = max(1, n_rays // RAYS_PER_IMG)
    per = n_rays // n_img
    pix = rng.integers(0, res, size=(n_img * per, 2)).astype(np.float64) + 0.5
    d = np.stack([(pix[:, 0] - res / 2) / (0.9 * res), (pix[:, 1] - res / 2) / (0.9 * res), -np.ones(n_img * per)], 1)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    cams = rng.integers(0, n_cam, size=n_img).astype(np.int64)
    return np.zeros((n_img * per, 3), np.float32), d.astype(np.float32), cams


def make_targets(n_rays, step, seed=0):
    rng = np.random.default_rng(seed * 7919 + step + 1)
    return (rng.uniform(0, 1, (n_rays, 3)).astype(np.float32), rng.integers(0, C_SEM, n_rays).astype(np.int64),
            rng.integers(0, C_INST, n_rays).astype(np.int64))


NEF_KW = dict(grid_type="PermutoGrid", interpolation_type='linear', multiscale_type='cat', feature_dim=F, num_lods=L,
              base_lod=2, hidden_dim=64, num_layers=1, view_multires=4, pos_multires=10, embedder_type='positional',
              activation_type='relu', layer_type='none', num_classes=C_SEM, num_instances=C_INST,
              sem_num_layers=1, sem_hidden_dim=64, inst_num_layers=2, inst_hidden_dim=64, sem_softmax=True,
              inst_softmax=True, sem_detach=True, inst_detach=True, panoptic_features_type='delta', blas_level=LEVEL,
              coarsest_scale=1.0, finest_scale=1e-4, capacity_log_2=CAP_LOG2, delta_capacity_log_2=CAP_LOG2)


def nef_kwargs(cfg):
    """Constructor arguments of the field of a BASELINE config (configs/bup20/best.yaml shapes)."""
    kw = dict(NEF_KW)
    if cfg['grid'] == 'hashtorch':      # BASELINE.md section 2: L=16, F=2, T=2^19, base 16, finest 2048
        kw.update(grid_type="HashGridTorch", num_lods=16, codebook_bitwidth=19)
    elif cfg['grid'] == 'tcnn':         # BASELINE.md section 3 row 3: L=14, F=2, T=2^19, base 16, x2 per level
        kw.update(grid_type="HashGridTinyCudaNN", num_lods=14, codebook_bitwidth=19)
    if cfg['field'] == 'nef':
        kw.update(panoptic_features_type=None)
    return kw


def loss_fn(rb_rgb, rb_sem, rb_inst, t_rgb, t_sem, t_inst):
    """rgb L1 x10 + semantic NLL x0.1 + instance NLL (reference pc_nerf/trainer.py:442-480, log(x + 1e-27) :459).  On CUDA tensors
    the three terms and their gradients are one kernel each way (pagnerf_b200.loss.panoptic_loss); the torch formulation below is
    what it is checked against (tests/test_gpu_parity.py::test_fused_panoptic_loss) and what the CPU reference arm runs."""
    if rb_rgb.is_cuda and os.environ.get("BENCH_TORCH_LOSS") != "1":
        from pagnerf_b200.loss import panoptic_loss
        return panoptic_loss(rb_rgb, rb_sem, rb_inst, t_rgb, t_sem, t_inst, 10.0, 0.1, 1.0, 1e-27)
    l = 10.0 * torch.abs(rb_rgb - t_rgb).mean()
    # nll_loss(log(p + eps), t) == -mean(log(p[i, t_i] + eps)): same value and gradient, but the log / its backward touch N
    # entries instead of N x C, and torch's single-block nll_loss reduction kernels (20 us each at N = 16384) are avoided --
    # the loss is outside the measured hot path (SURVEY 8f rank 3), it only has to drive the backward
    l = l - 0.1 * torch.log(rb_sem.gather(1, t_sem[:, None]) + 1e-27).mean()
    l = l - 1.0 * torch.log(rb_inst.gather(1, t_inst[:, None]) + 1e-27).mean()
    return l


class Workload:
    """The hot path of one BASELINE config on one GPU through the plugin classes."""

    def __init__(self, device, n_rays=None, seed=0, n_batches=4, amp=True, dd=False, config=2, march='ray'):
        """dd: the PanopticDDensity field + tracer pair (7 of the reference's 13 bup20 configs) instead of the delta field."""
        self.amp = amp
        from pagnerf_b200.pc_nerf import PanopticDeltaNeF, PanopticDDensityNeF, PanopticNeF
        from pagnerf_b200.tracers import PanopticPackedRFTracer, PanopticDDensityPackedRFTracer
        from pagnerf_b200 import spc
        cfg = self.cfg = CONFIGS[config]
        n_rays = int(n_rays or cfg['rays'])
        torch.manual_seed(seed)
        self.device, self.n_rays, self.S, self.far = device, n_rays, cfg['S'], cfg['far']
        cls = PanopticNeF if cfg['field'] == 'nef' else (PanopticDDensityNeF if dd else PanopticDeltaNeF)
        self.nef = cls(**nef_kwargs(cfg))
        grids = [self.nef.grid] + ([self.nef.delta_grid] if hasattr(self.nef, 'delta_grid') else [])
        octree = spc.unbatched_points_to_octree(torch.from_numpy(make_scene(LEVEL, seed)), LEVEL) if cfg['scene'] == 'pruned' else None
        for g in grids:
            if cfg['grid'] == 'permuto':
                g.init_from_scales()
            elif cfg['grid'] == 'hashtorch':
                g.init_from_geometric(16, 2048, 16)          # config_parser.py:733 (tree_type geometric)
            else:
                g.init_from_resolutions([16 * 2 ** i for i in range(14)])
            if octree is not None:
                g.blas_init(octree)
        with torch.no_grad():  # random-init field, but opaque enough that compositing terminates like a trained one
            for g in grids:
                for name in ('lattice_values', 'params', 'embeddings_weight'):
                    if hasattr(g.embedder, name):
                        getattr(g.embedder, name).mul_(1e3)
        self.nef = self.nef.to(device)
        self.tracer = (PanopticDDensityPackedRFTracer if dd else PanopticPackedRFTracer)(
            raymarch_type=march, num_steps=(cfg['S'] if march == 'ray' else 2), bg_color='white', ray_max_travel=2.0)
        self.params = [p for p in self.nef.parameters()]
        self.channels = ['rgb', 'depth', 'semantics', 'inst_embedding']
        self.pipe = self.optimizer = None
        if cfg.get('pose'):
            # bundle adjustment (pc_nerf/ba_pipeline.py): 42 trainable camera poses, frame 0 anchored
            from pagnerf_b200.pc_nerf import BAPipeline
            self.pipe = BAPipeline(self.nef, torch.from_numpy(make_cameras(0)), self.tracer, anchor_frame_idxs=[0], near=NEAR, far=self.far).to(device)
            self.params.append(self.pipe.camera_extrinsics)
        if cfg.get('adam'):
            # the reference's parameter groups (pc_nerf/trainer.py:229-300; best.yaml: lr 1e-3, grid / delta-grid lr x 100,
            # extrinsics lr 1e-4, wisp's Adam eps 1e-15)
            from pagnerf_b200.optim import FusedAdam
            named = dict(self.nef.named_parameters())
            groups = [dict(params=[p for n, p in named.items() if 'decoder' in n], lr=1e-3, name='decoder'),
                      dict(params=[p for n, p in named.items() if 'decoder' not in n and 'delta_grid' in n], lr=1e-1, name='delta_grid'),
                      dict(params=[p for n, p in named.items() if 'decoder' not in n and 'delta_grid' not in n], lr=1e-1, name='grid')]
            if self.pipe is not None:
                groups.append(dict(params=[self.pipe.camera_extrinsics], lr=1e-4, name='extrinsics'))
            self.optimizer = FusedAdam(groups, eps=1e-15)
        # pool of host (pinned) batches; step i uses batch i % n_batches
        self.host = []
        for b in range(n_batches):
            if self.pipe is not None:
                o, d, cams = make_base_rays(n_rays, b, seed)
            else:
                o, d = make_rays(n_rays, b, seed, confined=(cfg['scene'] == 'dense'))
            tr, ts, ti = make_targets(n_rays, b, seed)
            hb = [torch.from_numpy(x) for x in ((o, d, tr, ts, ti) + ((cams,) if self.pipe is not None else ()))]
            if device.type == 'cuda':
                hb = [x.pin_memory() for x in hb]
            self.host.append(hb)
        self.dev = [[x.to(device) for x in hb] for hb in self.host]
        self.step_idx = 0
        self.keep_rb = True

    def h2d_bytes(self):
        return sum(x.numel() * x.element_size() for x in self.host[0])

    def render(self, o, d, cams=None):
        from pagnerf_b200.wisp_compat import Rays
        rays = Rays(origins=o, dirs=d, dist_min=NEAR, dist_max=self.far)
        if self.pipe is not None:      # camera-space base rays -> world rays through the trainable poses, then the trace
            return self.pipe(channels=self.channels, rays=rays, cam_ids=cams, lod_idx=None, stage='train')
        return self.tracer(self.nef, channels=self.channels, rays=rays, lod_idx=None, stage='train')

    def after_backward(self):
        """What follows loss.backward() in the reference's step: (multi-GPU) the all-reduce of the gradients produced outside the
        fused trace -- the pose table --, then optimizer.step() (pc_nerf/trainer.py:582-590)."""
        import torch.distributed as dist
        if self.pipe is not None and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            g = self.pipe.camera_extrinsics.grad
            if g is not None:
                dist.all_reduce(g, op=dist.ReduceOp.AVG)
        if self.optimizer is not None:
            self.optimizer.step()

    def loss_of(self, o, d, tr, ts, ti, cams=None):
        """forward + loss of one step (what a trainer's step() does between zero_grad and backward)."""
        # the reference's training step runs under autocast (pc_nerf/trainer.py:429): fp16-rounded coords,
        # fp16-operand / fp32-accumulate decoders; the loss scaling of its GradScaler happens inside our kernels
        with torch.autocast('cuda', dtype=torch.float16, enabled=self.amp):
            rb = self.render(o, d, cams)
            loss = loss_fn(rb.rgb.float(), rb.semantics.float(), rb.inst_embedding.float(), tr, ts, ti)
        # NB: keeping `rb` alive keeps its autograd graph -- and the parameters' AccumulateGrad nodes, which remember the
        # stream they were created on -- alive; CUDA-graph capture needs them re-created on the capture stream.
        self.last_rb = rb if self.keep_rb else None
        # detached views of the rendered channels (no autograd graph): under CUDA-graph replay these are the graph's static
        # output buffers, refreshed by every replay; --dump-outputs reads them
        self.last_out = {c: getattr(rb, c).detach() for c in self.channels + ['alpha'] if getattr(rb, c, None) is not None}
        return loss

    def batch(self, from_host=False):
        b = self.step_idx % len(self.host)
        self.step_idx += 1
        if from_host:
            return self.host[b]
        return self.dev[b]

    def forward_backward(self, batch=None, from_host=False):
        b = self.batch(from_host)
        if from_host:
            b = [x.to(self.device, non_blocking=True) for x in b]
        for p in self.params:
            p.grad = None
        loss = self.loss_of(*b)
        loss.backward()
        self.after_backward()
        return {"rb": self.last_rb, "loss": loss, "ridx": getattr(self.tracer, "_last_ridx", torch.zeros(1, device=self.device))}


def build_workload(device, n_rays=N_RAYS, seed=0):
    return Workload(device, n_rays, seed)


# ------------------------------------------------------------------------------------------------
# CPU reference arm: the reference's own torch CPU path (north_star / BASELINE.md section 2), bounded sample
# ------------------------------------------------------------------------------------------------
class CpuReference:
    """grids/hash_grid_torch.HashEmbedder (x2: colour + delta grid; L=16, F=2, T=2^19, base 16, finest 2048) + torch nn.Linear
    decoders (density 32-64-16, colour 43-64-64-3, semantics 32-64-6, instances 32-64-64-200; stop-gradient and fusion as
    pc_nerf/panoptic_delta_nef.py:170-257) + torch compositing (exponential_integration / sum_reduce restated with cumsum, two
    integrations, alpha on top, white background, tracers/panoptic_packed_rf_tracer.py:134-205), fixed dense packing (every ray
    keeps S jittered samples: the reference has no CPU marcher), L1 rgb + NLL semantics + NLL instances, loss.backward(); fp32,
    no autocast, no optimiser step.  The hash grid is oracle/hashgrid.HashEmbedderOracle: same torch ops as the reference file,
    pinned to it bit-exactly (indices) / 1e-6 (features) by tests/golden/hash_torch.npz -- /root/reference itself does not exist
    on the GPU box.  This is the only CPU-runnable path the reference has (its permutohedral / tcnn grids are CUDA extensions)."""

    def __init__(self, n_rays, S, delta=True, seed=0):
        from oracle.field import FieldOracle
        from oracle.hashgrid import HashEmbedderOracle
        torch.manual_seed(seed)
        grid = HashEmbedderOracle(16, 2, 19, 16, 2048, seed=seed)
        dgrid = HashEmbedderOracle(16, 2, 19, 16, 2048, seed=seed + 1) if delta else None
        with torch.no_grad():
            grid.embeddings.mul_(1e3)
            if dgrid is not None:
                dgrid.embeddings.mul_(1e3)
        self.field = FieldOracle(grid, dgrid, feat_dim=32, num_classes=C_SEM, num_instances=C_INST)
        self.n_rays, self.S, self.seed, self.i = n_rays, S, seed, 0

    def step(self, train=True):
        from oracle.field import trace_oracle
        N, S = self.n_rays, self.S
        o, d = [torch.from_numpy(x) for x in make_rays(N, self.i, self.seed, confined=True)]
        tr, ts, ti = [torch.from_numpy(x) for x in make_targets(N, self.i, self.seed)]
        g = torch.Generator().manual_seed(self.i)
        self.i += 1
        t = (torch.arange(S, dtype=torch.float32)[None, :] + torch.rand(N, S, generator=g)) * (1.7 / S)      # near 0, far 1.7
        samples = (o[:, None, :] + d[:, None, :] * t[:, :, None]).reshape(N * S, 1, 3)
        deltas = torch.diff(t, dim=1, prepend=torch.zeros(N, 1)).reshape(N * S, 1)
        boundary = torch.zeros(N * S, dtype=torch.bool)
        boundary[::S] = True
        ridx = torch.arange(N).repeat_interleave(S)
        for p in self.field.parameters():
            p.grad = None
        chans = ['rgb', 'depth', 'semantics', 'inst_embedding']
        with torch.set_grad_enabled(train):
            out = trace_oracle(self.field, o, d, ridx, samples, t.reshape(N * S, 1), deltas, boundary, chans)
            if not train:
                return 0.0
            loss = loss_fn(out['rgb'], out['semantics'], out['inst_embedding'], tr, ts, ti)
        loss.backward()
        return float(loss.detach())


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def time_cpu_reference(n_rays, S, steps, warmup, delta=True, train=True):
    """-> (rays/s, s/step, threads) of the reference's torch CPU path on all host cores."""
    torch.set_num_threads(os.cpu_count())
    ref = CpuReference(n_rays, S, delta=delta)
    for _ in range(warmup):
        ref.step(train)
    t0 = time.perf_counter()
    for _ in range(steps):
        ref.step(train)
    dt = (time.perf_counter() - t0) / steps
    return n_rays / dt, dt, torch.get_num_threads()


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
                for n, v in zip(names, f[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# main
# ------------------------------------------------------------------------------------------------
def measured_traffic(kernel):
    """dram bytes per launch of `kernel` from the committed ncu --set full capture of this same command
    (profiles/r02_traffic.json: {entry point: {"dram_bytes": .., "samples": ..}}), rescaled to this run's sample count."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            hit = json.load(open(p)).get(kernel)
            if hit:
                return hit
    return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return j["hbm_gbs"], j.get("bf16_tflops_sustained", j["bf16_tflops"]), "measured (MEASURED_PEAKS.json; bf16 sustained)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


DUMP_MAX_ELEMENTS = 1 << 20      # per array: 4 MB as float32
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """--dump-outputs: write {name: tensor} as path/<name>.npy, float64 kept, everything else as float32.  An array of more than
    DUMP_MAX_ELEMENTS elements is stored as a 1-D sample of its flattened elements at sorted indices drawn with a fixed seed: the
    same positions for the same shape in every run, so that the dumps of two builds can be compared element for element."""
    out = {}
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMENTS:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_MAX_ELEMENTS, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        out[name] = t.cpu().numpy().astype(np.float64 if t.dtype == torch.float64 else np.float32)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


def _leave(world, dist=None):
    """Multi-rank exit: barrier (every rank still alive), then tear the NCCL communicator down properly.  A watchdog turns a
    teardown that hangs (captured graphs still holding NCCL kernels have done that) into a loud message instead of a stuck job."""
    if world <= 1:
        return
    sys.stdout.flush()
    sys.stderr.flush()
    torch.cuda.synchronize()

    def _watchdog():
        time.sleep(30.0)
        print("[bench] WARNING: NCCL teardown did not finish within 30 s; exiting the process directly", file=sys.stderr, flush=True)
        os._exit(0)

    threading.Thread(target=_watchdog, daemon=True).start()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def algo_table(levels):
    """ALGORITHMIC bytes / flops per packed sample of every entry point (SURVEY 8d; DESIGN.md "Kernels"); `levels` = grid levels.
    Encoders: 12 B position + vertex reads/RMW (4 x 8 B per level permutohedral, 8 x 8 B hash: the tables are f32) + features
    (f32 rows, or halfs in the fp16 operand-image interchange)."""
    Lv = levels
    IN = 2 * Lv
    dc = 2 * (IN * 64 + 64 * 16 + 43 * 64 + 64 * 64 + 64 * 3)
    pan = 2 * (IN * 64 + 64 * C_SEM + IN * 64 + 64 * 64 + 64 * C_INST)
    t = {
        "pag_permuto_fwd_dyn": ("l2", 12 + Lv * 4 * 8 + Lv * 2 * 4), "pag_permuto_bwd_dyn": ("l2", 12 + Lv * 2 * 4 + 2 * Lv * 4 * 8),
        "pag_permuto_fwd_img16_dyn": ("l2", 12 + Lv * 4 * 8 + Lv * 2 * 2), "pag_permuto_bwd_img16_dyn": ("l2", 12 + Lv * 2 * 2 + 2 * Lv * 4 * 8),
        "pag_permuto_fwd": ("l2", 12 + Lv * 4 * 8 + Lv * 2 * 4), "pag_permuto_bwd": ("l2", 12 + Lv * 2 * 4 + 2 * Lv * 4 * 8),
        "pag_hash_fwd_dyn": ("l2", 12 + Lv * 8 * 8 + Lv * 2 * 4), "pag_hash_bwd_dyn": ("l2", 12 + Lv * 2 * 4 + 2 * Lv * 8 * 8),
        "pag_hash_fwd_img16_dyn": ("l2", 12 + Lv * 8 * 8 + Lv * 2 * 2), "pag_hash_bwd_img16_dyn": ("l2", 12 + Lv * 2 * 2 + 2 * Lv * 8 * 8),
        "pag_composite_fwd": ("hbm", 4 + 4 + 4 + 12 + 8), "pag_composite_bwd": ("hbm", 2 * (4 + 4 + 4 + 12) + 8),
    }
    for k in ("pag_decode_dc_fwd_tc_dyn", "pag_decode_dc_fwd_tc", "pag_decode_dc_fwd"):
        t[k] = ("tensor", dc)
    for k in ("pag_decode_dc_bwd_tc_dyn", "pag_decode_dc_bwd_tc", "pag_decode_dc_bwd"):
        t[k] = ("tensor", 3 * dc)
    for k in ("pag_pan_composite_fwd_tc", "pag_decode_pan_fwd_tc", "pag_decode_pan_fwd"):
        t[k] = ("tensor", pan)
    for k in ("pag_decode_pan_bwd_tc", "pag_decode_pan_bwd"):
        t[k] = ("tensor", 3 * pan)
    t["pag_pan_composite_bwd_tc"] = ("tensor", 4 * pan)      # forward recomputed inside the backward
    return t


def l2_probe(device):
    """Measured L2 read bandwidth (GB/s): pag_l2_stream_probe streams a 64 MB buffer (resident in the 126 MB L2 after the
    first pass) with coalesced 16-byte loads."""
    from pagnerf_b200 import _lib
    buf = torch.zeros(64 << 20, dtype=torch.uint8, device=device)
    sink = torch.zeros(148 * 8 * 256, dtype=torch.float32, device=device)
    iters = 8
    for _ in range(2):
        _lib.call("pag_l2_stream_probe", _lib.ptr(buf), buf.numel(), iters, _lib.ptr(sink))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        _lib.call("pag_l2_stream_probe", _lib.ptr(buf), buf.numel(), iters, _lib.ptr(sink))
    e1.record()
    torch.cuda.synchronize()
    return buf.numel() * iters * 5 / (e0.elapsed_time(e1) * 1e-3) / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE config, 1-based (default 2 = the headline)")
    ap.add_argument("--march", default="ray", choices=["ray", "voxel"], help="octree marching mode of the training trace (config 2)")
    ap.add_argument("--rays", type=int, default=None, help="rays per step per GPU (default: the config's)")
    ap.add_argument("--cpu-sample-rays", type=int, default=1024, help="rays per step of the CPU reference leg (bounded sample)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time the eager step instead of the CUDA-graph replay")
    ap.add_argument("--infer-precision", default="fp32", choices=["fp32", "tc"],
                    help="config 5: decoders in exact fp32 (the reference validates without autocast, pc_nerf/trainer.py:683) or on the "
                         "tensor cores (fp16 operands); fp32 is the reported value, tc is reported beside it")
    ap.add_argument("--dd", action="store_true", help="PanopticDDensity field + tracer (own panoptic density stream) instead of the "
                                                      "BASELINE config-2 delta field; informational, not the headline workload")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (rank 0's): training: the "
                         "loss, the rendered channels and every parameter gradient; config 5: the frame's rgb, depth and label maps "
                         "(git ignores bench_outputs/)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    cfg = CONFIGS[args.config]
    infer = cfg['mode'] == 'infer'
    if args.steps is None:
        args.steps = 10 if infer else (50 if cfg['rays'] > 16384 else 200)
    if args.warmup is None:
        args.warmup = 3 if infer else 10
    rays = int(args.rays or cfg['rays'])
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    workload = cfg['workload'].replace("PanopticDeltaNeF", "PanopticDDensityNeF + DD tracer") if args.dd else cfg['workload']
    if args.march == 'voxel':
        workload = workload.replace("occtree 'ray' march 128 steps", "occtree 'voxel' march, 2 samples per voxel, ray_max_travel 2.0")
    config = {"workload": workload + ("; rgb+depth+semantics(6)+inst(200); fwd+bwd" if not infer else ""),
              "baseline_config": args.config, "rays_per_gpu": rays if not infer else rays // world,
              "parallelism": (f"ray-sharded dp{world}" if world > 1 else "single")}
    metric = ("inference frames/s (1 MP rgb+depth+semantic+instance maps)" if infer
              else "train rays/s (march+encode+decode+composite+backward)")
    unit = "frames/s" if infer else "rays/s"

    if args.impl == "reference":
        if rank != 0:
            return 0
        # the reference's torch CPU path on a bounded sample of the workload: cpu_sample_rays rays x 64 samples per step
        # (BASELINE.md section 2 packing); config 1 IS that path at its full 4 096 rays.  K steps after W warm-ups, as asked.
        n_cpu = rays if args.config == 1 else min(rays, args.cpu_sample_rays)
        rps, dt, threads = time_cpu_reference(n_cpu, 64, args.steps, args.warmup, delta=(cfg['field'] != 'nef'), train=not infer)
        value = rps / (1024 * 1024) if infer else rps
        out = {"impl": "reference", "metric": metric, "value": value, "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": "f32", "data": "synthetic", "config": config,
               "cpu_baseline": {"value": value, "unit": unit, "cores": threads, "kind": "port", "cpu": cpu_model(),
                                "sample": f"{n_cpu} rays x 64 samples per step (dense packing), the reference's torch CPU path: HashEmbedder x"
                                          f"{1 if cfg['field'] == 'nef' else 2} (L=16,T=2^19) + nn.Linear decoders + torch compositing, "
                                          + ("forward only" if infer else "fwd + loss + backward") + ", fp32, all host threads"},
               "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(out))
        return 0

    import torch.distributed as dist
    from pagnerf_b200 import _lib, parallel

    def trace(msg):      # BENCH_TRACE=1: progress marks on stderr (debugging multi-rank runs)
        if os.environ.get("BENCH_TRACE"):
            print(f"[bench rank {rank}] {msg}", file=sys.stderr, flush=True)

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
        trace("process group up")
    if infer:
        return bench_inference(args, cfg, config, metric, unit, rank, world, device, dist)
    # BENCH_SAME_SEED=1 (diagnostic): every rank traces the same rays -> no load imbalance between the ranks
    wl = Workload(device, rays, seed=0 if os.environ.get('BENCH_SAME_SEED') == '1' else rank, dd=args.dd, config=args.config, march=args.march)
    trace("workload built")
    transport, transport_fallback = None, None
    if world > 1:
        from pagnerf_b200 import ops
        # gradient exchange issued from inside the fused backward.  Default: the tables live in symmetric memory and are reduced in
        # place by csrc/allreduce.cu over NVLink / NVSwitch peer memory (exact fp32); PAGNERF_GRAD_TRANSPORT=fp32|fp16 selects NCCL.
        transport = os.environ.get("PAGNERF_GRAD_TRANSPORT", "symm")
        if transport == "symm":
            # symmetric memory needs P2P / multicast capable peers: probe it once (collectively); without it the exchange falls
            # back to NCCL (exact fp32) and the JSON line says so -- never silently
            ok = 1
            try:
                from pagnerf_b200.parallel import SymmetricGradBuffers
                SymmetricGradBuffers({"probe": 1024}, device)
            except Exception as e:      # noqa: BLE001 -- any failure of the symmetric allocation / rendezvous
                ok = 0
                print(f"[bench] rank {rank}: symmetric memory unavailable ({e!r}); falling back to NCCL fp32", file=sys.stderr, flush=True)
            flag = torch.tensor([ok], device=device, dtype=torch.int32)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) == 0:
                transport, transport_fallback = "fp32", "symmetric memory unavailable on this box -> NCCL fp32"
        ops.set_grad_sync(True, reserved_sms=int(os.environ.get("BENCH_RESERVED_SMS", 0)), transport=transport)

    def step(from_host):
        return wl.forward_backward(from_host=from_host)

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(args.warmup, 3)):
        step(False)
        trace(f"warm-up step {i} enqueued")
    sync()
    trace("warm-up done")
    fused = torch.is_tensor(getattr(wl.tracer, 'last_num_samples', None))     # device-side sample count <=> sync-free fused trace
    # ---- CUDA-graph capture of the whole step (the fused path has static launch geometry) ---------------------------
    graphed, graph_note = None, "eager (--no-graph)" if args.no_graph else "eager (step-by-step plugin path: one host sync per march)"
    # multi-rank: NCCL all-reduces issued inside the backward are captured with the step (every rank captures the same sequence)
    if fused and not args.no_graph:
        # a failing capture fails the bench: an eager number must never be reported under the graph-replay label
        from pagnerf_b200.graph import GraphedStep
        wl.keep_rb, wl.last_rb = False, None
        graphed = GraphedStep(wl.loss_of, wl.dev[0], wl.params, wl.nef, post_backward=wl.after_backward)
        graph_note = "whole step (fwd + loss + bwd%s) replayed as one CUDA graph" % (" + NCCL gradient all-reduce" if world > 1 else "")
        trace("graph captured")

    def run(from_host):
        if graphed is None:
            return step(from_host)["loss"]
        return graphed(*wl.batch(from_host))      # host batches are pinned: copy_ into the static buffers is the H2D

    for _ in range(3):
        run(False)
    # ---- device-resident timing (value) ------------------------------------------------------------
    sync()
    clocks = ClockSampler(local) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = run(False)
    e1.record()
    sync()
    ms = e0.elapsed_time(e1) / args.steps
    trace(f"timed region done: {ms:.3f} ms/step")
    if args.dump_outputs and rank == 0:      # before the phases below run more steps over the same buffers
        named = list(wl.nef.named_parameters()) + ([("camera_extrinsics", wl.pipe.camera_extrinsics)] if wl.pipe is not None else [])
        dump_outputs(args.dump_outputs, {"loss": loss, **wl.last_out, **{"grad." + n: p.grad for n, p in named if p.grad is not None}})
    t_host0 = time.perf_counter()           # CPU time to enqueue a step into an empty stream (GPU-bound when << ms_per_step)
    for _ in range(3):
        run(False)
    host_enqueue_ms = (time.perf_counter() - t_host0) * 1e3 / 3
    sync()
    # ---- end-to-end timing (host pinned inputs -> H2D -> step -> D2H loss) -------------------------
    for _ in range(2):
        run(True)
    sync()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        _ = float(run(True).item())
    t1.record()
    sync()
    ms_e2e = t0.elapsed_time(t1) / args.steps
    # ---- multi-GPU: the same graph with the gradient all-reduces switched off = compute only; the difference is the exposed
    #      all-reduce time (SURVEY 8e "allreduce exposed ms") ------------------------------------------------------------
    ms_nosync = None
    if world > 1 and graphed is not None:
        from pagnerf_b200 import ops as _o
        _o.set_grad_sync(False)
        g2 = GraphedStep(wl.loss_of, wl.dev[0], wl.params, wl.nef, post_backward=wl.after_backward)
        for _ in range(3):
            g2(*wl.batch(False))
        sync()
        n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0.record()
        for _ in range(args.steps):
            g2(*wl.batch(False))
        n1.record()
        sync()
        ms_nosync = n0.elapsed_time(n1) / args.steps
        del g2
        _o.set_grad_sync(True, reserved_sms=int(os.environ.get("BENCH_RESERVED_SMS", 0)), transport=transport)
    # ---- per-entry-point CUDA-event timing of the same step, eager (events cannot be read back from a graph) ---------
    ksteps = min(args.steps, 20)
    sync()
    wl.keep_rb = True
    from pagnerf_b200 import ops as _ops
    _ops.BRANCH_OVERLAP = False            # serialise the two branch streams so that per-kernel durations are exclusive
    _lib.timing_reset(True)
    l0 = _lib.launch_count
    for _ in range(ksteps):
        step(False)
    sync()
    launches = (_lib.launch_count - l0) // ksteps
    per_kernel = _lib.timing_report()
    for v in per_kernel.values():
        v["ms_per_step"] = v["ms_total"] / ksteps
    _lib.timing_reset(False)
    _ops.BRANCH_OVERLAP = True
    clk = clocks.stop() if clocks else None
    t = torch.tensor([ms, ms_e2e, ms_nosync or 0.0], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e, ms_nosync = float(t[0]), float(t[1]), (float(t[2]) if ms_nosync is not None else None)
    if rank != 0:
        _leave(world, dist)
        return 0

    hbm, tf, how = peaks()
    ALGO = algo_table(cfg['levels'])
    top = max(per_kernel.items(), key=lambda kv: kv[1]["ms_per_step"]) if per_kernel else None
    roof = None
    n_samples = wl.tracer.last_num_samples if hasattr(wl.tracer, "last_num_samples") else None
    if torch.is_tensor(n_samples):
        n_samples = int(n_samples.item())
    # zero-density samples are dropped after the density pass (exact): the kernels downstream of the compaction process
    # the live samples only; kernels launched twice per step (main + delta grid / density-only + full decode) see both counts
    live = getattr(_ops.FusedTraceFn, "last_live_dev", None)
    n_live = int(live.item()) if (fused and torch.is_tensor(live)) else n_samples
    n_all = n_samples
    l2_gbs = l2_probe(device)
    if top and top[0] in ALGO and n_samples:
        bound, per = ALGO[top[0]]
        dur = top[1]["ms_per_launch"] * 1e-3
        if bound in ("hbm", "l2"):
            ach = per * n_samples / dur / 1e9
            peak = l2_gbs if bound == "l2" else hbm
            roof = {"kernel": top[0], "bound": bound, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                    "frac_of_hbm_peak": ach / hbm, "hbm_peak": hbm,
                    "note": "gather/scatter over tables that stay L2 resident (DRAM traffic is ~0.1x the algorithmic bytes): the bound is the "
                            "L2 -> SM path, peak = L2 read bandwidth measured live by pag_l2_stream_probe (64 MB buffer, coalesced 16-byte "
                            "loads); the same figure against the measured HBM copy peak is kept as frac_of_hbm_peak" if bound == "l2" else None}
        else:
            ach = per * n_samples / dur / 1e12
            roof = {"kernel": top[0], "bound": "tensor", "achieved": ach, "peak": tf, "unit": "TFLOP/s", "frac": ach / tf, "traffic": None,
                    "note": "decoder flops vs the bf16 tensor peak"}
        tr = measured_traffic(top[0])
        if tr:
            roof["traffic"] = tr["dram_bytes"] * n_samples / tr["samples"]
            roof["traffic_source"] = "ncu --set full dram__bytes_read+write per launch (profiles/), scaled by packed samples"
        roof["peak_source"] = how
        roof["share_of_step"] = top[1]["ms_per_step"] / ms
        roof["samples_per_launch"] = n_samples
    # ---- encoder vs the memory system (BASELINE metric "encoder GB/s vs peak"; SURVEY 8d) -------------------------------
    encoder = encoder_report(wl, per_kernel, ALGO, n_all, n_live, hbm, l2_gbs, device) if cfg['grid'] == 'permuto' and fused else None
    cpu = None
    if not args.no_cpu_baseline:
        n_cpu = min(rays, args.cpu_sample_rays)
        v, dt, threads = time_cpu_reference(n_cpu, 64, 3, 1, delta=(cfg['field'] != 'nef'))
        cpu = {"value": v, "unit": "rays/s", "cores": threads, "kind": "port", "cpu": cpu_model(),
               "sample": f"{n_cpu} rays x 64 samples per step x 3 steps (dense packing), the reference's torch CPU path: HashEmbedder x"
                         f"{1 if cfg['field'] == 'nef' else 2} (L=16,T=2^19) + nn.Linear decoders + torch compositing, fwd + loss + backward, fp32"}
    total_rays = rays * world
    result = {"metric": metric, "value": total_rays / (ms * 1e-3),
              "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms,
              "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
              "dtype": "fp16 operands / f32 accumulate (decoders, tcgen05) + f32 (encoders, compositing) = the reference's autocast",
              "data": "synthetic",
              "config": config,
              "details": dict(l2="no explicit flush: ray batches cycle and the per-step working set (tables + their gradients + per-sample "
                                 "features and feature gradients, > 400 MB) exceeds the 126 MB L2",
                              packed_samples_per_step=n_all, live_samples_per_step=n_live, execution=graph_note,
                              kernel_breakdown="per-entry-point CUDA events over %d eager steps of the same workload" % ksteps),
              "e2e": {"value": total_rays / (ms_e2e * 1e-3), "unit": "rays/s", "h2d_bytes_per_step": wl.h2d_bytes(),
                      "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e},
              "gpu_launches": int(launches), "host_enqueue_ms_per_step": round(host_enqueue_ms, 3), "clocks": clk, "roofline": roof, "encoder": encoder, "cpu_baseline": cpu,
              "kernels_ms_per_step": {k: round(v["ms_per_step"], 4) for k, v in sorted(per_kernel.items(), key=lambda kv: -kv[1]["ms_per_step"])}}
    if ms_nosync is not None:
        result["allreduce"] = {"transport": {"symm": "own kernel over NVLink/NVSwitch peer memory (symmetric buffers; multimem.ld_reduce/st through the "
                                                     "switch multicast address at > 2 ranks, peer loads/stores at 2), exact fp32",
                                             "fp32": "NCCL all-reduce, fp32", "fp16": "NCCL all-reduce, tables as fp16 under a shared scale"}[transport],
                               "ms_per_step_without_allreduce": ms_nosync, "exposed_ms": ms - ms_nosync,
                               "note": "same CUDA graph captured with the gradient all-reduces switched off, max over ranks"}
        if transport_fallback:
            result["allreduce"]["fallback"] = transport_fallback
    print(json.dumps(result))
    _leave(world, dist)
    return 0


def make_frame_rays(res=1024, seed=0):
    """All res x res pixel rays of one pinhole camera of the synthetic pass (same intrinsics / pose family as make_rays)."""
    rng = np.random.default_rng(seed * 100003 + 77)
    cam = np.array([rng.uniform(-0.8, 0.8), rng.uniform(-0.05, 0.05), 0.9])
    ys, xs = np.meshgrid(np.arange(res) + 0.5, np.arange(res) + 0.5, indexing="ij")
    d = np.stack([(xs - res / 2) / (0.9 * res), (ys - res / 2) / (0.9 * res), -np.ones_like(xs)], -1).reshape(-1, 3)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return np.tile(cam, (res * res, 1)).astype(np.float32), d.astype(np.float32)


def bench_inference(args, cfg, config, metric, unit, rank, world, device, dist):
    """BASELINE config 5: full-frame render (pc_nerf/trainer.py:637-649 batch_render + :683 no autocast), frames/s.  One frame is
    split into row blocks across the ranks (strong scaling; the only exchange is the gather of the finished map tiles), every
    rank renders its block in chunks of `render_batch` rays under torch.no_grad()."""
    from pagnerf_b200 import _lib
    from pagnerf_b200.wisp_compat import Rays
    total = int(args.rays or cfg['rays'])
    res = int(round(total ** 0.5))
    assert res * res == total, "config 5 renders a square frame"
    per = total // world
    chunk = min(per, int(os.environ.get("BENCH_RENDER_BATCH", 131072)))
    wl = Workload(device, n_rays=4096, seed=0, n_batches=1, config=5)
    o_np, d_np = make_frame_rays(res)
    lo = rank * per
    host_o = torch.from_numpy(o_np[lo:lo + per]).pin_memory()
    host_d = torch.from_numpy(d_np[lo:lo + per]).pin_memory()
    dev_o, dev_d = host_o.to(device), host_d.to(device)
    chans = ['rgb', 'depth', 'semantics', 'inst_embedding']
    host_out = [torch.empty(per, 3).pin_memory(), torch.empty(per, 1).pin_memory(),
                torch.empty(per, dtype=torch.uint8).pin_memory(), torch.empty(per, dtype=torch.uint8).pin_memory()]

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def render_frame(o, d, precision):
        """-> rgb [per,3], depth [per,1], semantic labels u8 [per], instance labels u8 [per] (argmax maps, as evaluate_metrics)."""
        wl.nef.decoder_precision = 'fp16' if precision == 'tc' else 'fp32'
        outs = []
        with torch.no_grad():
            for c0 in range(0, per, chunk):
                rb = wl.tracer(wl.nef, channels=chans, rays=Rays(origins=o[c0:c0 + chunk], dirs=d[c0:c0 + chunk], dist_min=NEAR, dist_max=FAR),
                               lod_idx=None, stage='val')
                outs.append((rb.rgb, rb.depth, rb.semantics.argmax(-1).to(torch.uint8), rb.inst_embedding.argmax(-1).to(torch.uint8)))
        return [torch.cat([x[i] for x in outs]) for i in range(4)]

    def gather(maps):
        if world == 1:
            return maps
        out = []
        for m in maps:
            full = torch.empty((per * world,) + tuple(m.shape[1:]), dtype=m.dtype, device=device)
            dist.all_gather_into_tensor(full, m.contiguous())
            out.append(full)
        return out

    last_maps = {}

    def time_frames(precision, steps, warmup, e2e):
        for _ in range(max(warmup, 1)):
            gather(render_frame(dev_o, dev_d, precision))
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            if e2e:
                o, d = host_o.to(device, non_blocking=True), host_d.to(device, non_blocking=True)
                maps = render_frame(o, d, precision)
                for dst, src in zip(host_out, maps):
                    dst.copy_(src, non_blocking=True)
                torch.cuda.current_stream().synchronize()      # the frame is on the host
            else:
                last_maps[precision] = gather(render_frame(dev_o, dev_d, precision))
        e1.record()
        sync()
        t = torch.tensor([e0.elapsed_time(e1) / steps], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    prec = args.infer_precision
    clocks = ClockSampler(device.index or 0) if rank == 0 else None
    ms = time_frames(prec, args.steps, max(args.warmup, 3), False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(("rgb", "depth", "semantic_labels", "instance_labels"), last_maps[prec])))
    ms_e2e = time_frames(prec, args.steps, 1, True)
    other = 'tc' if prec == 'fp32' else 'fp32'
    ms_other = time_frames(other, max(2, args.steps // 3), 2, False)
    clk = clocks.stop() if clocks else None
    # per-entry-point breakdown of one frame (selected precision)
    wl.nef.decoder_precision = 'fp16' if prec == 'tc' else 'fp32'
    sync()
    _lib.timing_reset(True)
    l0 = _lib.launch_count
    render_frame(dev_o, dev_d, prec)
    per_kernel = _lib.timing_report()
    launches = _lib.launch_count - l0
    _lib.timing_reset(False)
    if rank != 0:
        _leave(world, dist)
        return 0
    hbm, tf, how = peaks()
    ALGO = algo_table(cfg['levels'])
    n_samples = 0
    with torch.no_grad():
        from pagnerf_b200 import ops
        blas = wl.nef.grid.blas
        for c0 in range(0, per, chunk):
            n_samples += int(ops.raymarch_ray(blas.octree, blas.prefix, dev_o[c0:c0 + chunk], dev_d[c0:c0 + chunk], LEVEL, wl.S, NEAR, FAR, seed=0)[6][-1])
    top = max(per_kernel.items(), key=lambda kv: kv[1]["ms_total"]) if per_kernel else None
    roof = None
    if top and top[0] in ALGO:
        bound, b = ALGO[top[0]]
        dur = top[1]["ms_total"] * 1e-3
        l2_gbs = l2_probe(device)
        if bound == "tensor":
            ach = b * n_samples / dur / 1e12
            roof = {"kernel": top[0], "bound": "tensor", "achieved": ach, "peak": tf, "unit": "TFLOP/s", "frac": ach / tf, "traffic": None}
        else:
            ach = b * n_samples / dur / 1e9
            peak = l2_gbs if bound == "l2" else hbm
            roof = {"kernel": top[0], "bound": bound, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None}
        roof.update(peak_source=how, share_of_step=top[1]["ms_total"] / ms, samples_per_launch=n_samples / max(top[1]["launches"], 1))
    cpu = None
    if not args.no_cpu_baseline:
        v, dt, threads = time_cpu_reference(args.cpu_sample_rays, 64, 3, 1, train=False)
        cpu = {"value": v / total, "unit": unit, "cores": threads, "kind": "port", "cpu": cpu_model(),
               "sample": f"{args.cpu_sample_rays} rays x 64 samples x 3 steps, forward only, the reference's torch CPU path, scaled to {total} rays per frame"}
    dt_note = {"fp32": "f32 (exact FMA decoders; the reference validates without autocast)", "tc": "fp16 operands / f32 accumulate (tcgen05 decoders) + f32"}
    result = {"metric": metric, "value": 1e3 / ms, "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms,
              "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": dt_note[prec], "data": "synthetic", "config": config,
              "details": dict(render_batch=chunk, packed_samples_per_frame_rank0=n_samples, rays_per_rank=per,
                              live_fraction_last_chunk=getattr(wl.nef, 'last_live_fraction', None),
                              live_note="share of the packed samples whose integration weight exceeds ops.LIVE_WEIGHT_EPS (2^-30); when below "
                                        "ops.LIVE_COMPACT_FRAC the colour decoder, the delta-grid lookup and the heads run on those samples only",
                              other_precision={"dtype": dt_note[other], "frames_per_s": 1e3 / ms_other, "ms_per_frame": ms_other}),
              "e2e": {"value": 1e3 / ms_e2e, "unit": unit, "h2d_bytes_per_step": per * 24, "d2h_bytes_per_step": per * (12 + 4 + 1 + 1), "ms_per_step": ms_e2e,
                      "note": "pinned host rays -> H2D -> render -> argmax label maps -> D2H of rgb, depth, semantic and instance label maps (this rank's block)"},
              "gpu_launches": int(launches), "clocks": clk, "roofline": roof, "cpu_baseline": cpu,
              "kernels_ms_per_frame": {k: round(v["ms_total"], 4) for k, v in sorted(per_kernel.items(), key=lambda kv: -kv[1]["ms_total"])}}
    print(json.dumps(result))
    _leave(world, dist)
    return 0


def encoder_report(wl, per_kernel, ALGO, n_all, n_live, hbm, l2_gbs, device):
    """Permutohedral forward against the memory system: algorithmic GB/s vs HBM peak, vertex gathers vs the random-gather probe, and
    the L2-sector roofline: 32-byte sectors a warp instruction really touches (computed from this batch's lattice indices: lanes of
    a warp that hit the same sector share it) x 32 B / time, against the measured L2 read bandwidth."""
    from pagnerf_b200 import _lib, ops
    enc_name = "pag_permuto_fwd_img16_dyn" if "pag_permuto_fwd_img16_dyn" in per_kernel else "pag_permuto_fwd_dyn"
    enc = per_kernel.get(enc_name)
    if not enc or not n_all:
        return None
    enc_bytes = ALGO[enc_name][1]
    emb = wl.nef.grid.embedder
    table = emb.lattice_values.detach()
    entries = table.numel() // 2
    sink = torch.empty(n_all, device=device)
    for _ in range(3):
        _lib.call("pag_gather_probe", _lib.ptr(table), entries, n_all, 96, _lib.ptr(sink))
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for _ in range(10):
        _lib.call("pag_gather_probe", _lib.ptr(table), entries, n_all, 96, _lib.ptr(sink))
    g1.record()
    torch.cuda.synchronize()      # rank 0 only from here on: no barrier
    probe_gbs = n_all * 96 * 8 / (g0.elapsed_time(g1) / 10 * 1e-3) / 1e9
    t_enc = enc["ms_per_launch"] * 1e-3
    n_enc = (n_all + n_live) / 2          # two launches per step: colour grid (all samples) and delta grid (live samples)
    # sectors per warp instruction on a sample of the batch: one marched ray batch, first 32k packed samples
    sectors = None
    try:
        o, d = wl.dev[0][0], wl.dev[0][1]
        blas = wl.nef.grid.blas
        r = ops.raymarch_ray(blas.octree, blas.prefix, o, d, LEVEL, wl.S, NEAR, wl.far, seed=1)
        pos = r[2].reshape(-1, 3)[:32768].half().float().contiguous()
        m = (pos.shape[0] // 32) * 32
        idx, _, _ = ops.permuto_indices(pos[:m], emb.capacity, emb.scale_factor, emb.random_shift_per_level)      # [L, m, 4]
        sec = (idx.to(torch.int64) >> 2).view(idx.shape[0], m // 32, 32, 4).permute(0, 1, 3, 2)      # 8-byte entries: 4 per sector
        srt = torch.sort(sec, dim=-1).values
        distinct = 1 + (srt[..., 1:] != srt[..., :-1]).sum(-1)          # [L, warps, 4] sectors per warp-wide gather
        sectors = float(distinct.sum()) / m                                  # sectors per sample (<= 4 L)
        ln = torch.sort(sec >> 2, dim=-1).values                              # 128-byte lines: 16 entries each
        lines = float((1 + (ln[..., 1:] != ln[..., :-1]).sum(-1)).sum()) / m     # L1 wavefronts per sample (<= 4 L)
    except Exception as e:      # diagnostic only
        sectors = None
    rep = {"kernel": enc_name, "ms_per_launch": round(enc["ms_per_launch"], 4), "samples_per_launch": n_enc,
           "algorithmic_bytes_per_sample": enc_bytes,
           "algorithmic_GBps": enc_bytes * n_enc / t_enc / 1e9, "hbm_peak_GBps": hbm, "frac_of_hbm_peak": enc_bytes * n_enc / t_enc / 1e9 / hbm,
           "vertex_gather_GBps": 768 * n_enc / t_enc / 1e9, "achievable_gather_GBps": probe_gbs,
           "frac_of_achievable_gather": 768 * n_enc / t_enc / 1e9 / probe_gbs,
           "l2_read_peak_GBps": l2_gbs,
           "note": "algorithmic bytes = 12 pos + 768 vertex reads + features out (192 f32 / 96 fp16 image); achievable = pag_gather_probe: uniformly "
                   "random 8-byte loads, 16 in flight per thread, from the same 50 MB table (a lower bound of the achievable rate: neighbouring "
                   "samples share coarse-level vertices, the probe's addresses do not); l2_sector_*: distinct 32-byte sectors per warp-wide "
                   "gather (from this batch's lattice indices) x 32 B against the measured L2 read bandwidth"}
    if sectors is not None:
        sec_gbs = sectors * 32 * n_enc / t_enc / 1e9
        rep.update(l2_sectors_per_sample=sectors, l2_sector_GBps=sec_gbs, l2_sector_frac=sec_gbs / l2_gbs)
        # the tighter bound of a scattered gather: the L1/LSU processes ONE 128-byte line (wavefront) per cycle per SM whatever
        # the bytes used from it (B300_MICROARCH.md: rt_L1tex_wf ~ 1.0 cyc/wf); a warp-wide 8-byte gather that touches k distinct
        # lines costs k cycles of that pipe.  peak = 148 SMs x SM clock.
        clk = 1.965e9
        wf_rate = lines * n_enc / t_enc
        rep.update(l1_wavefronts_per_sample=lines, l1_wavefront_rate_G_per_s=wf_rate / 1e9, l1_wavefront_peak_G_per_s=148 * clk / 1e9,
                   l1_wavefront_frac=wf_rate / (148 * clk),
                   l1_note="distinct 128-byte lines per warp-wide vertex gather (this batch's lattice indices), one L1/LSU wavefront per "
                           "cycle per SM at 1965 MHz: the bound the kernel actually runs against (ncu: l1tex 69 %, lts 49 %, dram 4 %)")
    return rep


if __name__ == "__main__":
    sys.exit(main())
