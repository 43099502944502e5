"""CPU: host-side logic, the C-ABI library's symbol table, state_dict compatibility, multi-process plumbing."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol(cuda_lib):
    """The built .so loads and exports every prototype of include/pagnerf_b200.h (no compute call without a GPU)."""
    from pagnerf_b200 import _lib
    protos = _lib.parse_header()
    assert len(protos) >= 26
    out = subprocess.check_output(["nm", "-D", "--defined-only", _lib.LIB_PATH], text=True)
    exported = set(re.findall(r"\bT (pag_\w+)", out))
    assert set(protos) == exported, (set(protos) ^ exported)
    for name in protos:
        assert getattr(cuda_lib, name).argtypes is not None


def test_ops_refuse_cpu_tensors(cuda_lib):
    """No CPU fallback: the product path raises on CPU tensors instead of routing anywhere else."""
    from pagnerf_b200 import ops
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        ops.permuto_encode(torch.zeros(4, 3), torch.zeros(2, 8, 2), torch.ones(2, 3), torch.zeros(2, 3), torch.ones(2))
    with pytest.raises(RuntimeError, match="CUDA tensors only"):
        ops.octree_query(torch.zeros(1, dtype=torch.uint8), torch.zeros(2, dtype=torch.int32), torch.zeros(3, 3), 1)


def test_product_never_imports_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "pagnerf_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f


@pytest.mark.parametrize("level", [1, 3, 5])
def test_spc_build_matches_oracle(level):
    from oracle import spc as ospc
    from pagnerf_b200 import spc
    rng = np.random.default_rng(level)
    pts = rng.integers(0, 1 << level, size=(max(4, 8 ** level // 5), 3)).astype(np.int16)
    oc_ref = ospc.points_to_octree(pts, level)
    oc = spc.unbatched_points_to_octree(torch.from_numpy(pts), level)
    assert np.array_equal(oc.numpy(), oc_ref)
    p, py, pre = spc.scan_octree(oc, level)
    p_ref, py_ref, pre_ref = ospc.scan_octree(oc_ref, level)
    assert np.array_equal(p.numpy(), p_ref) and np.array_equal(py.numpy(), py_ref) and np.array_equal(pre.numpy(), pre_ref)
    assert spc.octree_max_level(oc) == level
    lp = spc.unbatched_get_level_points(p, py, level)
    assert set(map(tuple, lp.tolist())) == set(map(tuple, pts.tolist()))


def test_dense_octree_sizes_level7():
    """OctreeAS.init_dense(7): 299 593 bytes, 2 396 745 points, 2 097 152 leaves (SURVEY A.1)."""
    from pagnerf_b200 import spc
    blas = spc.OctreeAS('cpu')
    blas.init_dense(7)
    assert blas.octree.shape[0] == 299593 and blas.points.shape[0] == 2396745
    assert int(blas.pyramid[0, 7]) == 2097152 and tuple(blas.pyramid.shape) == (2, 9)


def test_plugin_surface_and_state_dict_keys():
    """Constructor kwargs, attributes and state_dict keys the reference's trainer / checkpoints rely on."""
    import bench
    from pagnerf_b200.pc_nerf import PanopticDeltaNeF
    from pagnerf_b200.tracers import PanopticPackedRFTracer
    kw = dict(bench.NEF_KW, blas_level=3, capacity_log_2=8, delta_capacity_log_2=7, some_unrelated_cli_arg=1)
    nef = PanopticDeltaNeF(**kw)
    nef.grid.init_from_scales(); nef.delta_grid.init_from_scales()
    assert nef.grid.capacity == 256 and nef.delta_grid.capacity == 128
    keys = set(nef.state_dict().keys())
    for g in ("grid", "delta_grid"):
        for k in ("blas_octree", "blas_points", "blas_prefix", "blas_pyramid", "embedder.lattice_values",
                  "embedder.random_shift_per_level", "embedder.scale_factor", "embedder.anneal_window"):
            assert f"{g}.{k}" in keys
    names = [n for n, _ in nef.named_parameters()]
    # optimiser grouping by substring (pc_nerf/trainer.py:240-258): decoder -> inst -> sem -> delta_grid -> grid
    assert sum('decoder' in n for n in names) == 20
    assert [n for n in names if 'decoder' not in n] == ['grid.embedder.lattice_values', 'delta_grid.embedder.lattice_values']
    assert float(nef.decoder_density.lout.bias[0]) == 1.0
    assert nef.get_supported_channels() == {"density", "rgb", "semantics", "inst_embedding"}
    assert nef.grid.num_lods == 24 and nef.grid.active_lods[-1] == 23 and nef.grid.multiscale_type == 'cat'
    assert nef.lod_weights.shape == (48,)
    tr = PanopticPackedRFTracer(raymarch_type='ray', num_steps=512, ray_max_travel=2.0, ray_sparcity_reg=0.0, extra=1)
    assert tr.raymarch_type == 'ray' and tr.num_steps == 512 and tr.get_required_nef_channels() == {'rgb', 'density'}
    tr.raymarch_type, tr.num_steps = 'voxel', 2   # pc_nerf/trainer.py:364-366 mutates these
    # pruned accel-struct round-trips through state_dict even though its size changed
    from pagnerf_b200 import spc
    oc = spc.unbatched_points_to_octree(torch.tensor([[0, 0, 0], [7, 7, 7], [3, 4, 5]], dtype=torch.int16), 3)
    nef.grid.blas_init(oc); nef.delta_grid.blas_init(oc)
    nef2 = PanopticDeltaNeF(**kw)
    nef2.grid.init_from_scales(); nef2.delta_grid.init_from_scales()
    nef2.load_state_dict(nef.state_dict())
    assert torch.equal(nef2.grid.blas.octree.cpu(), oc) and nef2.grid.blas.max_level == 3


def test_decoder_kernel_family_selection():
    """Which decoder kernels a call gets (host logic only): tensor cores under autocast; exact FP32 otherwise -- the register-tiled
    forward kernels only when nothing is differentiated, the one-sample-per-thread kernels (they have a backward) under grad."""
    import bench
    from pagnerf_b200 import ops
    from pagnerf_b200.pc_nerf import PanopticDeltaNeF
    assert ops.dc_mode(True, 48) is True
    assert ops.dc_mode(False, 48) is False
    with torch.no_grad():
        assert ops.dc_mode(False, 48) == 'tiled' and ops.dc_mode(False, 30) is False and ops.dc_mode(True, 48) is True
    nef = PanopticDeltaNeF(**dict(bench.NEF_KW, blas_level=3, capacity_log_2=8, delta_capacity_log_2=7))
    chans = {'rgb', 'semantics', 'inst_embedding'}
    nef.decoder_precision = 'fp32'
    assert not nef.fused_panoptic_ok(chans)
    with torch.no_grad():
        assert nef.fused_panoptic_ok(chans) and not nef.fused_panoptic_ok({'rgb'})
        tiled0, ops.TILED_F32 = ops.TILED_F32, False
        try:
            assert not nef.fused_panoptic_ok(chans)
        finally:
            ops.TILED_F32 = tiled0
    nef.decoder_precision = 'fp16'
    assert nef.fused_panoptic_ok(chans)
    nef.decoder_precision = 'auto'
    assert not nef._use_tc()
    assert nef.grid.interpolate_needs_pidx is False          # the tracer may march without octree point indices


def test_view_embedding_double_angle_recurrence_error_bound():
    """csrc/decoder_tiled.cu builds the octaves sin / cos(2^f v), f = 1..3, from one sincos per component by angle doubling in
    fp32; the comment there promises <= 1e-6 absolute against the directly evaluated embedding for |v| <= 1 (unit directions)."""
    import numpy as np
    v = np.linspace(-1.0, 1.0, 200001).astype(np.float32)
    sn, cs = np.sin(v.astype(np.float64)).astype(np.float32), np.cos(v.astype(np.float64)).astype(np.float32)
    worst = 0.0
    for f in range(4):
        a = v.astype(np.float64) * (1 << f)
        worst = max(worst, float(np.abs(sn - np.sin(a)).max()), float(np.abs(cs - np.cos(a)).max()))
        s2 = (np.float32(2.0) * sn) * cs
        c2 = (np.float32(-2.0) * sn).astype(np.float64) * sn.astype(np.float64) + 1.0      # fmaf(-2 sn, sn, 1): one rounding
        sn, cs = s2.astype(np.float32), c2.astype(np.float32)
    assert worst <= 1e-6, worst


def test_dd_plugin_surface():
    """PanopticDDensityNeF / PanopticDDensityPackedRFTracer (SURVEY 8f rank 2): reference names, channels and state_dict keys
    (pc_nerf/panoptic_dd_nef.py:41-58,121-128; tracers/panoptic_dd_packed_rf_tracer.py)."""
    import bench
    from pagnerf_b200.pc_nerf import PanopticDDensityNeF
    from pagnerf_b200.tracers import PanopticDDensityPackedRFTracer, PanopticPackedRFTracer
    kw = dict(bench.NEF_KW, blas_level=3, capacity_log_2=8, delta_capacity_log_2=7)
    nef = PanopticDDensityNeF(**kw)
    nef.grid.init_from_scales(); nef.delta_grid.init_from_scales()
    assert nef.delta_grid.capacity == 128
    keys = set(nef.state_dict().keys())
    for k in ("decoder_delta_density.layers.0.weight", "decoder_delta_density.layers.0.bias",
              "decoder_delta_density.lout.weight", "decoder_delta_density.lout.bias", "delta_grid.embedder.lattice_values"):
        assert k in keys
    assert nef.decoder_delta_density.lout.weight.shape == (1, 64) and nef.decoder_delta_density.layers[0].weight.shape == (64, 48)
    assert nef.get_supported_channels() == {"density", "rgb", "delta_density", "panoptic_density", "semantics", "inst_embedding"}
    assert nef.get_nef_type() == 'delta_panoptic_nef'
    tr = PanopticDDensityPackedRFTracer(raymarch_type='ray', num_steps=512, ray_max_travel=2.0)
    assert isinstance(tr, PanopticPackedRFTracer) and tr.panoptic_channels == {'semantics', 'inst_embedding'}
    # the collapsed delta-density head (two Linear layers, activation 'none') is the same linear map
    table, dtable, wts = nef.fused_trace_tensors()
    assert len(wts) == 22 and wts[20].shape == (1, 48) and wts[21].shape == (1,)
    x = torch.randn(5, 48)
    ref = nef.decoder_delta_density(x)
    assert torch.allclose(x @ wts[20].T + wts[21], ref, atol=1e-5)


def test_unsupported_configs_fail_loudly():
    import bench
    from pagnerf_b200.pc_nerf import PanopticNeF
    from pagnerf_b200.pc_nerf.panoptic_nef import _decoder_tensors
    nef = PanopticNeF(**dict(bench.NEF_KW, blas_level=2, capacity_log_2=6, hidden_dim=128, panoptic_features_type=None,
                             sem_hidden_dim=128, inst_hidden_dim=128))
    with pytest.raises(NotImplementedError):
        _decoder_tensors(nef.decoder_density, 1)
    with pytest.raises(NotImplementedError):
        PanopticNeF(**dict(bench.NEF_KW, grid_type="OctreeGrid"))


def test_wisp_compat_dispatch_and_renderbuffer():
    from pagnerf_b200.wisp_compat import RenderBuffer, Rays
    a = RenderBuffer(rgb=torch.zeros(3, 3), alpha=torch.zeros(3, 1), depth=None, semantics=torch.zeros(3, 6))
    b = RenderBuffer(rgb=torch.ones(2, 3), alpha=torch.ones(2, 1), semantics=torch.ones(2, 6))
    c = a + b
    assert c.rgb.shape == (5, 3) and c.semantics.shape == (5, 6) and c.depth is None
    assert c.reshape(5, -1).rgb.shape == (5, 3)
    r = Rays(origins=torch.zeros(10, 3), dirs=torch.ones(10, 3), dist_min=0.0, dist_max=2.0)
    assert len(r) == 10 and [len(x) for x in r.split(4)] == [4, 4, 2] and r.reshape(2, 5, 3).origins.shape == (2, 5, 3)


def test_header_cites_reference_for_each_section():
    src = open(os.path.join(ROOT, "include", "pagnerf_b200.h")).read()
    for cite in ("grids/occtree.py:85-91", "grids/permuto_grid.py:57-62,71", "grids/hash_grid_tinycudann.py:24-34,41",
                 "grids/hash_grid_torch.py:13-108", "pc_nerf/panoptic_nef.py:114-164", "tracers/panoptic_packed_rf_tracer.py:134-205"):
        assert cite in src, cite


_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from pagnerf_b200 import parallel
dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{sys.argv[2]}", rank=int(sys.argv[3]), world_size=2)
rank = dist.get_rank()
torch.manual_seed(0)
big = torch.nn.Parameter(torch.zeros(1 << 20, 2)); small = [torch.nn.Parameter(torch.zeros(5, 3)), torch.nn.Parameter(torch.zeros(7))]
params = [big] + small + [torch.nn.Parameter(torch.zeros(2))]      # last one has no grad
g = torch.Generator().manual_seed(100 + rank)
big.grad = torch.rand(big.shape, generator=g); small[0].grad = torch.rand(5, 3, generator=g); small[1].grad = torch.rand(7, generator=g)
local = [p.grad.clone() for p in params[:3]]
n = parallel.allreduce_grads(params, average=False)
assert n == 2, n
other = []
g2 = torch.Generator().manual_seed(100 + (1 - rank))
other = [torch.rand(big.shape, generator=g2), torch.rand(5, 3, generator=g2), torch.rand(7, generator=g2)]
for p, a, b in zip(params[:3], local, other):
    assert torch.allclose(p.grad, a + b), "allreduce mismatch"
assert parallel.shard_images(7, rank, 2) == list(range(rank, 7, 2))
dist.destroy_process_group()
print("OK", rank)
'''


def test_grad_allreduce_world_size_2_gloo(tmp_path):
    """Ray-sharded DP exchange step (grid tables + flattened decoder bucket) on 2 CPU processes over gloo."""
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, str(port), str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=180)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0 and f"OK {r}" in o, o


def test_lattice_hash_linear_form_is_the_loop_form():
    """csrc/permuto.cu evaluates the lattice-vertex hash as base + r*(m+m^2+m^3) - 4*sum [rank_i > 3-r] m^(3-i) (three multiplies
    per level); the oracle / the published algorithm iterate k = (k + key_i) * m per vertex.  Same uint32 wrap-around result."""
    import numpy as np
    M1 = 2531011
    M2 = (M1 * M1) & 0xFFFFFFFF
    M3 = (M2 * M1) & 0xFFFFFFFF
    MS = (M1 + M2 + M3) & 0xFFFFFFFF
    rng = np.random.default_rng(0)
    for _ in range(5000):
        rem = [int(x) for x in rng.integers(-50000, 50000, 3)]
        rank = [int(x) for x in rng.integers(0, 4, 3)]
        base = ((rem[0] & 0xFFFFFFFF) * M3 + (rem[1] & 0xFFFFFFFF) * M2 + (rem[2] & 0xFFFFFFFF) * M1) & 0xFFFFFFFF
        for r in range(4):
            k = 0
            for i in range(3):
                key = rem[i] + r - (4 if rank[i] > 3 - r else 0)
                k = ((k + key) * M1) & 0xFFFFFFFF
            lin = (base + r * MS) & 0xFFFFFFFF
            for i, P in enumerate((M3, M2, M1)):
                if rank[i] > 3 - r:
                    lin = (lin - 4 * P) & 0xFFFFFFFF
            assert k == lin


def test_pose_oracle_properties():
    """oracle/pose.py (the checker of csrc/pose.cu): Gram-Schmidt rows are a proper rotation, view matrices round-trip through
    the 9-parameter layout, and inv_transform_rays inverts the view transform; autograd matches finite differences."""
    import torch
    from oracle import pose
    gen = torch.Generator().manual_seed(0)
    p = torch.randn(5, 9, generator=gen, dtype=torch.float64)
    R = pose.rot6d_to_matrix(p[:, :6])
    assert torch.allclose(R @ R.transpose(1, 2), torch.eye(3, dtype=torch.float64).expand(5, 3, 3), atol=1e-12)
    assert torch.allclose(torch.linalg.det(R), torch.ones(5, dtype=torch.float64), atol=1e-12)
    V = torch.eye(4, dtype=torch.float64).repeat(5, 1, 1)
    V[:, :3, :3], V[:, :3, 3] = R, p[:, 6:]
    assert torch.allclose(pose.params_from_view_matrix(V)[:, :6], torch.cat([R[:, 0], R[:, 1]], 1))
    xw = torch.randn(5 * 3, 3, generator=gen, dtype=torch.float64)                       # world points
    xc = (torch.einsum('cij,cbj->cbi', R, xw.reshape(5, 3, 3)) + p[:, None, 6:]).reshape(-1, 3)   # view transform
    back, _ = pose.transform_rays(pose.params_from_view_matrix(V), torch.arange(5), xc, xc)
    assert torch.allclose(back, xw, atol=1e-10)
    q = p.clone().requires_grad_(True)
    bo, bd = torch.randn(10, 3, generator=gen, dtype=torch.float64), torch.randn(10, 3, generator=gen, dtype=torch.float64)
    assert torch.autograd.gradcheck(lambda z: pose.transform_rays(z, torch.tensor([1, 4]), bo, bd), (q,), atol=1e-6)


def test_loss_oracle_basics():
    """oracle/losses.py (the checker of csrc/loss.cu): consistent predictions give zero loss, one wrong pixel trains the whole image,
    labels beyond the id table fall back to id 1 (loss/lin_assignment_things.py:31,48-55,84)."""
    import torch
    from oracle.losses import lin_assignment_things_loss, virtual_labels
    R, C = 64, 6
    gt = torch.zeros(1, R, dtype=torch.int64)
    gt[0, :20], gt[0, 20:40] = 4, 11
    p = torch.full((1, R, C), 0.02)
    p[0, :20, 3], p[0, 20:40, 1], p[0, 40:, 0] = 0.9, 0.9, 0.9
    p = p / p.sum(-1, keepdim=True)
    loss, virt = lin_assignment_things_loss(p, gt, gt == 0)
    assert float(loss.abs().max()) == 0.0 and virt[0, 0] == 3 and virt[0, 25] == 1 and virt[0, 50] == 0
    p[0, 0, 3], p[0, 0, 5] = 0.02, 0.9
    loss, _ = lin_assignment_things_loss(p / p.sum(-1, keepdim=True), gt, gt == 0)
    assert float(loss.min()) > 0.0
    many = torch.arange(1, 9)                      # 8 labels, 5 ids: the 3 largest labels are not assigned
    v = virtual_labels(torch.softmax(torch.randn(8, C), -1), many)
    assert (v[5:] == 1).all() and sorted(v[:5].tolist()) == [1, 2, 3, 4, 5]


def test_ba_pipeline_surface_and_pose_layout():
    """BAPipeline (pc_nerf/ba_pipeline.py:10-92): constructor forms, the 9-parameter `camera_extrinsics` layout (first two rows of
    the view rotation + translation), cam-id mapping, anchor mask registration; the transform itself refuses CPU tensors."""
    import torch
    from oracle import pose as opose
    from pagnerf_b200.pc_nerf import BAPipeline
    V = torch.eye(4).repeat(3, 1, 1)
    V[:, :3, 3] = torch.tensor([[0.1, 0.2, 0.3], [0.0, 0.0, 1.0], [-1.0, 0.5, 0.0]])
    pipe = BAPipeline(None, V, None, anchor_frame_idxs=[0])
    assert tuple(pipe.camera_extrinsics.shape) == (3, 9)
    assert torch.equal(pipe.camera_extrinsics.detach(), opose.params_from_view_matrix(V))
    assert 'camera_extrinsics' in dict(pipe.named_parameters())
    assert pipe.cameras.extrinsics.parameters() is pipe.camera_extrinsics and len(pipe.cameras) == 3

    class Cam:      # kaolin-like duck type
        def __init__(self, v): self.extrinsics, self.near, self.far = self, 0.0, 2.0; self._v = v
        def view_matrix(self): return self._v[None]
    pipe2 = BAPipeline(None, {"a": Cam(V[0]), "b": Cam(V[1])}, None)
    assert pipe2.cam_id_to_idx == {"a": 0, "b": 1} and pipe2.cameras.far == 2.0
    assert pipe2.get_camera_indices(["b", "a"]).tolist() == [1, 0]
    from pagnerf_b200.wisp_compat import Rays
    with pytest.raises(RuntimeError):
        pipe.transform_rays(Rays(origins=torch.zeros(6, 3), dirs=torch.ones(6, 3)), torch.tensor([0, 1, 2]))


def test_fused_adam_refuses_cpu_and_amsgrad():
    import torch
    from pagnerf_b200.optim import FusedAdam
    p = torch.nn.Parameter(torch.zeros(4))
    with pytest.raises(NotImplementedError):
        FusedAdam([p], amsgrad=True)
    opt = FusedAdam([dict(params=[p], lr=0.1)], eps=1e-15)
    assert opt.param_groups[0]['lr'] == 0.1 and opt.param_groups[0]['betas'] == (0.9, 0.999)
    p.grad = torch.ones(4)
    with pytest.raises(RuntimeError):
        opt.step()


def test_bench_dump_outputs_format(tmp_path):
    """bench.py --dump-outputs writer: float32 (float64 kept), small arrays whole, large ones as the same seeded sample every time."""
    import bench
    big = torch.arange(3 * bench.DUMP_MAX_ELEMENTS, dtype=torch.float64).reshape(3, -1)
    arrays = {"loss": torch.tensor(2.5), "hit": torch.tensor([True, False]), "grad.a": torch.ones(4, 5, dtype=torch.float16), "big": big}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    a = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in arrays}
    assert a["loss"].dtype == np.float32 and a["loss"] == 2.5
    assert a["hit"].tolist() == [1.0, 0.0] and a["grad.a"].dtype == np.float32 and a["grad.a"].shape == (4, 5)
    assert a["big"].dtype == np.float64 and a["big"].shape == (bench.DUMP_MAX_ELEMENTS,)
    assert np.all(np.diff(a["big"]) > 0), "distinct elements in index order"
    assert np.array_equal(a["big"], np.load(tmp_path / "b" / "big.npy")), "same sample positions in every run"
    with pytest.raises(RuntimeError, match="limit"):
        bench.dump_outputs(str(tmp_path / "c"), {f"x{i}": torch.zeros(bench.DUMP_MAX_ELEMENTS) for i in range(17)})
    assert not (tmp_path / "c").exists()


def test_bench_configs_build_and_reference_arm_line():
    """bench.py plumbing on the CPU: every BASELINE config's field constructs with the documented shapes, the confined rays of the
    dense configs stay inside the cube, and `--impl reference` prints one JSON line with the same `config` object our arm prints."""
    import json
    import numpy as np
    import torch
    import bench
    shapes = {1: ("HashGridTorch", 16, True), 2: ("PermutoGrid", 24, True), 3: ("HashGridTinyCudaNN", 14, False)}
    for cid, (gtype, levels, delta) in shapes.items():
        wl = bench.Workload(torch.device('cpu'), n_rays=64, n_batches=1, config=cid)
        assert type(wl.nef.grid).__name__ == gtype and wl.nef.grid.num_lods == levels and hasattr(wl.nef, 'delta_grid') == delta
    o, d = bench.make_rays(4096, 0, 0, confined=True)
    pts = o[:, None, :] + d[:, None, :] * np.linspace(0, 1.7, 33)[None, :, None]
    assert np.abs(pts).max() < 1.0, "dense N x S packing: every sample inside the unit cube"
    V = bench.make_cameras(0)
    assert V.shape == (42, 4, 4) and np.allclose(V[:, :3, :3] @ np.transpose(V[:, :3, :3], (0, 2, 1)), np.eye(3), atol=1e-6)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--cpu-sample-rays", "64"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["steps"] == 1 and line["unit"] == "rays/s" and line["cpu_baseline"]["kind"] == "port"
    assert line["config"]["baseline_config"] == 2 and line["config"]["rays_per_gpu"] == 16384
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["value"] > 0
