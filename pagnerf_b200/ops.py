"""Torch-facing wrappers (allocation + autograd) over the C ABI in include/pagnerf_b200.h.

PyTorch is plumbing here: it owns device memory, streams and the autograd graph; every arithmetic
step of the hot path is one of our sm_100a kernels.  All functions require CUDA tensors and raise
otherwise -- there is deliberately no CPU or library fallback.
"""
import os

import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import _lib
from ._lib import call, ptr, ptr_array, query_i64


def _chk(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("pagnerf_b200 ops run on CUDA tensors only (no CPU fallback)")


def _f32(t):
    if t is None:
        return None
    return t.detach().to(torch.float32).contiguous()


# ------------------------------------------------------------------------------------------------
# octree / marching
# ------------------------------------------------------------------------------------------------
_LINSPACE = {}


def _linspace(S, device):
    key = (S, str(device))
    if key not in _LINSPACE:
        _LINSPACE[key] = torch.linspace(0.0, 1.0, S, dtype=torch.float32).to(device)  # CPU arithmetic == oracle
    return _LINSPACE[key]


def octree_query(octree, prefix, coords, level):
    """kaolin.ops.spc.unbatched_query -> int32 [P] (-1 = empty)."""
    _chk(octree, prefix, coords)
    c = _f32(coords).reshape(-1, 3)
    out = torch.empty(c.shape[0], dtype=torch.int32, device=c.device)
    call("pag_octree_query", ptr(octree), ptr(prefix), ptr(c), c.shape[0], int(level), ptr(out))
    return out


def raymarch_ray(octree, prefix, origins, dirs, level, num_samples, dist_min, dist_max, jitter=None, seed=0):
    """'ray' mode.  Returns ridx i64[M], pidx i64[M], samples f32[M,1,3], depths f32[M,1], deltas f32[M,1],
    boundary bool[M], offsets i64[N+1] (per-ray packed start; offsets[N] = M)."""
    _chk(octree, prefix, origins, dirs)
    o, d = _f32(origins), _f32(dirs)
    N, S, dev = o.shape[0], int(num_samples), o.device
    lin = _linspace(S, dev)
    pidx_tmp = torch.empty(max(N * S, 1), dtype=torch.int32, device=dev)
    counts = torch.empty(max(N, 1), dtype=torch.int32, device=dev)
    offsets = torch.empty(N + 1, dtype=torch.int64, device=dev)
    jit = _f32(jitter) if jitter is not None else None
    near, rng = float(dist_min), float(torch.tensor(float(dist_max) - float(dist_min), dtype=torch.float32))
    call("pag_march_ray_count", ptr(o), ptr(d), N, S, ptr(lin), ptr(jit), int(seed), near, rng,
         ptr(octree), ptr(prefix), int(level), ptr(pidx_tmp), ptr(counts), ptr(offsets), None)
    M = int(offsets[-1].item())  # the one host sync the tensor-shaped plugin API needs
    ridx = torch.empty(M, dtype=torch.int64, device=dev)
    pidx = torch.empty(M, dtype=torch.int64, device=dev)
    samples = torch.empty(M, 1, 3, dtype=torch.float32, device=dev)
    depths = torch.empty(M, 1, dtype=torch.float32, device=dev)
    deltas = torch.empty(M, 1, dtype=torch.float32, device=dev)
    boundary = torch.empty(M, dtype=torch.bool, device=dev)
    if M:
        call("pag_march_ray_emit", ptr(o), ptr(d), N, S, ptr(lin), ptr(jit), int(seed), near, rng,
             ptr(pidx_tmp), ptr(offsets), ptr(ridx), ptr(pidx), ptr(samples), ptr(depths), ptr(deltas), ptr(boundary), None)
    return ridx, pidx, samples, depths, deltas, boundary, offsets


def raymarch_ray_bits(bits, origins, dirs, level, num_samples, dist_min, dist_max, seed=0):
    """'ray' mode against the occupancy bit field of `level` (OctreeAS.level_bits): one cached word per step instead of an octree
    descent, no point indices.  Same samples, bit for bit, as raymarch_ray.  Returns ridx i64[M], None, samples f32[M,1,3],
    depths f32[M,1], deltas f32[M,1], boundary bool[M], offsets i64[N+1]."""
    _chk(bits, origins, dirs)
    o, d = _f32(origins), _f32(dirs)
    N, S, dev = o.shape[0], int(num_samples), o.device
    lin = _linspace(S, dev)
    masks = torch.empty(max(N, 1) * ((S + 31) // 32), dtype=torch.int32, device=dev)
    counts = torch.empty(max(N, 1), dtype=torch.int32, device=dev)
    offsets = torch.empty(N + 1, dtype=torch.int64, device=dev)
    near, rng = float(dist_min), float(torch.tensor(float(dist_max) - float(dist_min), dtype=torch.float32))
    call("pag_march_ray_bits_count", ptr(o), ptr(d), N, S, ptr(lin), None, int(seed), near, rng, ptr(bits), int(level),
         ptr(masks), ptr(counts), ptr(offsets), None)
    M = int(offsets[-1].item())  # the one host sync the tensor-shaped plugin API needs
    ridx = torch.empty(M, dtype=torch.int64, device=dev)
    samples = torch.empty(M, 1, 3, dtype=torch.float32, device=dev)
    depths = torch.empty(M, 1, dtype=torch.float32, device=dev)
    deltas = torch.empty(M, 1, dtype=torch.float32, device=dev)
    if M:
        call("pag_march_ray_bits_emit", ptr(o), ptr(d), N, S, ptr(lin), None, int(seed), near, rng, ptr(masks), ptr(offsets),
             ptr(ridx), ptr(samples), ptr(depths), ptr(deltas), None)
    # pack boundaries without a second host sync: rays with samples mark their first packed row (empty rays add 0 at the next ray's row)
    first = torch.zeros(M + 1, dtype=torch.int32, device=dev)
    first.scatter_add_(0, offsets[:-1], (counts[:N] > 0).to(torch.int32))
    boundary = first[:M] > 0
    return ridx, None, samples, depths, deltas, boundary, offsets


def raytrace(octree, prefix, origins, dirs, level):
    """kaolin unbatched_raytrace(return_depth=True, with_exit=True) -> ridx i64[K], pidx i64[K], depth f32[K,2], offsets."""
    _chk(octree, prefix, origins, dirs)
    o, d = _f32(origins), _f32(dirs)
    N, dev = o.shape[0], o.device
    counts = torch.empty(max(N, 1), dtype=torch.int32, device=dev)
    offsets = torch.empty(N + 1, dtype=torch.int64, device=dev)
    call("pag_raytrace_count", ptr(octree), ptr(prefix), ptr(o), ptr(d), N, int(level), ptr(counts), ptr(offsets))
    K = int(offsets[-1].item())
    ridx = torch.empty(K, dtype=torch.int64, device=dev)
    pidx = torch.empty(K, dtype=torch.int64, device=dev)
    depth = torch.empty(K, 2, dtype=torch.float32, device=dev)
    if K:
        call("pag_raytrace_emit", ptr(octree), ptr(prefix), ptr(o), ptr(d), N, int(level), ptr(offsets),
             ptr(ridx), ptr(pidx), ptr(depth))
    return ridx, pidx, depth, offsets


def raymarch_voxel(octree, prefix, origins, dirs, level, num_samples, jitter=None, seed=0):
    """'voxel' mode.  Returns ridx i64[K], pidx i64[K], samples f32[K,S,3], depths f32[K,S,1], deltas f32[K*S,1],
    boundary bool[K*S], offsets i64[N+1] (per-ray first nugget)."""
    ridx, pidx, depth, offsets = raytrace(octree, prefix, origins, dirs, level)
    o, d = _f32(origins), _f32(dirs)
    K, S, dev = ridx.shape[0], int(num_samples), o.device
    samples = torch.empty(K, S, 3, dtype=torch.float32, device=dev)
    depths = torch.empty(K, S, 1, dtype=torch.float32, device=dev)
    deltas = torch.empty(K * S, 1, dtype=torch.float32, device=dev)
    boundary = torch.empty(K * S, dtype=torch.bool, device=dev)
    jit = _f32(jitter) if jitter is not None else None
    if K:
        call("pag_voxel_samples", ptr(o), ptr(d), ptr(ridx), ptr(depth), K, S, ptr(jit), int(seed),
             ptr(samples), ptr(depths), ptr(deltas), ptr(boundary))
    return ridx, pidx, samples, depths, deltas, boundary, offsets


def max_travel_mask(ridx, depths, ray_first, max_travel):
    """tracers/panoptic_packed_rf_tracer.py:88-99 -> bool[K] keep mask over nuggets."""
    K = ridx.shape[0]
    S = depths.shape[1] if depths.dim() > 1 else 1
    keep = torch.empty(K, dtype=torch.bool, device=ridx.device)
    if K:
        call("pag_max_travel_mask", ptr(ridx), ptr(depths.contiguous()), K, S, ptr(ray_first), float(max_travel), ptr(keep))
    return keep


def mark_pack_boundaries(ids):
    _chk(ids)
    ids64 = ids.to(torch.int64).contiguous()
    out = torch.empty(ids64.shape[0], dtype=torch.bool, device=ids.device)
    call("pag_mark_pack_boundaries", ptr(ids64), ids64.shape[0], ptr(out))
    return out


def ray_offsets(ridx, num_rays):
    """offsets i64[R+1] from an ascending ridx (lower_bound per ray)."""
    _chk(ridx)
    r64 = ridx.to(torch.int64).contiguous()
    off = torch.empty(num_rays + 1, dtype=torch.int64, device=ridx.device)
    call("pag_ray_offsets", ptr(r64), r64.shape[0], int(num_rays), ptr(off))
    return off


class RaySamplesFn(Function):
    """Re-attaches the marcher's sample positions to the ray tensors for autograd:
    samples = o[ridx] + d[ridx] * t   (values come from the marcher kernel, bit-exact)."""

    @staticmethod
    def forward(ctx, origins, dirs, samples, depths, offsets):
        ctx.save_for_backward(depths, offsets)
        ctx.n = origins.shape[0]
        return samples.clone()

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        depths, offsets = ctx.saved_tensors
        # packs here are rays over *nuggets x samples*: offsets index rows of g.view(-1, 3)
        g2 = _f32(g).reshape(-1, 3)
        t = depths.reshape(-1, 1)
        go = torch.empty(ctx.n, 3, dtype=torch.float32, device=g.device)
        gd = torch.empty(ctx.n, 3, dtype=torch.float32, device=g.device)
        gt = (g2 * t).contiguous()
        call("pag_sum_reduce_fwd", ptr(g2), 3, ptr(offsets), ctx.n, ptr(go))
        call("pag_sum_reduce_fwd", ptr(gt), 3, ptr(offsets), ctx.n, ptr(gd))
        return go, gd, None, None, None


class PoseTransformFn(Function):
    """BAPipeline.transform_rays (pc_nerf/ba_pipeline.py:85-92): camera-space base rays -> world-space rays through the 9
    pose parameters per camera (6-D rotation + translation), directions renormalised; backward reduces d/d(o, d) to the
    parameter rows, one CTA per camera (csrc/pose.cu)."""

    @staticmethod
    def forward(ctx, params, cam_idx, base_o, base_d):
        _chk(params, cam_idx, base_o, base_d)
        p = _f32(params)
        ci = cam_idx.to(torch.int64).contiguous()
        bo, bd = _f32(base_o).reshape(-1, 3), _f32(base_d).reshape(-1, 3)
        C = ci.shape[0]
        if C == 0 or bo.shape[0] % C:
            raise ValueError("base rays must be grouped by camera with the same number of rays per camera")
        B = bo.shape[0] // C
        o, d = torch.empty_like(bo), torch.empty_like(bd)
        call("pag_pose_transform_fwd", ptr(p), ptr(ci), ptr(bo), ptr(bd), C, B, ptr(o), ptr(d))
        ctx.save_for_backward(p, ci, bo, bd)
        ctx.shape = params.shape
        return o, d

    @staticmethod
    @once_differentiable
    def backward(ctx, g_o, g_d):
        p, ci, bo, bd = ctx.saved_tensors
        C = ci.shape[0]
        gp = torch.zeros_like(p)
        go = _f32(g_o) if g_o is not None else None
        gd = _f32(g_d) if g_d is not None else None
        if go is not None or gd is not None:
            call("pag_pose_transform_bwd", ptr(p), ptr(ci), ptr(bo), ptr(bd), ptr(go), ptr(gd), C, bo.shape[0] // C, ptr(gp))
        return gp.reshape(ctx.shape), None, None, None


def pose_transform(params, cam_idx, base_o, base_d):
    return PoseTransformFn.apply(params, cam_idx, base_o, base_d)


# ------------------------------------------------------------------------------------------------
# encoders
# ------------------------------------------------------------------------------------------------
class PermutoEncodeFn(Function):
    @staticmethod
    def forward(ctx, pos, table, scale_factor, shift, anneal, n_agg_levels):
        _chk(pos, table, scale_factor, shift, anneal)
        p = _f32(pos).reshape(-1, 3)
        L, cap, F = table.shape
        out = torch.empty(p.shape[0], L * F, dtype=torch.float32, device=p.device)
        tb = table.detach().contiguous()
        call("pag_permuto_fwd", ptr(p), p.shape[0], ptr(tb), cap, L, F, ptr(scale_factor), ptr(shift), ptr(anneal), ptr(out))
        ctx.save_for_backward(p, tb, scale_factor, shift, anneal)
        ctx.n_agg = int(n_agg_levels)
        ctx.pos_shape = pos.shape
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        p, tb, sf, sh, an = ctx.saved_tensors
        L, cap, F = tb.shape
        g = _f32(g)
        need_pos, need_tab = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        gpos = torch.empty_like(p) if need_pos else None
        gtab = torch.zeros_like(tb)
        call("pag_permuto_bwd", ptr(p), p.shape[0], ptr(tb), cap, L, F, ptr(sf), ptr(sh), ptr(an), ptr(g),
             ptr(gtab), ptr(gpos), ctx.n_agg)
        return (gpos.reshape(ctx.pos_shape) if need_pos else None), (gtab if need_tab else None), None, None, None, None


def permuto_encode(pos, table, scale_factor, shift, anneal, n_agg_levels=0):
    return PermutoEncodeFn.apply(pos, table, scale_factor, shift, anneal, n_agg_levels)


def permuto_indices(pos, capacity, scale_factor, shift):
    p = _f32(pos).reshape(-1, 3)
    L, M = scale_factor.shape[0], p.shape[0]
    idx = torch.empty(L, M, 4, dtype=torch.int32, device=p.device)
    rank = torch.empty(L, M, 4, dtype=torch.int32, device=p.device)
    bary = torch.empty(L, M, 4, dtype=torch.float32, device=p.device)
    call("pag_permuto_indices", ptr(p), M, int(capacity), L, ptr(scale_factor), ptr(shift), ptr(idx), ptr(rank), ptr(bary))
    return idx, rank, bary


class HashEncodeFn(Function):
    @staticmethod
    def forward(ctx, pos, table, flavour, fparam, res, offset, size, round_half, n_agg_levels):
        _chk(pos, table, fparam, offset, size)
        p = _f32(pos).reshape(-1, 3)
        L = fparam.shape[0]
        tb = table.detach().contiguous().view(-1, 2)
        out = torch.empty(p.shape[0], L * 2, dtype=torch.float32, device=p.device)
        call("pag_hash_fwd", int(flavour), ptr(p), p.shape[0], ptr(tb), L, 2, ptr(fparam), ptr(res), ptr(offset),
             ptr(size), ptr(out), int(round_half))
        ctx.save_for_backward(p, tb, fparam, res, offset, size)
        ctx.flavour, ctx.n_agg, ctx.pos_shape, ctx.tab_shape = int(flavour), int(n_agg_levels), pos.shape, table.shape
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        p, tb, fparam, res, offset, size = ctx.saved_tensors
        L = fparam.shape[0]
        g = _f32(g)
        need_pos, need_tab = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        gpos = torch.empty_like(p) if need_pos else None
        gtab = torch.zeros_like(tb)
        call("pag_hash_bwd", ctx.flavour, ptr(p), p.shape[0], ptr(tb), L, 2, ptr(fparam), ptr(res), ptr(offset), ptr(size),
             ptr(g), ptr(gtab), ptr(gpos), ctx.n_agg)
        return ((gpos.reshape(ctx.pos_shape) if need_pos else None), (gtab.view(ctx.tab_shape) if need_tab else None),
                None, None, None, None, None, None, None)


def hash_encode(pos, table, flavour, fparam, res, offset, size, round_half=False, n_agg_levels=0):
    return HashEncodeFn.apply(pos, table, flavour, fparam, res, offset, size, round_half, n_agg_levels)


def hash_indices(pos, flavour, fparam, res, offset, size):
    p = _f32(pos).reshape(-1, 3)
    L, M = fparam.shape[0], p.shape[0]
    idx = torch.empty(L, M, 8, dtype=torch.int32, device=p.device)
    call("pag_hash_indices", int(flavour), ptr(p), M, L, ptr(fparam), ptr(res), ptr(offset), ptr(size), ptr(idx))
    return idx


# ------------------------------------------------------------------------------------------------
# decoders
# ------------------------------------------------------------------------------------------------
HIDDEN = 64
VIEW_DIM = 27
# Rendering under torch.no_grad(): samples whose integration weight is exactly 0 (transmittance underflowed behind an opaque
# surface, or sigma == 0) add exactly nothing to any map, so the colour decoder, the delta-grid lookup and the panoptic heads
# run on the other samples only when those are fewer than this share of the packed samples (0 disables, > 1 forces).
LIVE_COMPACT_FRAC = float(os.environ.get('PAGNERF_LIVE_COMPACT_FRAC', '0.7'))
# A sample counts as live when its weight exceeds this.  0 keeps every non-zero weight (bit-exact skipping).  The default 2^-30
# also drops the samples behind an opaque surface whose weight is positive but below the fp32 resolution of the composited sums
# (the weights of a ray sum to <= 1; <= 128 dropped terms of <= 2^-30 each move a map by <= 1.2e-7, the size of the fp32 rounding of
# the sum itself and 1000x below the 1e-4 parity tolerance; renderers usually stop rays at a transmittance of 1e-4).
LIVE_WEIGHT_EPS = float(os.environ.get('PAGNERF_LIVE_WEIGHT_EPS', str(2.0 ** -30)))
TILED_F32 = os.environ.get('PAGNERF_TILED_F32', '1') == '1'     # 0: the one-sample-per-thread FP32 forward also for inference
GRAD_TARGET = 1024.0   # upstream gradients are rescaled so that their max magnitude sits near 2^10 in fp16


def grad_scale(*grads):
    """Power-of-two loss scale for the fp16 tensor-core backward (device scalar, no host sync):
    2^floor(log2(GRAD_TARGET / max|g|)).  Plays the role of torch.cuda.amp.GradScaler inside the op."""
    gs = [g for g in grads if g is not None]
    assert 1 <= len(gs) <= 2
    return grad_scale_dyn(gs[0], gs[1] if len(gs) > 1 else None, None)


_SCALE_SCRATCH = {}


def grad_scale_dyn(a, b, m_dev, wa=1, wb=1):
    """One-launch device-side loss scale; with m_dev only the first m_dev[0]*w elements of a / b are scanned."""
    dev = a.device
    # two zeroed words per (device, stream): the kernel's last block resets them, so they are zeroed exactly once
    key = (str(dev), torch.cuda.current_stream().cuda_stream)
    scratch = _SCALE_SCRATCH.get(key)
    if scratch is None:
        scratch = _SCALE_SCRATCH[key] = torch.zeros(2, dtype=torch.int32, device=dev)
    out = torch.empty(1, dtype=torch.float32, device=dev)
    call("pag_grad_scale", ptr(a), a.numel(), int(wa), ptr(b), b.numel() if b is not None else 0, int(wb), ptr(m_dev),
         GRAD_TARGET, ptr(scratch), ptr(out))
    return out


def dc_mode(use_tc, IN):
    """Kernel family for DecodeDCFn: tensor cores / register-tiled FP32 (inference, torch.no_grad()) / per-thread FP32."""
    if use_tc:
        return True
    return 'tiled' if (TILED_F32 and IN % 4 == 0 and not torch.is_grad_enabled()) else False


class DecodeDCFn(Function):
    """density + color decoders.  feats [M,IN], ray_d [M//S, 3] -> sigma [M], rgb [M,3] (or None).
    use_tc: True (tensor cores), False (exact FP32, differentiable) or 'tiled' (exact FP32, forward only: the caller promises
    that nothing is differentiated -- see dc_mode())."""

    @staticmethod
    def forward(ctx, feats, lodw, ray_d, S, want_rgb, use_tc, *weights):
        _chk(feats, ray_d, *weights)
        f = _f32(feats)
        M, IN = f.shape
        rd = _f32(ray_d)
        w = [_f32(x) for x in weights]
        sigma = torch.empty(M, dtype=torch.float32, device=f.device)
        rgb = torch.empty(M, 3, dtype=torch.float32, device=f.device) if want_rgb else None
        lw = _f32(lodw)
        # exact-FP32 inference (nothing to differentiate): the register-tiled forward (csrc/decoder_tiled.cu)
        tiled = use_tc == 'tiled'
        use_tc = use_tc is True
        entry = "pag_decode_dc_fwd_tc" if use_tc else ("pag_decode_dc_fwd_tiled" if tiled else "pag_decode_dc_fwd")
        call(entry, ptr(f), ptr(lw), ptr(rd), int(S), M, IN, ptr_array(w), HIDDEN, VIEW_DIM, int(bool(want_rgb)), ptr(sigma), ptr(rgb))
        ctx.save_for_backward(f, lw, rd, *w)
        ctx.S, ctx.want_rgb, ctx.use_tc = int(S), bool(want_rgb), bool(use_tc)
        return sigma, rgb

    @staticmethod
    @once_differentiable
    def backward(ctx, g_sigma, g_rgb):
        f, lw, rd, *w = ctx.saved_tensors
        M, IN = f.shape
        gs = _f32(g_sigma) if g_sigma is not None else None
        gr = _f32(g_rgb) if (g_rgb is not None and ctx.want_rgb) else None
        grads = [torch.zeros_like(x) for x in w]
        need_f, need_d = ctx.needs_input_grad[0], ctx.needs_input_grad[2]
        gf = torch.empty_like(f) if need_f else None
        gd = torch.empty(M, 3, dtype=torch.float32, device=f.device) if need_d else None
        if ctx.use_tc:
            sc = grad_scale(gs, gr)      # held in a local: the tensor must outlive the enqueue of the kernel that reads it
            call("pag_decode_dc_bwd_tc", ptr(f), ptr(lw), ptr(rd), ctx.S, M, IN, ptr_array(w), ptr_array(grads), HIDDEN,
                 VIEW_DIM, ptr(gs), ptr(gr), ptr(sc), ptr(gf), ptr(gd))
        else:
            call("pag_decode_dc_bwd", ptr(f), ptr(lw), ptr(rd), ctx.S, M, IN, ptr_array(w), ptr_array(grads), HIDDEN,
                 VIEW_DIM, ptr(gs), ptr(gr), ptr(gf), ptr(gd))
        if need_d:
            gd = gd.view(-1, ctx.S, 3).sum(1) if ctx.S > 1 else gd
        if gr is None:      # the colour decoder was not evaluated / got no gradient: its parameters receive None, like autograd's
            grads[4:10] = [None] * 6
        return (gf, None, gd, None, None, None, *grads)


class LinearHeadFn(Function):
    """y[m] = b + sum_k (feats + dfeats)[m,k] * lodw[k] * w[k]  (csrc/decoder.cu linear_head_*): the activation-free
    delta-density head of PanopticDDensityNeF after collapsing its two Linear layers on the host."""

    @staticmethod
    def forward(ctx, feats, dfeats, lodw, w, b):
        _chk(feats, dfeats, w, b)
        f, df = _f32(feats), _f32(dfeats)
        M, IN = f.shape
        lw, w_, b_ = _f32(lodw), _f32(w).reshape(-1), _f32(b).reshape(-1)
        y = torch.empty(M, dtype=torch.float32, device=f.device)
        call("pag_linear_head_fwd", ptr(f), ptr(df), ptr(lw), M, IN, ptr(w_), ptr(b_), ptr(y))
        ctx.save_for_backward(f, df, lw, w_)
        ctx.shapes = (w.shape, b.shape)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        f, df, lw, w_ = ctx.saved_tensors
        M, IN = f.shape
        g_ = _f32(g).reshape(-1)
        need_x = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        gx = torch.empty_like(f) if need_x else None
        gw = torch.zeros(IN, dtype=torch.float32, device=f.device)
        gb = torch.zeros(1, dtype=torch.float32, device=f.device)
        call("pag_linear_head_bwd", ptr(f), ptr(df), ptr(lw), M, IN, ptr(w_), ptr(g_), ptr(gx), ptr(gw), ptr(gb))
        return (gx if ctx.needs_input_grad[0] else None, gx if (ctx.needs_input_grad[1] and df is not None) else None, None,
                gw.reshape(ctx.shapes[0]), gb.reshape(ctx.shapes[1]))


class DecodePanFn(Function):
    """semantic + instance decoders on panop = (feats + dfeats) * lodw."""

    @staticmethod
    def forward(ctx, feats, dfeats, lodw, Cs, Ci, sem_softmax, inst_softmax, inst_temperature, use_tc, *weights):
        _chk(feats, dfeats, *weights)
        f = _f32(feats)
        df = _f32(dfeats)
        M, IN = f.shape
        w = [_f32(x) for x in weights]
        sem = torch.empty(M, Cs, dtype=torch.float32, device=f.device) if Cs else None
        inst = torch.empty(M, Ci, dtype=torch.float32, device=f.device) if Ci else None
        lw = _f32(lodw)
        ctx.use_tc = bool(use_tc)
        call("pag_decode_pan_fwd_tc" if use_tc else "pag_decode_pan_fwd", ptr(f), ptr(df), ptr(lw), M, IN, ptr_array(w), HIDDEN, int(Cs), int(Ci),
             int(bool(sem_softmax)), int(bool(inst_softmax)), float(inst_temperature), ptr(sem), ptr(inst))
        ctx.save_for_backward(f, df, lw, sem, inst, *w)
        ctx.cfg = (int(Cs), int(Ci), int(bool(sem_softmax)), int(bool(inst_softmax)), float(inst_temperature))
        return sem, inst

    @staticmethod
    @once_differentiable
    def backward(ctx, g_sem, g_inst):
        f, df, lw, sem, inst, *w = ctx.saved_tensors
        Cs, Ci, ss, is_, it = ctx.cfg
        M, IN = f.shape
        gs = _f32(g_sem) if (g_sem is not None and Cs) else None
        gi = _f32(g_inst) if (g_inst is not None and Ci) else None
        grads = [torch.zeros_like(x) for x in w]
        need = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        gp = torch.empty_like(f) if need else None
        if ctx.use_tc:
            sc = grad_scale(gs, gi)
            call("pag_decode_pan_bwd_tc", ptr(f), ptr(df), ptr(lw), M, IN, ptr_array(w), ptr_array(grads), HIDDEN, Cs, Ci, ss, is_, it,
                 ptr(sem), ptr(inst), ptr(gs), ptr(gi), ptr(sc), ptr(gp))
        else:
            call("pag_decode_pan_bwd", ptr(f), ptr(df), ptr(lw), M, IN, ptr_array(w), ptr_array(grads), HIDDEN, Cs, Ci, ss, is_, it,
                 ptr(sem), ptr(inst), ptr(gs), ptr(gi), ptr(gp))
        if gs is None:      # a head that was not requested leaves its parameters without gradient (None), like autograd would
            grads[0:4] = [None] * 4
        if gi is None:
            grads[4:10] = [None] * 6
        return (gp if ctx.needs_input_grad[0] else None, gp if ctx.needs_input_grad[1] else None,
                None, None, None, None, None, None, None, *grads)


# ------------------------------------------------------------------------------------------------
# compositing
# ------------------------------------------------------------------------------------------------
class CompositeFn(Function):
    """Fused PanopticPackedRFTracer integration (tracers/panoptic_packed_rf_tracer.py:134-205).
    Inputs are packed per sample; `offsets` [R+1] gives each ray's packed range.  Dense [R,*] outputs."""

    @staticmethod
    def forward(ctx, sigma, deltas, depths, rgb, sem, inst, offsets, bg_white):
        _chk(sigma, deltas, offsets)
        sg, dl = _f32(sigma).reshape(-1), _f32(deltas).reshape(-1)
        dp = _f32(depths).reshape(-1) if depths is not None else None
        c = _f32(rgb).reshape(-1, 3) if rgb is not None else None
        se = _f32(sem) if sem is not None else None
        ins = _f32(inst) if inst is not None else None
        R, M, dev = offsets.shape[0] - 1, sg.shape[0], sg.device
        Cs = se.shape[1] if se is not None else 0
        Ci = ins.shape[1] if ins is not None else 0
        w = torch.empty(M, dtype=torch.float32, device=dev)
        T = torch.empty(M, dtype=torch.float32, device=dev)
        alpha = torch.empty(R, 1, dtype=torch.float32, device=dev)
        hit = torch.empty(R, dtype=torch.bool, device=dev)
        rgb_o = torch.empty(R, 3, dtype=torch.float32, device=dev) if c is not None else None
        rgbsum = torch.empty(R, 3, dtype=torch.float32, device=dev) if c is not None else None
        dep_o = torch.empty(R, 1, dtype=torch.float32, device=dev) if dp is not None else None
        sem_o = torch.empty(R, Cs, dtype=torch.float32, device=dev) if se is not None else None
        inst_o = torch.empty(R, Ci, dtype=torch.float32, device=dev) if ins is not None else None
        call("pag_composite_fwd", ptr(sg), ptr(dl), ptr(dp), ptr(c), ptr(se), Cs, ptr(ins), Ci, ptr(offsets), R,
             int(bool(bg_white)), ptr(w), ptr(T), ptr(alpha), ptr(hit), ptr(rgb_o), ptr(rgbsum), ptr(dep_o), ptr(sem_o), ptr(inst_o))
        ctx.save_for_backward(sg, dl, dp, c, offsets, w, T, alpha, rgbsum)
        ctx.cfg = (int(bool(bg_white)), Cs, Ci, sigma.shape, None if rgb is None else rgb.shape)
        ctx.mark_non_differentiable(hit, w)
        return alpha, hit, rgb_o, dep_o, sem_o, inst_o, w

    @staticmethod
    @once_differentiable
    def backward(ctx, g_alpha, g_hit, g_rgb, g_depth, g_sem, g_inst, g_w):
        sg, dl, dp, c, offsets, w, T, alpha, rgbsum = ctx.saved_tensors
        bgw, Cs, Ci, sig_shape, rgb_shape = ctx.cfg
        R, M, dev = offsets.shape[0] - 1, sg.shape[0], sg.device
        ga = _f32(g_alpha) if g_alpha is not None else None
        gr = _f32(g_rgb) if (g_rgb is not None and c is not None) else None
        gd = _f32(g_depth) if (g_depth is not None and dp is not None) else None
        gs = _f32(g_sem) if (g_sem is not None and Cs) else None
        gi = _f32(g_inst) if (g_inst is not None and Ci) else None
        g_sigma = torch.zeros(M, dtype=torch.float32, device=dev)
        g_rgb_s = torch.empty(M, 3, dtype=torch.float32, device=dev) if gr is not None else None
        g_sem_s = torch.empty(M, Cs, dtype=torch.float32, device=dev) if gs is not None else None
        g_inst_s = torch.empty(M, Ci, dtype=torch.float32, device=dev) if gi is not None else None
        call("pag_composite_bwd", ptr(sg), ptr(dl), ptr(dp), ptr(c), ptr(offsets), R, bgw, ptr(w), ptr(T), ptr(alpha),
             ptr(rgbsum), ptr(ga), ptr(gr), ptr(gd), ptr(gs), Cs, ptr(gi), Ci, ptr(g_sigma), ptr(g_rgb_s), ptr(g_sem_s), ptr(g_inst_s))
        return (g_sigma.reshape(sig_shape), None, None,
                g_rgb_s.reshape(rgb_shape) if g_rgb_s is not None else None, g_sem_s, g_inst_s, None, None)


def composite(sigma, deltas, depths, rgb, sem, inst, offsets, bg_white=True):
    """-> alpha [R,1], hit [R], rgb [R,3], depth [R,1], sem [R,Cs], inst [R,Ci], w [M] (detached weights)."""
    return CompositeFn.apply(sigma, deltas, depths, rgb, sem, inst, offsets, bg_white)


def _pan_bwd_workspace(M, IN, Cs, Ci, device):
    return _ws("pag_pan_composite_bwd_workspace", device, M, IN, Cs, Ci)


class _Workspace:
    """Partial weight-gradient workspace of a backward entry point (torch-allocated: graph safe).  The tensor must outlive the
    ENQUEUE of the kernel that uses it -- hold the object in a local until after the call; once the kernel is queued the caching
    allocator's stream-ordered reuse makes dropping it safe."""

    def __init__(self, query, device, *args):
        nbytes = query_i64(query, *[int(a) for a in args])
        self.t = torch.empty(nbytes // 4, dtype=torch.float32, device=device) if nbytes else None
        self.args = (ptr(self.t), nbytes) if nbytes else (None, 0)


def _ws(query, device, *args):
    return _Workspace(query, device, *args)


def pan_composite_f32(feats, dfeats, lodw, w, alpha, ridx, N, Cs, Ci, sem_softmax, inst_softmax, inst_temperature, *weights):
    """Exact-FP32 semantic + instance heads fused with their compositing, forward only (inference; csrc/decoder_tiled.cu):
    per-ray maps [N,Cs], [N,Ci] -- the [M,C] probabilities never reach HBM."""
    _chk(feats, dfeats, w, alpha, ridx, *weights)
    with torch.no_grad():
        f, df = _f32(feats), _f32(dfeats)
        M, IN = f.shape
        wt = [_f32(x) for x in weights]
        lw = _f32(lodw)
        w_, a_ = _f32(w).reshape(-1), _f32(alpha).reshape(-1)
        r_ = ridx.to(torch.int64).contiguous()
        sem = torch.zeros(N, Cs, dtype=torch.float32, device=f.device) if Cs else None
        inst = torch.zeros(N, Ci, dtype=torch.float32, device=f.device) if Ci else None
        call("pag_pan_composite_fwd_f32", ptr(f), ptr(df), ptr(lw), M, IN, ptr_array(wt), HIDDEN, int(Cs), int(Ci),
             int(bool(sem_softmax)), int(bool(inst_softmax)), float(inst_temperature), ptr(w_), ptr(a_), ptr(r_), ptr(sem), ptr(inst))
    return sem, inst


def pan_labels_f32(feats, dfeats, lodw, Cs, Ci, sem_softmax, inst_softmax, inst_temperature, *weights):
    """Exact-FP32 semantic + instance heads reduced to labels, forward only (map export; csrc/decoder_tiled.cu):
    -> (sem_label i64[M], sem_score f32[M], inst_label i64[M], inst_score f32[M]), None for a head with C = 0.  label = argmax of
    the logits (lowest class on ties), score = that class's value of the head's output channel -- the [M,C] tensors never exist."""
    _chk(feats, dfeats, *weights)
    with torch.no_grad():
        f, df = _f32(feats), _f32(dfeats)
        M, IN = f.shape
        wt = [_f32(x) for x in weights]
        lw = _f32(lodw)
        dev = f.device
        sl = torch.empty(M, dtype=torch.int64, device=dev) if Cs else None
        ss = torch.empty(M, dtype=torch.float32, device=dev) if Cs else None
        il = torch.empty(M, dtype=torch.int64, device=dev) if Ci else None
        is_ = torch.empty(M, dtype=torch.float32, device=dev) if Ci else None
        call("pag_pan_labels_fwd_f32", ptr(f), ptr(df), ptr(lw), M, IN, ptr_array(wt), HIDDEN, int(Cs), int(Ci),
             int(bool(sem_softmax)), int(bool(inst_softmax)), float(inst_temperature), ptr(sl), ptr(ss), ptr(il), ptr(is_))
    return sl, ss, il, is_


def map_cell_points(cells, level, k):
    """Sub-cell centres of the leaf cells i16[C,3] of `level`: -> f32[C*k^3, 3] (csrc/mapping.cu pag_map_cell_points)."""
    _chk(cells)
    c = cells.to(torch.int16).contiguous()
    xyz = torch.empty(c.shape[0] * k ** 3, 3, dtype=torch.float32, device=c.device)
    call("pag_map_cell_points", ptr(c), c.shape[0], int(level), int(k), ptr(xyz))
    return xyz


def map_instance_stats(xyz, rgb, semantic, instance, Cs, Ci, thing_mask):
    """-> count i64[Ci], sum_xyz f64[Ci,3], sum_rgb f64[Ci,3], votes i64[Ci,Cs], bbox_min / bbox_max f32[Ci,3], errors i64[1]
    (points with an out-of-range label, counted on the device; csrc/mapping.cu pag_map_instance_stats)."""
    _chk(xyz, rgb, semantic, instance)
    dev = xyz.device
    x, r = _f32(xyz).reshape(-1, 3), _f32(rgb).reshape(-1, 3)
    s, q = semantic.to(torch.int64).contiguous(), instance.to(torch.int64).contiguous()
    P = x.shape[0]
    count = torch.zeros(Ci, dtype=torch.int64, device=dev)
    sum_xyz = torch.zeros(Ci, 3, dtype=torch.float64, device=dev)
    sum_rgb = torch.zeros(Ci, 3, dtype=torch.float64, device=dev)
    votes = torch.zeros(Ci, Cs, dtype=torch.int64, device=dev)
    bmin = torch.full((Ci, 3), float('inf'), dtype=torch.float32, device=dev)
    bmax = torch.full((Ci, 3), float('-inf'), dtype=torch.float32, device=dev)
    errors = torch.zeros(1, dtype=torch.int64, device=dev)
    call("pag_map_instance_stats", ptr(x), ptr(r), ptr(s), ptr(q), P, int(Cs), int(Ci), int(thing_mask) & 0xFFFFFFFF, ptr(count),
         ptr(sum_xyz), ptr(sum_rgb), ptr(votes), ptr(bmin), ptr(bmax), ptr(errors))
    return count, sum_xyz, sum_rgb, votes, bmin, bmax, errors


def map_components(xyz, semantic, instance, level, k, Cs, Ci, thing_mask, connectivity, min_points):
    """Connected components of a labelled lattice map (xyz f32[P,3]; csrc/mapping.cu pag_map_components) -> component i64[P],
    info i64[4] = (K, points off the lattice, duplicate points, points with an out-of-range label), both on the device."""
    _chk(xyz, semantic, instance)
    if xyz.dtype != torch.float32:
        raise TypeError(f"map_components: xyz must be float32 (the lattice is defined bit for bit in fp32), got {xyz.dtype}")
    x = xyz.detach().reshape(-1, 3).contiguous()
    s, q = semantic.to(torch.int64).contiguous(), instance.to(torch.int64).contiguous()
    P = x.shape[0]
    component = torch.empty(P, dtype=torch.int64, device=x.device)
    info = torch.empty(4, dtype=torch.int64, device=x.device)
    ws = _ws("pag_map_components_workspace", x.device, P)
    call("pag_map_components", ptr(x), ptr(s), ptr(q), P, int(level), int(k), int(Cs), int(Ci), int(thing_mask) & 0xFFFFFFFF,
         int(connectivity), int(min_points), *ws.args, ptr(component), ptr(info))
    return component, info


def map_component_stats(xyz, rgb, semantic, instance, component, Cs, K):
    """Per-object statistics of map_components' labelling -> count i64[K], sum_xyz f64[K,3], sum_rgb f64[K,3], votes i64[K,Cs],
    bbox_min / bbox_max f32[K,3], instance i64[K] (csrc/mapping.cu pag_map_component_stats)."""
    _chk(xyz, rgb, semantic, instance, component)
    dev = xyz.device
    x, r = _f32(xyz).reshape(-1, 3), _f32(rgb).reshape(-1, 3)
    s, q = semantic.to(torch.int64).contiguous(), instance.to(torch.int64).contiguous()
    comp = component.to(torch.int64).contiguous()
    count = torch.zeros(K, dtype=torch.int64, device=dev)
    sum_xyz = torch.zeros(K, 3, dtype=torch.float64, device=dev)
    sum_rgb = torch.zeros(K, 3, dtype=torch.float64, device=dev)
    votes = torch.zeros(K, Cs, dtype=torch.int64, device=dev)
    bmin = torch.full((K, 3), float('inf'), dtype=torch.float32, device=dev)
    bmax = torch.full((K, 3), float('-inf'), dtype=torch.float32, device=dev)
    inst = torch.empty(K, dtype=torch.int64, device=dev)
    call("pag_map_component_stats", ptr(x), ptr(r), ptr(s), ptr(q), ptr(comp), x.shape[0], int(Cs), int(K), ptr(count), ptr(sum_xyz),
         ptr(sum_rgb), ptr(votes), ptr(bmin), ptr(bmax), ptr(inst))
    return count, sum_xyz, sum_rgb, votes, bmin, bmax, inst


def map_index(xyz, level, k):
    """Lattice index of a map (xyz f32[P,3]; csrc/mapping.cu pag_map_index) -> keys i64[C], points i32[C], info i64[4] = (points
    inserted, points off the lattice, duplicate points), all on the device.  Allocates the 12 C-byte table and info only."""
    _chk(xyz)
    if xyz.dtype != torch.float32:
        raise TypeError(f"map_index: xyz must be float32 (the lattice is defined bit for bit in fp32), got {xyz.dtype}")
    x = xyz.detach().reshape(-1, 3).contiguous()
    P = x.shape[0]
    C = query_i64("pag_map_index_bytes", P) // 12
    keys = torch.empty(C, dtype=torch.int64, device=x.device)
    points = torch.empty(C, dtype=torch.int32, device=x.device)
    info = torch.empty(4, dtype=torch.int64, device=x.device)
    call("pag_map_index", ptr(x), P, int(level), int(k), ptr(keys), ptr(points), C, ptr(info))
    return keys, points, info


def map_lookup_points(keys, points, level, k, xyz, radius, component=None):
    """Nearest map point (and its component) of each query xyz f32[Q,3] in a map_index table (csrc/mapping.cu
    pag_map_lookup_points) -> point i64[Q], object i64[Q] or None.  Allocates the outputs only (for contiguous inputs)."""
    _chk(keys, points, xyz, component)
    x = xyz.detach().reshape(-1, 3).contiguous()
    Q = x.shape[0]
    point = torch.empty(Q, dtype=torch.int64, device=x.device)
    obj = torch.empty(Q, dtype=torch.int64, device=x.device) if component is not None else None
    call("pag_map_lookup_points", ptr(keys), ptr(points), keys.numel(), int(level), int(k), ptr(x), Q, int(radius),
         ptr(component), ptr(point), ptr(obj))
    return point, obj


def map_lookup_rays(keys, points, level, k, origins, dirs, depth, alpha, min_alpha, radius, component=None):
    """map_lookup_points for the surface point o + d (depth / alpha) of each rendered ray (origins / dirs f32[Q,3], depth / alpha
    f32[Q]; csrc/mapping.cu pag_map_lookup_rays); rays with alpha < min_alpha resolve to -1."""
    _chk(keys, points, origins, dirs, depth, alpha, component)
    o, d = origins.detach().reshape(-1, 3).contiguous(), dirs.detach().reshape(-1, 3).contiguous()
    t, a = depth.detach().reshape(-1).contiguous(), alpha.detach().reshape(-1).contiguous()
    Q = o.shape[0]
    point = torch.empty(Q, dtype=torch.int64, device=o.device)
    obj = torch.empty(Q, dtype=torch.int64, device=o.device) if component is not None else None
    call("pag_map_lookup_rays", ptr(keys), ptr(points), keys.numel(), int(level), int(k), ptr(o), ptr(d), ptr(t), ptr(a),
         float(min_alpha), Q, int(radius), ptr(component), ptr(point), ptr(obj))
    return point, obj


def map_project(xyz, view, intrinsics, H, W, h, near, max_radius, component=None):
    """Z-buffered splatting of the map points xyz f32[P,3] into B views (view f32[B,4,4], intrinsics f32[B,4]; csrc/mapping.cu
    pag_map_project) -> point i64[B,H,W], depth f32[B,H,W], object i64[B,H,W] or None.  Allocates the u64 depth buffer and the
    outputs only (for contiguous inputs)."""
    _chk(xyz, view, intrinsics, component)
    x = xyz.detach().reshape(-1, 3).contiguous()
    V, K = view.detach().contiguous(), intrinsics.detach().contiguous()
    B = V.shape[0]
    dev = x.device
    zbuf = torch.empty(B * H * W, dtype=torch.int64, device=dev)
    point = torch.empty(B, H, W, dtype=torch.int64, device=dev)
    depth = torch.empty(B, H, W, dtype=torch.float32, device=dev)
    obj = torch.empty(B, H, W, dtype=torch.int64, device=dev) if component is not None else None
    call("pag_map_project", ptr(x), x.shape[0], ptr(V), ptr(K), B, int(H), int(W), float(h), float(near), int(max_radius), ptr(zbuf),
         ptr(component), ptr(point), ptr(depth), ptr(obj))
    return point, depth, obj


def silhouette_bitmap_words(total_words, H, W, cap_bytes):
    """-> (words of the bitmap buffer, rounds) pag_map_visibility_silhouette takes for `total_words` words of pair bitmaps under a
    cap of cap_bytes (include/pagnerf_b200.h)"""
    cap = int(cap_bytes) // 4
    if total_words <= cap:
        return total_words, int(total_words > 0)
    step = cap - H * ((W + 31) // 32)
    if step <= 0:
        raise ValueError(f"a silhouette bitmap cap of {cap_bytes} bytes does not exceed the largest bitmap of a {H} x {W} view")
    return cap, -(-total_words // step)


def map_visibility(xyz, view, intrinsics, H, W, h, near, max_radius, component, K, cap_bytes):
    """Per-(view, object) visibility of the map points xyz f32[P,3] in B views (csrc/mapping.cu pag_map_visibility and
    pag_map_visibility_silhouette) -> visible i64[B,K], silhouette i64[B,K], bbox i32[B,K,4] on the device, and on the host the
    number of points whose component lies outside [-1, K) and the total words of the silhouette bitmaps.  One host read between the
    two entries (those two numbers); the silhouettes are skipped when the first is not 0.  Allocates the outputs, the u64 depth
    buffer (freed before the bitmaps), 28 bytes of workspace per pair and at most cap_bytes of bitmaps."""
    _chk(xyz, view, intrinsics, component)
    x = xyz.detach().reshape(-1, 3).contiguous()
    V, Kc = view.detach().contiguous(), intrinsics.detach().contiguous()
    comp = component.contiguous()
    B, P, dev = V.shape[0], x.shape[0], x.device
    N = B * K
    visible = torch.empty(B, K, dtype=torch.int64, device=dev)
    silhouette = torch.empty(B, K, dtype=torch.int64, device=dev)
    bbox = torch.empty(B, K, 4, dtype=torch.int32, device=dev)
    box = torch.empty(N, 4, dtype=torch.int32, device=dev)
    words = torch.empty(N, dtype=torch.int32, device=dev)
    offset = torch.empty(N + 2, dtype=torch.int64, device=dev)
    args = (ptr(x), P, ptr(V), ptr(Kc), B, int(H), int(W), float(h), float(near), int(max_radius), ptr(comp), int(K))
    zbuf = torch.empty(B * H * W if N > 0 and P > 0 else 0, dtype=torch.int64, device=dev)      # nothing to splat otherwise
    call("pag_map_visibility", *args, ptr(zbuf), ptr(box), ptr(words), ptr(offset), ptr(visible), ptr(silhouette), ptr(bbox))
    del zbuf
    total, bad = offset[N:].tolist()                # the one host read
    if bad == 0 and total > 0:
        n_words, _ = silhouette_bitmap_words(total, H, W, cap_bytes)
        bits = torch.empty(n_words, dtype=torch.int32, device=dev)
        call("pag_map_visibility_silhouette", *args, ptr(box), ptr(words), ptr(offset), total, ptr(bits), n_words, ptr(silhouette))
    return visible, silhouette, bbox, bad, total


SHAPE_ACC_WORDS = 22      # i64 accumulators per object of pag_map_shape (include/pagnerf_b200.h)


def map_shape(xyz, level, k, component, K):
    """Size and orientation of each of K map objects (xyz f32[P,3] on the lattice, component i64[P]; csrc/mapping.cu pag_map_shape)
    -> covariance f64[K,3,3], variance f64[K,3], axes f64[K,3,3], center f64[K,3], extent f64[K,3], acc i64[K,22] (the workspace:
    moments, then the order-preserving images of the projections' minima and maxima) and errors i64[2] = (points off the lattice,
    points with a component outside [-1, K)), all on the device.  Allocates the outputs, 176 bytes of workspace per object and 16
    bytes of error counts (for contiguous inputs)."""
    _chk(xyz, component)
    if xyz.dtype != torch.float32:
        raise TypeError(f"map_shape: xyz must be float32 (the lattice is defined bit for bit in fp32), got {xyz.dtype}")
    x = xyz.detach().reshape(-1, 3).contiguous()
    comp = component.contiguous()
    dev = x.device
    f64 = lambda *s: torch.empty(*s, dtype=torch.float64, device=dev)
    cov, var, axes, center, extent = f64(K, 3, 3), f64(K, 3), f64(K, 3, 3), f64(K, 3), f64(K, 3)
    acc = torch.empty(K, SHAPE_ACC_WORDS, dtype=torch.int64, device=dev)
    errors = torch.empty(2, dtype=torch.int64, device=dev)
    call("pag_map_shape", ptr(x), x.shape[0], int(level), int(k), ptr(comp), int(K), ptr(acc), ptr(cov), ptr(var), ptr(axes),
         ptr(center), ptr(extent), ptr(errors))
    return cov, var, axes, center, extent, acc, errors


class PanCompositeFn(Function):
    """Semantic + instance heads fused with their (detached-weight) compositing: per-ray outputs [N,Cs], [N,Ci].
    Tensor-core kernels only (training mode); csrc/decoder_tc_fused.cu."""

    @staticmethod
    def forward(ctx, feats, dfeats, lodw, w, alpha, ridx, N, Cs, Ci, sem_softmax, inst_softmax, inst_temperature, *weights):
        _chk(feats, dfeats, w, alpha, ridx, *weights)
        f, df = _f32(feats), _f32(dfeats)
        M, IN = f.shape
        wt = [_f32(x) for x in weights]
        lw = _f32(lodw)
        w_, a_ = _f32(w).reshape(-1), _f32(alpha).reshape(-1)
        r_ = ridx.to(torch.int64).contiguous()
        sem = torch.zeros(N, Cs, dtype=torch.float32, device=f.device) if Cs else None
        inst = torch.zeros(N, Ci, dtype=torch.float32, device=f.device) if Ci else None
        lse = torch.empty(M, dtype=torch.float32, device=f.device) if (Ci and inst_softmax) else None
        call("pag_pan_composite_fwd_tc", ptr(f), ptr(df), ptr(lw), M, IN, ptr_array(wt), HIDDEN, int(Cs), int(Ci),
             int(bool(sem_softmax)), int(bool(inst_softmax)), float(inst_temperature), ptr(w_), ptr(a_), ptr(r_), ptr(sem), ptr(inst),
             ptr(lse), None, 0)
        ctx.lse = lse
        ctx.save_for_backward(f, df, lw, w_, a_, r_, *wt)
        ctx.cfg = (int(Cs), int(Ci), int(bool(sem_softmax)), int(bool(inst_softmax)), float(inst_temperature))
        return sem, inst

    @staticmethod
    @once_differentiable
    def backward(ctx, g_sem, g_inst):
        f, df, lw, w_, a_, r_, *wt = ctx.saved_tensors
        Cs, Ci, ss, is_, it = ctx.cfg
        M, IN = f.shape
        gs = _f32(g_sem) if (g_sem is not None and Cs) else None
        gi = _f32(g_inst) if (g_inst is not None and Ci) else None
        grads = [torch.zeros_like(x) for x in wt]
        need = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        gp = torch.empty_like(f) if need else None
        if gs is not None or gi is not None:
            wsp = _pan_bwd_workspace(M, IN, Cs, Ci, f.device)
            sc = grad_scale(gs, gi)
            call("pag_pan_composite_bwd_tc", ptr(f), ptr(df), ptr(lw), M, IN, ptr_array(wt), ptr_array(grads), HIDDEN, Cs, Ci,
                 ss, is_, it, ptr(w_), ptr(a_), ptr(r_), int(a_.shape[0]), ptr(gs), ptr(gi), ptr(ctx.lse), ptr(sc), ptr(gp), None,
                 *wsp.args, 0, None, None)
        elif gp is not None:
            gp.zero_()
        return (gp if ctx.needs_input_grad[0] else None, gp if ctx.needs_input_grad[1] else None,
                None, None, None, None, None, None, None, None, None, None, *grads)


# ---- kaolin.render.spc compatible pieces (used by callers that integrate by hand) -----------------
def _pack_offsets(boundary):
    b = boundary.to(torch.bool)
    starts = torch.nonzero(b).flatten()
    return torch.cat([starts, torch.tensor([b.shape[0]], device=b.device, dtype=torch.int64)]).contiguous()


class SumReduceFn(Function):
    @staticmethod
    def forward(ctx, x, offsets):
        x2 = _f32(x)
        R = offsets.shape[0] - 1
        out = torch.empty(R, x2.shape[1], dtype=torch.float32, device=x2.device)
        call("pag_sum_reduce_fwd", ptr(x2), x2.shape[1], ptr(offsets), R, ptr(out))
        ctx.save_for_backward(offsets)
        ctx.shape = x2.shape
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        (offsets,) = ctx.saved_tensors
        gx = torch.zeros(ctx.shape, dtype=torch.float32, device=g.device)
        call("pag_sum_reduce_bwd", ptr(_f32(g)), ctx.shape[1], ptr(offsets), offsets.shape[0] - 1, ptr(gx))
        return gx, None


def sum_reduce(x, boundary):
    """kaolin.render.spc.sum_reduce: [M,C] -> [R,C]."""
    return SumReduceFn.apply(x, _pack_offsets(boundary))


class ExpIntFn(Function):
    @staticmethod
    def forward(ctx, tau, offsets):
        t = _f32(tau).reshape(-1)
        w = torch.empty_like(t)
        T = torch.empty_like(t)
        call("pag_expint_fwd", ptr(t), ptr(offsets), offsets.shape[0] - 1, ptr(w), ptr(T))
        ctx.save_for_backward(w, T, offsets)
        ctx.shape = tau.shape
        return w.reshape(tau.shape)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        w, T, offsets = ctx.saved_tensors
        gt = torch.zeros_like(w)
        call("pag_expint_bwd", ptr(_f32(g).reshape(-1)), ptr(w), ptr(T), ptr(offsets), offsets.shape[0] - 1, ptr(gt))
        return gt.reshape(ctx.shape), None


def exponential_integration(feats, tau, boundary, exclusive=True):
    """kaolin.render.spc.exponential_integration -> (sum_reduce(feats*w) or feats, w)."""
    assert exclusive, "only the exclusive form is used by the reference (tracers/panoptic_packed_rf_tracer.py:135)"
    off = _pack_offsets(boundary)
    w = ExpIntFn.apply(tau, off)
    if feats is None or feats.numel() == 0:
        return feats, w
    return SumReduceFn.apply(feats * w, off), w


# ------------------------------------------------------------------------------------------------
# sync-free fused trace (training mode): march -> encode -> decode -> composite in one autograd node
# ------------------------------------------------------------------------------------------------
_GRAD_SYNC = {"group": None, "enabled": False, "transport": os.environ.get("PAGNERF_GRAD_TRANSPORT", "fp32"),
              "colour_first": os.environ.get("PAGNERF_COLOUR_FIRST", "0") == "1"}
_SIDE_STREAMS = {}
BRANCH_OVERLAP = True    # run the independent branches of the fused trace on two streams (bench.py disables it for its
                         # per-kernel CUDA-event pass so that kernel durations do not overlap)


def _side_stream(device, which=0):
    """Auxiliary streams per device for the branch-level concurrency inside the fused trace (0: panoptic branch, 1: colour-table
    all-reduce, 2: gradient-table zero fill)."""
    if not BRANCH_OVERLAP:
        return torch.cuda.current_stream()
    key = (str(device), which)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=device)
    return _SIDE_STREAMS[key]


def set_grad_sync(enabled, group=None, reserved_sms=0, transport=None, colour_first=None):
    """Ray-sharded data parallelism (SURVEY 8e): when enabled, FusedTraceFn.backward all-reduces (mean) the gradients it
    produces itself -- each grid table as soon as its scatter kernel is queued, on its own stream, so that the NCCL transfer over
    NVLink overlaps the rest of the backward; the flattened decoder gradients (one small bucket) at the end -- and returns
    already-reduced gradients.  One process per GPU, torch.distributed initialised by the caller.
      transport    'fp32' (exact mean) or 'fp16': the two 50 MB tables travel as halfs under a power-of-two scale shared by all
                   ranks (a 4-byte MIN all-reduce of the per-rank scales first); halves the bytes on the wire, 2^-11 relative
                   rounding per element -- inside north_star's 2e-3 for fp16 features.  Default: PAGNERF_GRAD_TRANSPORT or 'fp32'.
                   'symm': the gradient tables live in symmetric memory (parallel.SymmetricGradBuffers) and are reduced IN PLACE by
                   our own kernel over NVLink / NVSwitch peer memory (csrc/allreduce.cu: multimem.ld_reduce + multimem.st through the
                   switch's multicast address, exact fp32) instead of NCCL; the returned table gradients are views of those
                   persistent buffers -- valid until the next backward overwrites them (NCCL backend, one node).
      colour_first issue the colour chain (and the all-reduce of its table) before the panoptic chain instead of after it."""
    _GRAD_SYNC["enabled"], _GRAD_SYNC["group"] = bool(enabled), group
    if transport is not None:
        if transport not in ('fp32', 'fp16', 'symm'):
            raise ValueError("transport must be 'fp32', 'fp16' or 'symm'")
        _GRAD_SYNC["transport"] = transport
    if colour_first is not None:
        _GRAD_SYNC["colour_first"] = bool(colour_first)
    # leave a few SMs to the NCCL kernels: the persistent decoder kernels would otherwise hold every SM until they finish
    # and the "overlapped" all-reduce would start only then
    _lib.load().pag_set_reserved_sms(int(reserved_sms) if enabled else 0, None)


_SYMM = {}


def _symm_grads(device, n_table, n_dtable, n_flat):
    """Per-process symmetric gradient buffers for the 'symm' transport (created collectively at the first backward)."""
    key = (str(device), int(n_table), int(n_dtable), int(n_flat))
    sg = _SYMM.get(key)
    if sg is None:
        from .parallel import SymmetricGradBuffers
        sg = _SYMM[key] = SymmetricGradBuffers({'dtable': n_dtable, 'table': n_table, 'flat': n_flat}, device, _GRAD_SYNC["group"])
    return sg


def _use_symm():
    return _GRAD_SYNC["enabled"] and _GRAD_SYNC.get("transport") == 'symm'


def _dist_world():
    import torch.distributed as dist
    return dist.get_world_size(_GRAD_SYNC["group"])


def _allreduce_mean_async(t):
    """async mean all-reduce; NCCL has a native AVG, other backends (gloo in the tests) sum and divide on wait."""
    import torch.distributed as dist
    g = _GRAD_SYNC["group"]
    if dist.get_backend(g) == 'nccl':
        wk = dist.all_reduce(t, op=dist.ReduceOp.AVG, group=g, async_op=True)
        return lambda: wk.wait()
    wk = dist.all_reduce(t, op=dist.ReduceOp.SUM, group=g, async_op=True)

    def fin():
        wk.wait()
        t.mul_(1.0 / dist.get_world_size(g))
    return fin


def _table_reduce_async(t):
    """Mean all-reduce of a grid-table gradient on the CURRENT stream's timeline; returns fin() to call before the result is used.
    fp16 transport: |t|_max -> power-of-two scale (target 2^14 / world: the sum over the ranks stays below the fp16 maximum) ->
    MIN over the ranks (every rank must use the same scale) -> halfs -> SUM all-reduce -> floats / (scale * world)."""
    import torch.distributed as dist
    if _GRAD_SYNC.get("transport", "fp32") != 'fp16':
        return _allreduce_mean_async(t)
    g = _GRAD_SYNC["group"]
    world = dist.get_world_size(g)
    flat = t.reshape(-1)
    n = flat.numel()
    scr_key = (str(t.device), torch.cuda.current_stream().cuda_stream)
    scratch = _SCALE_SCRATCH.get(scr_key)
    if scratch is None:
        scratch = _SCALE_SCRATCH[scr_key] = torch.zeros(2, dtype=torch.int32, device=t.device)
    scale = torch.empty(1, dtype=torch.float32, device=t.device)
    call("pag_grad_scale", ptr(flat), n, 1, None, 0, 1, None, float(2.0 ** 14 / world), ptr(scratch), ptr(scale))
    dist.all_reduce(scale, op=dist.ReduceOp.MIN, group=g)
    h = torch.empty(n, dtype=torch.float16, device=t.device)
    call("pag_pack_f16", ptr(flat), n, ptr(scale), ptr(h))
    wk = dist.all_reduce(h, op=dist.ReduceOp.SUM, group=g, async_op=True)

    def fin():
        wk.wait()
        call("pag_unpack_f16", ptr(h), n, ptr(scale), 1.0 / world, ptr(flat))
    return fin


# FusedTraceFn can drop zero-density samples after a density-only pass (exact; see pag_compact_count).  It pays when a
# sizeable share of the packed samples is empty space (ReLU-clamped sigma == 0) -- typical of a trained scene; on a
# freshly initialised field (bench.py's synthetic weights: every sample has sigma > 0) the extra pass is pure overhead
# (+0.12 ms on 392 k samples), so it is opt-in: cfg['compact'] / ops.COMPACT_LIVE.
COMPACT_LIVE = False
# L2 persisting windows (north_star design constraint; opt-in, see DESIGN 4.1 for the measurement): during the forward each encoder's
# stream marks ITS table as persisting, during the backward its gradient table; everything else streams through the L2
L2_WINDOW = os.environ.get('PAGNERF_L2_WINDOW', '0') == '1'
SYMM_CHUNKS = int(os.environ.get('PAGNERF_SYMM_CHUNKS', '1'))
SYMM_SPLIT_LEVEL = int(os.environ.get('PAGNERF_SYMM_SPLIT_LEVEL', '0'))      # level ranges of the colour-table scatter / exchange pipeline ('symm' transport)


def _l2_window(t, hit_ratio=1.0):
    if L2_WINDOW:
        lib = _lib.load()
        rc = lib.pag_set_l2_window(ptr(t) if t is not None else None, int(t.numel() * t.element_size()) if t is not None else 0,
                                   float(hit_ratio), _lib.stream())
        if rc != 0:
            raise RuntimeError(f"pagnerf_b200.pag_set_l2_window failed: {rc}")


PREZERO = os.environ.get('PAGNERF_PREZERO', '1') == '1'
VOXEL_SPLIT = os.environ.get('PAGNERF_VOXEL_SPLIT', '0') == '1'
IMG16 = True   # fp16 operand-image interchange between encoders and tensor-core decoders inside FusedTraceFn


def _enc_levels(kind, spec):
    return int(spec[4]) if kind == 'permuto' else int(spec[5])


def _enc_fwd(kind, spec, samples, Mmax, m_dev, ph, table, out, img):
    """Grid encode of the fused trace.  permuto spec: (scale_factor, shift, anneal, capacity, L, n_agg);
    hash spec: (flavour, fparam, res, offset, size, L, round_half, n_agg, cast_half)."""
    if kind == 'permuto':
        sf, sh, an, cap, L, _ = spec
        call("pag_permuto_fwd_img16_dyn" if img else "pag_permuto_fwd_dyn", ptr(samples), Mmax, ptr(m_dev), ph, ptr(table), cap, L, 2,
             ptr(sf), ptr(sh), ptr(an), ptr(out))
    else:
        fl, fparam, res, offset, size, L, round_half, _, cast_half = spec
        if img:
            call("pag_hash_fwd_img16_dyn", int(fl), ptr(samples), Mmax, ptr(m_dev), int(bool(ph and cast_half)), ptr(table), L, 2, ptr(fparam),
                 ptr(res), ptr(offset), ptr(size), ptr(out))
        else:
            call("pag_hash_fwd_dyn", int(fl), ptr(samples), Mmax, ptr(m_dev), int(bool(ph and cast_half)), ptr(table), L, 2, ptr(fparam),
                 ptr(res), ptr(offset), ptr(size), ptr(out), int(bool(round_half)))


def _enc_bwd(kind, spec, samples, Mmax, m_dev, ph, table, g, scale, g_table, g_pos, img, l0=0, l1=None):
    if kind == 'permuto':
        sf, sh, an, cap, L, n_agg = spec
        if img:
            call("pag_permuto_bwd_img16_dyn", ptr(samples), Mmax, ptr(m_dev), ph, ptr(table), cap, L, 2, ptr(sf), ptr(sh), ptr(an),
                 ptr(g), ptr(scale), ptr(g_table), ptr(g_pos), int(n_agg), int(l0), int(L if l1 is None else l1))
        else:
            call("pag_permuto_bwd_dyn", ptr(samples), Mmax, ptr(m_dev), ph, ptr(table), cap, L, 2, ptr(sf), ptr(sh), ptr(an),
                 ptr(g), ptr(g_table), ptr(g_pos), int(n_agg))
    else:
        fl, fparam, res, offset, size, L, _, n_agg, cast_half = spec
        if img:
            call("pag_hash_bwd_img16_dyn", int(fl), ptr(samples), Mmax, ptr(m_dev), int(bool(ph and cast_half)), ptr(table), L, 2, ptr(fparam),
                 ptr(res), ptr(offset), ptr(size), ptr(g), ptr(scale), ptr(g_table), ptr(g_pos), int(n_agg))
        else:
            call("pag_hash_bwd_dyn", int(fl), ptr(samples), Mmax, ptr(m_dev), int(bool(ph and cast_half)), ptr(table), L, 2, ptr(fparam),
                 ptr(res), ptr(offset), ptr(size), ptr(g), ptr(g_table), ptr(g_pos), int(n_agg))


class FusedTraceFn(Function):
    """PanopticPackedRFTracer.trace for ('ray' marching, permutohedral grids, tensor-core decoders) as ONE autograd
    node: ~10 kernel launches forward / ~10 backward, no host synchronisation (the packed-sample count stays on the
    device: every kernel reads it from the marcher's scan), no torch glue between the kernels.  Work buffers are
    sized for the worst case N*S samples; only the first M rows are ever touched.

    cfg: dict(octree, prefix, level, S, near, far, seed, bg_white, pos_half, lodw,
              grid=(sf, shift, anneal, cap, L, n_agg), dgrid=(...) | None, pan_src in {'delta','separate','appearance','none'},
              want_rgb, want_depth, Cs, Ci, sem_softmax, inst_softmax, inst_temperature)
    """

    @staticmethod
    def forward(ctx, origins, dirs, cfg, table, dtable, *weights):
        _chk(origins, dirs, table, *weights)
        ctx.set_materialize_grads(False)      # outputs the loss does not use arrive as None: their backward chain is skipped
        o, d = _f32(origins), _f32(dirs)
        N, S, dev = o.shape[0], int(cfg['S']), o.device
        voxel = cfg.get('march', 'ray') == 'voxel'
        f32, i64 = torch.float32, torch.int64
        counts = torch.empty(max(N, 1), dtype=torch.int32, device=dev)
        offsets = torch.empty(N + 1, dtype=i64, device=dev)
        seed_dev = cfg.get('seed_dev')
        if voxel:
            # 'voxel' marching (kaolin raytrace nuggets, S samples per nugget) without a host sync: the nuggets live in buffers
            # sized for the DDA worst case (a ray crosses at most 3 * 2^level - 2 cells of the level's grid); only the first
            # K = nug_off[N] entries are ever touched.  The max-travel filter is folded into the kept-nugget count.
            level = int(cfg['level'])
            Kmax = max(N * (3 * (1 << level) - 2), 1)      # always the worst case: the staging rows are never clamped
            Mmax = Kmax * S
            cap = Kmax // max(N, 1)
            nug_off = torch.empty(N + 1, dtype=i64, device=dev)
            # ONE octree traversal per ray: nuggets are staged in the ray's own row (worst-case width), the max-travel filter and the
            # sample emit read the rows -- no second DFS, no packed nugget arrays
            stage = torch.empty(max(N, 1) * cap, 2, dtype=f32, device=dev)
            # (the 64-way split of every ray's traversal -- slot_counts argument -- is bit-identical but measured SLOWER on the bench
            # scene: 1.07 ms vs 0.42 ms for 16 384 rays; a million threads that mostly die after two box tests cost more than the
            # latency they hide.  VOXEL_SPLIT=1 keeps it reachable for scenes with much longer traversals.)
            slots = torch.empty(max(N, 1) * 64, dtype=torch.int32, device=dev) if VOXEL_SPLIT else None
            call("pag_raytrace_stage", ptr(cfg['octree']), ptr(cfg['prefix']), ptr(o), ptr(d), N, level, cap, ptr(counts), ptr(nug_off), ptr(stage),
                 ptr(slots))
            rel = torch.empty(max(N, 1) * cap, dtype=torch.int32, device=dev)
            mt = cfg.get('max_travel')
            call("pag_voxel_filter_count_staged", ptr(stage), ptr(nug_off), N, cap, S, int(cfg['seed']), ptr(seed_dev),
                 float(mt if mt is not None else 0.0), int(mt is not None), ptr(rel), ptr(counts), ptr(offsets))
            ridx = torch.empty(Mmax, dtype=i64, device=dev)
            samples = torch.empty(Mmax, 3, dtype=f32, device=dev)
            depths = torch.empty(Mmax, dtype=f32, device=dev)
            deltas = torch.empty(Mmax, dtype=f32, device=dev)
            call("pag_voxel_emit_staged", ptr(o), ptr(d), ptr(stage), ptr(rel), ptr(nug_off), ptr(offsets), N, cap, S,
                 int(cfg['seed']), ptr(seed_dev), ptr(ridx), ptr(samples), ptr(depths), ptr(deltas))
        else:
            Mmax = max(N * S, 1)
            lin = _linspace(S, dev)
            near = float(cfg['near'])
            rng = float(torch.tensor(float(cfg['far']) - near, dtype=f32))
            ridx = torch.empty(Mmax, dtype=i64, device=dev)
            samples = torch.empty(Mmax, 3, dtype=f32, device=dev)
            depths = torch.empty(Mmax, dtype=f32, device=dev)
            deltas = torch.empty(Mmax, dtype=f32, device=dev)
            bits = cfg.get('bits')
            if bits is not None:
                # occupancy bit field instead of the octree descent, 128-bit step masks instead of N*S point indices
                masks = torch.empty(max(N, 1) * ((S + 31) // 32), dtype=torch.int32, device=dev)
                call("pag_march_ray_bits_count", ptr(o), ptr(d), N, S, ptr(lin), None, int(cfg['seed']), near, rng, ptr(bits),
                     int(cfg['level']), ptr(masks), ptr(counts), ptr(offsets), ptr(seed_dev))
                call("pag_march_ray_bits_emit", ptr(o), ptr(d), N, S, ptr(lin), None, int(cfg['seed']), near, rng, ptr(masks),
                     ptr(offsets), ptr(ridx), ptr(samples), ptr(depths), ptr(deltas), ptr(seed_dev))
            else:
                pidx_tmp = torch.empty(Mmax, dtype=torch.int32, device=dev)
                call("pag_march_ray_count", ptr(o), ptr(d), N, S, ptr(lin), None, int(cfg['seed']), near, rng,
                     ptr(cfg['octree']), ptr(cfg['prefix']), int(cfg['level']), ptr(pidx_tmp), ptr(counts), ptr(offsets), ptr(seed_dev))
                call("pag_march_ray_emit", ptr(o), ptr(d), N, S, ptr(lin), None, int(cfg['seed']), near, rng, ptr(pidx_tmp),
                     ptr(offsets), ptr(ridx), None, ptr(samples), ptr(depths), ptr(deltas), None, ptr(seed_dev))
        m_dev = offsets[N:]                      # device-side packed-sample count M
        if seed_dev is not None and not cfg.get('fixed_jitter'):
            seed_dev.add_(1)                     # next replay / step draws the next jitter stream
        kind = cfg.get('grid_kind', 'permuto')
        L = _enc_levels(kind, cfg['grid'])
        IN = L * 2
        tb = table.detach().contiguous()
        ph = int(bool(cfg['pos_half']))
        # the two 50 MB gradient tables of the backward are zero-filled NOW, on their own stream, under the forward's latency-bound
        # decoder kernels (the fill is pure HBM write bandwidth the forward leaves idle) instead of at the head of the backward
        ctx.prezero = None
        if BRANCH_OVERLAP and PREZERO and ctx.needs_input_grad[3] and cfg.get('prezero', True):
            zs = _side_stream(dev, 2)
            if _use_symm():      # gradient tables in symmetric memory: reduced in place by csrc/allreduce.cu
                sg = _symm_grads(dev, tb.numel(), dtable.numel() if dtable is not None else 0, sum(x.numel() for x in weights))
                if getattr(sg, 'in_flight', False):
                    raise RuntimeError("pagnerf_b200: transport='symm' keeps ONE set of persistent gradient buffers per process -- a second "
                                       "fused trace was started before the backward of the previous one (gradient accumulation over "
                                       "several forwards needs transport='fp32')")
                sg.in_flight = True
                g_table0 = sg.view('table').view_as(tb)
                g_dtable0 = sg.view('dtable').view_as(dtable) if (dtable is not None and ctx.needs_input_grad[4]) else None
            else:
                g_table0 = torch.empty_like(tb)
                g_dtable0 = torch.empty_like(dtable) if (dtable is not None and ctx.needs_input_grad[4]) else None
            zs.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(zs):
                g_table0.zero_()
                if g_dtable0 is not None:
                    g_dtable0.zero_()
            ctx.prezero = (g_table0, g_dtable0, zs)
        # fp16 operand-image interchange between the encoders and the tensor-core decoders (one bulk copy per 128-sample tile
        # on the decoder side, coalesced 16-byte accesses on the encoder side); the f32 [M, 2L] layout stays for compaction
        # and for the hash grids
        dd = bool(cfg.get('dd'))      # PanopticDDensity field + tracer: own panoptic density stream, weights carry gradient
        # live-sample compaction drops samples whose COLOUR density is 0; with the DD field the panoptic density
        # relu(y0.detach() + delta_density) can be positive there, so the two are never combined
        compact = bool(cfg.get('compact', COMPACT_LIVE)) and not dd
        img = bool(cfg.get('img16', IMG16)) and not compact and IN % 4 == 0 and (kind == 'hash' or IN % 8 == 0) and (not dd or IN % 16 == 0)
        Tmax = (Mmax + 127) // 128
        nXc = ((IN + 15) // 16) * 2      # 16-byte chunks per row of an operand-image tile (features padded to a multiple of 16)

        def feat_buffer():
            return (torch.empty(Tmax, nXc, 128, 8, dtype=torch.float16, device=dev) if img
                    else torch.empty(Mmax, IN, dtype=f32, device=dev))

        feats = feat_buffer()
        _l2_window(tb)
        _enc_fwd(kind, cfg['grid'], samples, Mmax, m_dev, ph, tb, feats, img)
        w = [_f32(x) for x in weights]
        lodw = _f32(cfg['lodw'])
        want_rgb, want_depth = bool(cfg['want_rgb']), bool(cfg['want_depth'])
        Cs, Ci = int(cfg['Cs']), int(cfg['Ci'])
        src = cfg['pan_src'] if (Cs or Ci) else 'none'
        m_all = m_dev
        if compact:
            # density-only pass over every packed sample, then drop the ones with sigma == 0 (weight 0, gradient 0: exact)
            # from the list; everything below -- colour / panoptic decoders, delta-grid encode, the whole backward -- runs on
            # the survivors.  The list stays ray-sorted; offsets_c / its last entry replace offsets / the sample count.
            sigma0 = torch.empty(Mmax, dtype=f32, device=dev)
            call("pag_decode_dc_fwd_tc_dyn", ptr(feats), ptr(lodw), ptr(d), ptr(ridx), Mmax, ptr(m_dev), IN, ptr_array(w[:10]),
                 HIDDEN, VIEW_DIM, 0, ptr(sigma0), None, None, None, 0)
            offsets_c = torch.empty(N + 1, dtype=i64, device=dev)
            call("pag_compact_count", ptr(sigma0), ptr(offsets), N, ptr(counts), ptr(offsets_c))
            ridx_c = torch.empty(Mmax, dtype=i64, device=dev)
            samples_c = torch.empty(Mmax, 3, dtype=f32, device=dev)
            depths_c = torch.empty(Mmax, dtype=f32, device=dev)
            deltas_c = torch.empty(Mmax, dtype=f32, device=dev)
            feats_c = torch.empty(Mmax, IN, dtype=f32, device=dev)
            call("pag_compact_emit", ptr(sigma0), ptr(offsets), ptr(offsets_c), N, ptr(samples), ptr(depths), ptr(deltas), ptr(feats), IN,
                 ptr(ridx_c), ptr(samples_c), ptr(depths_c), ptr(deltas_c), ptr(feats_c))
            offsets, ridx, samples, depths, deltas, feats = offsets_c, ridx_c, samples_c, depths_c, deltas_c, feats_c
            m_dev = offsets[N:]
        FusedTraceFn.last_live_dev = m_dev
        dfeats = dtb = None
        main = torch.cuda.current_stream()
        side, ev_side = None, None
        if src in ('delta', 'separate'):
            # the delta-grid encode only needs the samples: run it on a side stream, concurrently with the colour
            # decode + scalar compositing (both kernels leave most of the L1 / LSU bandwidth idle)
            dtb = dtable.detach().contiguous()
            dfeats = feat_buffer()
            side = _side_stream(dev)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                _l2_window(dtb)
                _enc_fwd(kind, cfg['dgrid'], samples, Mmax, m_dev, ph, dtb, dfeats, img)
        sigma = torch.empty(Mmax, dtype=f32, device=dev)
        rgb = torch.empty(Mmax, 3, dtype=f32, device=dev) if want_rgb else None
        pe16 = None
        if want_rgb:      # per-ray fp16 view embedding: the decoders copy it instead of 24 sin/cos per sample
            pe16 = torch.empty(N, 32, dtype=torch.float16, device=dev)
            call("pag_view_pe16", ptr(d), N, ptr(pe16))
        ctx.pe16 = pe16
        y0_raw = torch.empty(Mmax, dtype=f32, device=dev) if (dd and (Cs or Ci)) else None
        call("pag_decode_dc_fwd_tc_dyn", ptr(feats), ptr(lodw), ptr(d), ptr(ridx), Mmax, ptr(m_dev), IN, ptr_array(w[:10]),
             HIDDEN, VIEW_DIM, int(want_rgb), ptr(sigma), ptr(rgb), ptr(y0_raw), ptr(pe16), int(img))
        wgt = torch.empty(Mmax, dtype=f32, device=dev)
        T = torch.empty(Mmax, dtype=f32, device=dev)
        alpha = torch.empty(N, 1, dtype=f32, device=dev)
        hit = torch.empty(N, dtype=torch.bool, device=dev)
        rgb_o = torch.empty(N, 3, dtype=f32, device=dev) if want_rgb else None
        rgbsum = torch.empty(N, 3, dtype=f32, device=dev) if want_rgb else None
        dep_o = torch.empty(N, 1, dtype=f32, device=dev) if want_depth else None
        bgw = int(bool(cfg['bg_white']))
        call("pag_composite_fwd", ptr(sigma), ptr(deltas), ptr(depths) if want_depth else None, ptr(rgb), None, 0, None, 0,
             ptr(offsets), N, bgw, ptr(wgt), ptr(T), ptr(alpha), ptr(hit), ptr(rgb_o), ptr(rgbsum), ptr(dep_o), None, None)
        sem_o = inst_o = None
        ctx.lse = None
        dd_saved = (None,) * 6
        if Cs or Ci:
            sem_o = torch.zeros(N, Cs, dtype=f32, device=dev) if Cs else None
            inst_o = torch.zeros(N, Ci, dtype=f32, device=dev) if Ci else None
            if side is not None:
                main.wait_stream(side)
            a, b = {'delta': (feats, dfeats), 'separate': (dfeats, None), 'appearance': (feats, None)}[src]
            lse = torch.empty(Mmax, dtype=f32, device=dev) if (Ci and cfg['inst_softmax']) else None
            pw, pa = wgt, alpha
            if dd:
                # panoptic density stream (pc_nerf/panoptic_dd_nef.py:236-245, tracers/panoptic_dd_packed_rf_tracer.py:128-137):
                # tau_p = relu(y0.detach() + delta_density(panop)) * delta -> integration weights that carry gradient
                tau_p = torch.empty(Mmax, dtype=f32, device=dev)
                call("pag_linear_head_fwd_dyn", ptr(a), ptr(b), ptr(lodw), Mmax, ptr(m_dev), IN, ptr(w[20]), ptr(w[21]), ptr(y0_raw), 1,
                     ptr(deltas), ptr(tau_p), int(img))
                pw = torch.empty(Mmax, dtype=f32, device=dev)
                T_p = torch.empty(Mmax, dtype=f32, device=dev)
                call("pag_expint_fwd", ptr(tau_p), ptr(offsets), N, ptr(pw), ptr(T_p))
                pa = torch.empty(N, 1, dtype=f32, device=dev)
                call("pag_sum_reduce_fwd", ptr(pw), 1, ptr(offsets), N, ptr(pa))
                dd_saved = (tau_p, pw, T_p, pa, sem_o, inst_o)
            call("pag_pan_composite_fwd_tc", ptr(a), ptr(b), ptr(lodw), Mmax, IN, ptr_array(w[10:20]), HIDDEN, Cs, Ci,
                 int(bool(cfg['sem_softmax'])), int(bool(cfg['inst_softmax'])), float(cfg['inst_temperature']),
                 ptr(pw), ptr(pa), ptr(ridx), ptr(sem_o), ptr(inst_o), ptr(lse), ptr(m_dev), int(img))
            ctx.lse = lse
        ctx.cfg, ctx.img, ctx.IN = cfg, img, IN
        ctx.save_for_backward(o, d, offsets, ridx, samples, depths, deltas, feats, dfeats, sigma, rgb, wgt, T, alpha, rgbsum,
                              tb, dtb, lodw, *dd_saved, *w)
        ctx.mark_non_differentiable(hit)
        ctx.last_m_dev = m_all
        return alpha, hit, rgb_o, dep_o, sem_o, inst_o, m_all

    @staticmethod
    @once_differentiable
    def backward(ctx, g_alpha, g_hit, g_rgb, g_depth, g_sem, g_inst, g_m):
        (o, d, offsets, ridx, samples, depths, deltas, feats, dfeats, sigma, rgb, wgt, T, alpha, rgbsum, tb, dtb, lodw,
         dd_tau, dd_w, dd_T, dd_alpha, dd_sem, dd_inst, *w) = ctx.saved_tensors
        cfg = ctx.cfg
        N, dev = o.shape[0], o.device
        img, IN = ctx.img, ctx.IN
        Mmax = samples.shape[0]
        Tmax = (Mmax + 127) // 128
        m_dev = offsets[N:]

        nXc = ((IN + 15) // 16) * 2

        def grad_buffer():      # feature gradients: fp16 operand images (still carrying the loss scale) or f32 rows
            return (torch.empty(Tmax, nXc, 128, 8, dtype=torch.float16, device=dev) if img
                    else torch.empty(Mmax, IN, dtype=torch.float32, device=dev))

        f32 = torch.float32
        kind = cfg.get('grid_kind', 'permuto')
        L = _enc_levels(kind, cfg['grid'])
        ph = int(bool(cfg['pos_half']))
        Cs, Ci = int(cfg['Cs']), int(cfg['Ci'])
        sync, fins = _GRAD_SYNC["enabled"], []
        smask = int(os.environ.get('PAGNERF_SYNC_MASK', '7'))      # debugging: bit 0 delta table, bit 1 colour table, bit 2 decoders
        sizes = [x.numel() for x in w]
        symm = _symm_grads(dev, tb.numel(), dtb.numel() if dtb is not None else 0, sum(sizes)) if (sync and _use_symm()) else None
        if symm is not None:
            symm.in_flight = False
            flat = symm.view('flat')
            flat.zero_()
        else:
            flat = torch.zeros(sum(sizes), dtype=f32, device=dev)          # all 20 decoder gradients: one memset
        grads = [t.view_as(x) for t, x in zip(flat.split(sizes), w)]
        gs = _f32(g_sem) if (g_sem is not None and Cs) else None
        gi = _f32(g_inst) if (g_inst is not None and Ci) else None
        main = torch.cuda.current_stream()
        # gradient tables: zero-filled during the forward on their own stream when the forward could tell they would be needed
        g_table0, g_dtable0, zs = ctx.prezero if ctx.prezero is not None else (None, None, None)
        ctx.prezero = None
        if zs is not None:
            main.wait_stream(zs)
        # 'keep': every temporary that a kernel on ANOTHER stream than its allocation stream touches stays referenced until the
        # streams have been joined at the end of this function -- a tensor that dies earlier goes back to its allocation
        # stream's pool and the next allocation there (e.g. the colour chain's gradient image) would alias it while the side
        # stream is still reading
        st = {'g_dtable': None, 'g_table': None, 'g_o': None, 'g_d': None, 'side': None, 'comm': None, 'keep': []}
        want_rgb, want_depth = bool(cfg['want_rgb']), bool(cfg['want_depth'])
        ga = _f32(g_alpha) if g_alpha is not None else None
        gr = _f32(g_rgb) if (g_rgb is not None and want_rgb) else None
        gd = _f32(g_depth) if (g_depth is not None and want_depth) else None
        need_rays = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        colour_ran = ga is not None or gr is not None or gd is not None

        def run_pan():
            # panoptic chain (heads backward -> delta-grid scatter [-> all-reduce]) on a side stream; it shares nothing
            # with the colour chain except read-only inputs, and the two sets of kernels overlap on the SMs
            src = cfg['pan_src']
            a, b = {'delta': (feats, dfeats), 'separate': (dfeats, None), 'appearance': (feats, None)}[src]
            need_gp = src in ('delta', 'separate')          # 'appearance': features are detached -> nothing upstream
            g_panop = grad_buffer() if need_gp else None
            side = st['side'] = _side_stream(dev)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                if need_gp:
                    if g_dtable0 is not None:
                        st['g_dtable'] = g_dtable0
                    elif symm is not None:
                        st['g_dtable'] = symm.view('dtable').view_as(dtb)
                        st['g_dtable'].zero_()
                    else:
                        st['g_dtable'] = torch.zeros_like(dtb)
                scale_p = grad_scale_dyn(gs if gs is not None else gi, gi if gs is not None else None, None)
                dds = (dd_tau, dd_w, dd_T, dd_alpha, dd_sem, dd_inst) if dd_tau is not None else None
                pw, pa = (dd_w, dd_alpha) if dds is not None else (wgt, alpha)
                gw_sem = torch.empty(Mmax, dtype=f32, device=dev) if (dds is not None and gs is not None) else None
                gw_inst = torch.empty(Mmax, dtype=f32, device=dev) if (dds is not None and gi is not None) else None
                wsp = _pan_bwd_workspace(Mmax, IN, Cs, Ci, dev)
                call("pag_pan_composite_bwd_tc", ptr(a), ptr(b), ptr(lodw), Mmax, IN, ptr_array(w[10:20]), ptr_array(grads[10:20]), HIDDEN,
                     Cs, Ci, int(bool(cfg['sem_softmax'])), int(bool(cfg['inst_softmax'])), float(cfg['inst_temperature']),
                     ptr(pw), ptr(pa), ptr(ridx), int(alpha.shape[0]), ptr(gs), ptr(gi), ptr(ctx.lse), ptr(scale_p), ptr(g_panop), ptr(m_dev),
                     *wsp.args, int(img), ptr(gw_sem), ptr(gw_inst))
                if dds is not None:
                    # the panoptic weights carry gradient: d L / d w_p -> reverse scan -> tau_p -> ReLU gate -> delta-density head
                    tau_p, _, T_p, _, sem_o, inst_o = dds
                    gwt = torch.empty(Mmax, dtype=f32, device=dev)
                    call("pag_dd_weight_grads", ptr(gs), ptr(sem_o) if gs is not None else None, Cs, ptr(gi),
                         ptr(inst_o) if gi is not None else None, Ci, ptr(pa), ptr(gw_sem), ptr(gw_inst), ptr(offsets), N, ptr(gwt))
                    gtau = torch.empty(Mmax, dtype=f32, device=dev)
                    call("pag_expint_bwd", ptr(gwt), ptr(pw), ptr(T_p), ptr(offsets), N, ptr(gtau))
                    call("pag_linear_head_bwd_dyn", ptr(a), ptr(b), ptr(lodw), Mmax, ptr(m_dev), IN, ptr(w[20]), ptr(gtau), ptr(tau_p),
                         ptr(deltas), ptr(g_panop), 1, ptr(grads[20]), ptr(grads[21]), int(img), ptr(scale_p))
                    st['keep'] += [gwt, gtau]
                st['keep'] += [g_panop, scale_p, gw_sem, gw_inst, wsp]
                if need_gp:
                    _l2_window(st['g_dtable'])
                    _enc_bwd(kind, cfg['dgrid'], samples, Mmax, m_dev, ph, dtb, g_panop, scale_p, st['g_dtable'], None, img)
                    if sync and symm is not None and (smask & 1):
                        symm.allreduce('dtable', channel=0)      # on the side stream: overlaps whatever of the backward is still queued
                    elif sync and (smask & 1):
                        fins.append((side, _table_reduce_async(st['g_dtable'])))   # overlaps whatever of the backward is still queued

        def run_colour():
            # scalar compositing backward -> per-sample sigma / rgb gradients -> density / colour decoders -> colour-grid scatter
            if g_table0 is not None:
                g_table = g_table0
            elif symm is not None:
                g_table = symm.view('table').view_as(tb)
                g_table.zero_()
            else:
                g_table = torch.zeros_like(tb)
            st['g_table'] = g_table
            g_sigma = torch.empty(Mmax, dtype=f32, device=dev)
            g_rgb_s = torch.empty(Mmax, 3, dtype=f32, device=dev) if gr is not None else None
            call("pag_composite_bwd", ptr(sigma), ptr(deltas), ptr(depths) if gd is not None else None, ptr(rgb), ptr(offsets), N,
                 int(bool(cfg['bg_white'])), ptr(wgt), ptr(T), ptr(alpha), ptr(rgbsum), ptr(ga), ptr(gr), ptr(gd), None, 0, None, 0,
                 ptr(g_sigma), ptr(g_rgb_s), None, None)
            scale = grad_scale_dyn(g_sigma, g_rgb_s, m_dev, 1, 3)
            g_feats = grad_buffer()
            g_dir = torch.empty(Mmax, 3, dtype=f32, device=dev) if ctx.needs_input_grad[1] else None
            wsd = _ws("pag_decode_dc_bwd_workspace", dev, Mmax, IN)
            call("pag_decode_dc_bwd_tc_dyn", ptr(feats), ptr(lodw), ptr(d), ptr(ridx), Mmax, ptr(m_dev), IN, ptr_array(w[:10]),
                 ptr_array(grads[:10]), HIDDEN, VIEW_DIM, ptr(g_sigma), ptr(g_rgb_s), ptr(scale), ptr(g_feats), ptr(g_dir),
                 ptr(ctx.pe16), *wsd.args, int(img))
            g_pos = torch.empty(Mmax, 3, dtype=f32, device=dev) if need_rays else None
            st['keep'] += [g_sigma, g_rgb_s, g_feats, g_dir, g_pos, scale, wsd]
            _l2_window(g_table)
            # 'symm' transport, opt-in (PAGNERF_SYMM_CHUNKS > 1): the colour table is the last gradient of the step, nothing is left
            # to hide its exchange behind -- scatter it in level ranges and let every finished range leave on the exchange stream
            # while the next one is being scattered.  Measured at 2 GPUs: 1 / 2 / 3 ranges = 1.53 / 1.51 / 1.55 ms (the extra passes
            # over the samples eat the overlap), so the default stays 1.
            nchunk = SYMM_CHUNKS if (sync and symm is not None and (smask & 2) and img and kind == 'permuto' and L % SYMM_CHUNKS == 0) else 1
            bounds = [(c * (L // nchunk), (c + 1) * (L // nchunk)) for c in range(nchunk)]
            if sync and symm is not None and (smask & 2) and img and kind == 'permuto' and 0 < SYMM_SPLIT_LEVEL < L:
                # uneven two-way split: the big first range leaves while the small last one is scattered, so that only a small
                # exchange is left exposed at the end of the step
                bounds, nchunk = [(0, SYMM_SPLIT_LEVEL), (SYMM_SPLIT_LEVEL, L)], 2
            per_level = tb.numel() // L
            for c in range(nchunk):
                l0, l1 = bounds[c]
                _enc_bwd(kind, cfg['grid'], samples, Mmax, m_dev, ph, tb, g_feats, scale, g_table, g_pos, img, l0, l1 if nchunk > 1 else None)
                if sync and (symm is not None or (smask & 2)):
                    comm = st['comm'] = _side_stream(dev, 1)
                    comm.wait_stream(main)
                    with torch.cuda.stream(comm):
                        if symm is not None and (smask & 2):
                            symm.allreduce('table', channel=1, sub=(l0 * per_level, (l1 - l0) * per_level))
                        elif symm is None and (smask & 2):
                            fins.append((comm, _table_reduce_async(g_table)))
            if need_rays:   # d samples / d (origin, dir): segment sums over each ray's packed range
                st['g_o'] = torch.empty(N, 3, dtype=f32, device=dev)
                st['g_d'] = torch.empty(N, 3, dtype=f32, device=dev)
                gpt = torch.addcmul(g_dir, g_pos, depths.unsqueeze(1)) if g_dir is not None else (g_pos * depths.unsqueeze(1))
                call("pag_sum_reduce_fwd", ptr(g_pos), 3, ptr(offsets), N, ptr(st['g_o']))
                call("pag_sum_reduce_fwd", ptr(gpt.contiguous()), 3, ptr(offsets), N, ptr(st['g_d']))

        pan_ran = gs is not None or gi is not None
        order = (run_colour, run_pan) if _GRAD_SYNC.get("colour_first") else (run_pan, run_colour)
        for fn in order:
            if (fn is run_pan and pan_ran) or (fn is run_colour and colour_ran):
                fn()
        for strm, fin in fins:      # finish each table's reduction on the stream that issued it (unpack kernels overlap too)
            with torch.cuda.stream(strm):
                fin()
        for strm in (st['side'], st['comm']):
            if strm is not None:
                main.wait_stream(strm)
        if sync and symm is not None and (smask & 4):
            symm.allreduce('flat', channel=2, max_ctas=16)
        elif sync and symm is None and (smask & 4):
            _allreduce_mean_async(flat)()
        g_table, g_dtable, g_o, g_d = st['g_table'], st['g_dtable'], st['g_o'], st['g_d']
        # parameters of heads that were not requested (or got no upstream gradient) receive None, like the reference's autograd
        gout = list(grads)
        if not colour_ran:
            gout[0:4] = [None] * 4
            g_table = None
        if not (colour_ran and gr is not None):
            gout[4:10] = [None] * 6
        if gs is None:
            gout[10:14] = [None] * 4
        if gi is None:
            gout[14:20] = [None] * 6
        if len(gout) > 20 and gs is None and gi is None:
            gout[20:] = [None] * (len(gout) - 20)
        return (g_o if ctx.needs_input_grad[0] else None, g_d if ctx.needs_input_grad[1] else None, None,
                g_table, g_dtable, *gout)
