"""PanopticNeF: grid encoder + density / color / semantic / instance decoders.

Drop-in for the reference class (pc_nerf/panoptic_nef.py:20-363): same constructor arguments,
attributes, parameter names (`grid.*`, `decoder_density.*`, `decoder_color.*`,
`decoder_semantics.*`, `decoder_inst.*`), channel dispatch and output shapes.  The forward itself
is two fused kernels (csrc/decoder.cu) on top of the grid's encode kernel instead of 9 GEMMs and
~15 elementwise launches.
"""
import logging as log

import numpy as np
import torch
import torch.nn.functional as F

from .. import ops, spc
from ..grids import HashGridTorch, HashGridTinyCudaNN, PermutoGrid
from ..wisp_compat import (BaseNeuralField, BasicDecoder, PerfTimer, get_activation_class, get_layer_class,
                           get_positional_embedder)


def _decoder_tensors(dec, n_hidden):
    """[W0,b0,(W1,b1,)Wout,bout] of a BasicDecoder; validates the shapes csrc/decoder.cu is built for."""
    if len(dec.layers) != n_hidden or any(l.out_features != ops.HIDDEN for l in dec.layers) or not dec.bias or dec.skip:
        raise NotImplementedError(
            "csrc/decoder.cu is specialised to the reference configuration (configs/bup20/*.yaml: hidden_dim 64, "
            "density/semantic decoders with 1 hidden layer, color/instance with 2, bias, no skip)")
    out = []
    for l in dec.layers:
        out += [l.weight, l.bias]
    return out + [dec.lout.weight, dec.lout.bias]


class PanopticNeF(BaseNeuralField):
    def __init__(self,
                 num_classes: int = -1, num_instances: int = -1,
                 sem_activation_type: str = None, sem_num_layers: int = None, sem_hidden_dim: int = None,
                 sem_normalize: bool = False, sem_softmax: bool = False, sem_sigmoid: bool = False, sem_detach: bool = True,
                 inst_num_layers: int = None, inst_hidden_dim: int = None, inst_normalize: bool = False,
                 inst_softmax: bool = False, inst_sigmoid: bool = False, inst_detach: bool = True,
                 panoptic_features_type: str = None, **kwargs):
        self.num_classes = num_classes
        self.num_instances = num_instances
        self.sem_activation_type = sem_activation_type
        self.sem_num_layers = sem_num_layers
        self.sem_hidden_dim = sem_hidden_dim
        self.sem_normalize = sem_normalize
        self.sem_softmax = sem_softmax
        self.sem_sigmoid = sem_sigmoid
        self.sem_detach = sem_detach
        self.inst_num_layers = inst_num_layers
        self.inst_hidden_dim = inst_hidden_dim
        self.inst_detach = inst_detach
        self.inst_softmax = inst_softmax
        self.inst_normalize = inst_normalize
        self.inst_sigmoid = inst_sigmoid
        self.panoptic_features_type = panoptic_features_type
        # the reference never assigns this attribute (latent AttributeError, SURVEY 8 a-5); define it
        self.inst_direct_pos = bool(kwargs.get('inst_direct_pos', False))
        super().__init__(**kwargs)

    # ---- construction (mirrors pc_nerf/panoptic_nef.py:72-196) ------------------------------------
    def init_embedder(self):
        self.view_embedder, self.view_embed_dim = get_positional_embedder(self.view_multires,
                                                                          self.embedder_type == "positional")
        log.info(f"View Embed Dim: {self.view_embed_dim}")

    def _compute_input_dimension(self):
        if self.position_input:
            raise NotImplementedError
        if self.multiscale_type == 'cat':
            self.effective_feature_dim = self.grid.feature_dim * self.num_lods
        elif self.multiscale_type == 'sum':
            self.effective_feature_dim = self.grid.feature_dim
        else:
            raise NotImplementedError(f"'{self.multiscale_type}' not supported by this neural field. "
                                      "supported options ['cat', 'sum']")
        self.input_dim_density = self.effective_feature_dim
        if self.panoptic_features_type == 'position':
            self.input_dim_inst = self.input_dim_sem = 3
        elif self.panoptic_features_type == 'pos_encoding':
            self.input_dim_inst = self.input_dim_sem = self.pos_embed_dim
        else:
            self.input_dim_inst = self.input_dim_sem = self.effective_feature_dim

    def init_decoder(self):
        self._compute_input_dimension()
        act, layer = get_activation_class(self.activation_type), get_layer_class(self.layer_type)
        self.decoder_density = BasicDecoder(input_dim=self.input_dim_density, output_dim=16, activation=act, bias=True,
                                            layer=layer, num_layers=self.num_layers, hidden_dim=self.hidden_dim, skip=[])
        self.decoder_density.lout.bias.data[0] = 1.0
        self.decoder_color = BasicDecoder(input_dim=16 + self.view_embed_dim, output_dim=3, activation=act, bias=True,
                                          layer=layer, num_layers=self.num_layers + 1, hidden_dim=self.hidden_dim, skip=[])
        self.sem_activation_type = self.sem_activation_type if self.sem_activation_type else self.activation_type
        self.sem_num_layers = self.sem_num_layers if self.sem_num_layers else self.num_layers
        self.sem_hidden_dim = self.sem_hidden_dim if self.sem_hidden_dim else self.hidden_dim
        sact = get_activation_class(self.sem_activation_type)
        self.decoder_semantics = BasicDecoder(input_dim=self.input_dim_sem, output_dim=self.num_classes, activation=sact,
                                              bias=True, layer=layer, num_layers=self.sem_num_layers,
                                              hidden_dim=self.sem_hidden_dim, skip=[])
        assert self.num_instances > 2, f"'num_instances' needs to be >= 2, but {self.num_classes} was given."
        self.inst_num_layers = self.inst_num_layers if self.inst_num_layers else self.num_layers
        self.inst_hidden_dim = self.inst_hidden_dim if self.inst_hidden_dim else self.hidden_dim
        self.decoder_inst = BasicDecoder(input_dim=self.input_dim_inst, output_dim=self.num_instances, activation=sact,
                                         bias=True, layer=layer, num_layers=self.inst_num_layers,
                                         hidden_dim=self.inst_hidden_dim, skip=[])

    def _get_grid_class(self):
        table = {"HashGridTorch": HashGridTorch, "HashGridTinyCudaNN": HashGridTinyCudaNN, "PermutoGrid": PermutoGrid}
        if self.grid_type not in table:
            raise NotImplementedError(f"'{self.grid_type}' not supproted")
        return table[self.grid_type]

    def init_grid(self):
        self.grid = self._get_grid_class()(self.feature_dim, base_lod=self.base_lod, num_lods=self.num_lods,
                                           interpolation_type=self.interpolation_type, multiscale_type='cat',
                                           **self.kwargs)
        self.lod_weights = torch.ones(self.num_lods * self.grid.feature_dim)

    def get_nef_type(self):
        return 'panoptic_nef'

    # ---- pruning (pc_nerf/panoptic_nef.py:207-237) ------------------------------------------------
    def _prune_grids(self):
        return [self.grid]

    def _prune_supported(self):
        # the base field prunes the hash grids only and raises for anything else (pc_nerf/panoptic_nef.py:211,235)
        return self.grid_type in ["HashGrid", "HashGridTorch", "HashGridTinyCudaNN", "TriplanarGrid"]

    def prune(self):
        if self.grid is None:
            return
        if not self._prune_supported():
            raise NotImplementedError
        density_decay = 0.6
        min_density = ((0.01 * 512) / np.sqrt(3))
        dev = self.device
        self.grid.occupancy = self.grid.occupancy.to(dev) * density_decay
        points = self.grid.dense_points.to(dev)
        res = 2.0 ** self.grid.blas_level
        samples = torch.rand(points.shape[0], 3, device=dev)
        samples = (points.float() + samples) / res * 2.0 - 1.0
        sample_views = F.normalize(torch.randn(samples.shape[0], 3, device=dev), dim=-1)
        with torch.no_grad():
            density = self.forward(coords=samples[:, None], ray_d=sample_views, channels="density")
        self.grid.occupancy = torch.stack([density[:, 0, 0], self.grid.occupancy], -1).max(dim=-1)[0]
        mask = self.grid.occupancy > min_density
        _points = points[mask]
        for grid in self._prune_grids():
            if mask.is_cuda and mask.numel() == 8 ** grid.blas_level:
                # device-side rebuild straight from the dense mask (csrc/octree.cu pag_octree_from_mask): same octree bytes as
                # unbatched_points_to_octree(points[mask]) -- `dense_points` is in Morton order
                grid.blas_init_from_mask(mask, register=self.grid_type == "PermutoGrid")
                continue
            octree = spc.unbatched_points_to_octree(_points, grid.blas_level, sorted=True)
            # PermutoGrid re-registers its checkpoint buffers (blas_octree / points / prefix / pyramid); the hash grids keep
            # the state_dict keys they were built with (pc_nerf/panoptic_delta_nef.py:98-104, pc_nerf/panoptic_nef.py:233)
            if self.grid_type == "PermutoGrid":
                grid.blas_init(octree)
            else:
                grid.blas.init(octree)

    # ---- forward ---------------------------------------------------------------------------------
    def forward(self, channels=None, **kwargs):
        kwargs['compute_channels'] = channels
        return super().forward(channels, **kwargs)

    def register_forward_functions(self):
        self._register_forward_function(self.rgb_semantics, ["density", "rgb", "semantics", "inst_embedding"])

    def _encode(self, grid, coords, lod_idx):
        feats = grid.interpolate(coords, lod_idx)
        feats = feats.reshape(-1, feats.shape[-1])
        if self.multiscale_type == 'sum':
            raise NotImplementedError("multiscale_type='sum' is not served by the fused decoders "
                                      "(every reference config uses 'cat', configs/bup20/*.yaml)")
        return feats

    # decoder arithmetic: 'auto' = tensor cores (fp16 operands, fp32 accumulate) under torch autocast -- what the
    # reference's training step runs (pc_nerf/trainer.py:429) -- and exact fp32 otherwise (validation, :683);
    # 'fp32' / 'fp16' force one of the two kernels.
    decoder_precision = 'auto'

    def _lodw(self, device):
        """lod_weights on `device`, cached (the attribute is a CPU tensor that LOD annealing may replace / edit)."""
        t = self.lod_weights
        key = (id(t), t._version, str(device))
        if getattr(self, '_lodw_key', None) != key:
            new = t.detach().to(device=device, dtype=torch.float32).contiguous()
            old = getattr(self, '_lodw_dev', None)
            if old is not None and old.shape == new.shape and old.device == new.device:
                old.copy_(new)      # in place: a captured CUDA graph (graph.GraphedStep) keeps reading the live weights
            else:
                self._lodw_dev = new
            self._lodw_key = key
        return self._lodw_dev

    def _use_tc(self):
        if self.decoder_precision == 'auto':
            return torch.is_autocast_enabled()
        return self.decoder_precision == 'fp16'

    def _dc(self, feats, ray_d, num_samples, want_rgb):
        w = _decoder_tensors(self.decoder_density, 1) + _decoder_tensors(self.decoder_color, 2)
        lodw = self._lodw(feats.device)
        return ops.DecodeDCFn.apply(feats, lodw, ray_d, num_samples, want_rgb, ops.dc_mode(self._use_tc(), feats.shape[-1]), *w)

    def _pan(self, feats, dfeats, want_sem, want_inst, inst_temperature=0.0):
        """semantic / instance heads on (feats + dfeats) * lod_weights; non-default sigmoid / normalize
        options are composed on the host from the raw logits."""
        w = _decoder_tensors(self.decoder_semantics, 1) + _decoder_tensors(self.decoder_inst, 2)
        lodw = self._lodw(feats.device)
        sem_plain = not (self.sem_sigmoid or self.sem_normalize)
        inst_plain = not (self.inst_sigmoid or self.inst_normalize)
        Cs = self.num_classes if want_sem else 0
        Ci = self.num_instances if want_inst else 0
        sem, inst = ops.DecodePanFn.apply(feats, dfeats, lodw, Cs, Ci, bool(self.sem_softmax and sem_plain),
                                          bool(self.inst_softmax and inst_plain),
                                          float(inst_temperature if inst_plain else 0.0), self._use_tc(), *w)
        if want_sem and not sem_plain:
            sem = torch.sigmoid(sem) if self.sem_sigmoid else sem
            sem = F.normalize(sem, dim=-1) if self.sem_normalize else sem
            sem = F.softmax(sem, dim=-1) if self.sem_softmax else sem
        if want_inst and not inst_plain:
            inst = torch.sigmoid(inst) if self.inst_sigmoid else inst
            inst = F.normalize(inst, dim=-1) if self.inst_normalize else inst
            inst = inst / inst_temperature if inst_temperature > 0.0 else inst
            inst = F.softmax(inst, dim=-1) if self.inst_softmax else inst
        return sem, inst

    # ---- fused decode + composite (used by PanopticPackedRFTracer.trace in training mode) --------------------
    def _panoptic_inputs(self, feats, coords, lod_idx, rows=None):
        """(a, b): the panoptic heads read (a + b) * lod_weights.  Base field: the (detached) colour features.
        rows (int64 [K], inference only): evaluate packed samples `rows` only -> [K, F] tensors."""
        a = feats.detach() if (self.sem_detach and self.inst_detach) else feats
        return (a if rows is None else a.index_select(0, rows)), None

    def fused_panoptic_ok(self, channels):
        """Can the semantic / instance heads be fused with their compositing?  Tensor-core mode: csrc/decoder_tc_fused.cu
        (forward + backward).  Exact-FP32 mode: only when nothing is differentiated (inference; csrc/decoder_tiled.cu)."""
        want = [c for c in ('semantics', 'inst_embedding') if c in channels]
        if not want:
            return False
        if not self._use_tc() and (torch.is_grad_enabled() or not ops.TILED_F32):
            return False
        return self._fused_heads_unsupported() is None

    def _fused_heads_unsupported(self):
        """None when the fused-head kernels (csrc/decoder_tc_fused.cu, csrc/decoder_tiled.cu) serve this field's semantic /
        instance heads, else the reason they do not."""
        if self.sem_sigmoid or self.sem_normalize or self.inst_sigmoid or self.inst_normalize or self.inst_direct_pos:
            return "sigmoid / normalize / inst_direct_pos head options"
        if not (self.sem_detach and self.inst_detach):
            return "non-detached panoptic heads (sem_detach / inst_detach False)"
        if self.multiscale_type != 'cat':
            return f"multiscale_type '{self.multiscale_type}'"
        if self.effective_feature_dim > 48 or self.effective_feature_dim % 4:
            return f"feature width {self.effective_feature_dim} (needs <= 48 and a multiple of 4)"
        if self.num_classes > 16 or self.num_instances > 208:
            return f"{self.num_classes} classes / {self.num_instances} instances (at most 16 / 208)"
        if self.panoptic_features_type not in (None, 'delta', 'separate', 'appearance'):
            return f"panoptic_features_type '{self.panoptic_features_type}'"
        return None

    def _pan_src(self):
        """Which features feed the panoptic heads in the fused kernels."""
        if not hasattr(self, 'delta_grid'):
            return 'appearance'
        return {None: 'delta', 'delta': 'delta', 'separate': 'separate', 'appearance': 'appearance'}.get(self.panoptic_features_type)

    def fused_trace_cfg(self, channels, rays, num_steps, bg_color, raymarch_type='ray', max_travel=None):
        """Configuration for ops.FusedTraceFn (sync-free training trace), or None when this field / request is not
        covered by it ('ray' marching on PermutoGrid fields with the reference decoder shapes, tensor-core mode)."""
        from ..grids import PermutoGrid, HashGridTinyCudaNN, HashGridTorch
        pan = [c for c in ('semantics', 'inst_embedding') if c in channels]
        if not self._use_tc() or not hasattr(self.grid, 'embedder'):
            return None
        if isinstance(self.grid, PermutoGrid):
            kind = 'permuto'
        elif isinstance(self.grid, (HashGridTinyCudaNN, HashGridTorch)):
            kind = 'hash'
        else:
            return None
        if pan and not self.fused_panoptic_ok(channels):
            return None
        if self.multiscale_type != 'cat' or self.effective_feature_dim > 48 or self.effective_feature_dim % 4:
            return None
        src = self._pan_src() if pan else 'none'
        if src is None:
            return None
        dev = rays.origins.device
        blas = self.grid.blas.to(dev)

        def enc(e):
            if kind == 'permuto':
                return (e.scale_factor, e.random_shift_per_level, e.anneal_window, e.capacity, e.nr_levels, e.n_agg_levels)
            if isinstance(self.grid, HashGridTinyCudaNN):      # flavour 0; autocast casts the coordinates to half (:36)
                return (0, e.level_scale, e.level_res, e.level_offset, e.level_size, e.n_levels, e.round_half, e.n_agg_levels, True)
            return (1, e.level_res, None, e.level_offset, e.level_size, e.n_levels, False, e.n_agg_levels, False)

        seed = blas.jitter_seed
        if not blas.fixed_jitter:
            blas.jitter_seed = (blas.jitter_seed + 1) & 0x7FFFFFFF
        dmin = float(rays.dist_min) if not torch.is_tensor(rays.dist_min) else float(rays.dist_min.flatten()[0])
        dmax = float(rays.dist_max) if not torch.is_tensor(rays.dist_max) else float(rays.dist_max.flatten()[0])
        return dict(octree=blas.octree, prefix=blas.prefix, level=self.grid.blas_level, S=int(num_steps), near=dmin, far=dmax,
                    march=raymarch_type, max_travel=max_travel,
                    bits=blas.level_bits(self.grid.blas_level) if self.grid.blas_level >= 2 else None,
                    seed=seed, fixed_jitter=bool(blas.fixed_jitter),
                    # the device-resident seed is for CUDA-graph capture / replay only (graph.GraphedStep); eager traces follow
                    # blas.jitter_seed like the step-by-step path
                    seed_dev=getattr(blas, 'seed_tensor', None) if getattr(blas, 'graph_seed_active', False) else None,
                    bg_white=(bg_color == 'white'), pos_half=torch.is_autocast_enabled(),
                    lodw=self._lodw(dev), grid_kind=kind, grid=enc(self.grid.embedder),
                    dgrid=enc(self.delta_grid.embedder) if src in ('delta', 'separate') else None, pan_src=src,
                    want_rgb='rgb' in channels, want_depth='depth' in channels,
                    Cs=self.num_classes if 'semantics' in channels else 0,
                    Ci=self.num_instances if 'inst_embedding' in channels else 0,
                    sem_softmax=bool(self.sem_softmax), inst_softmax=bool(self.inst_softmax),
                    inst_temperature=float(getattr(self, 'inst_soft_temperature', 0.0)))

    def fused_trace_tensors(self):
        """(color table, delta table | None, 20 decoder tensors) in the order ops.FusedTraceFn expects."""
        wts = (_decoder_tensors(self.decoder_density, 1) + _decoder_tensors(self.decoder_color, 2)
               + _decoder_tensors(self.decoder_semantics, 1) + _decoder_tensors(self.decoder_inst, 2))
        def table(e):
            for name in ('lattice_values', 'params', 'embeddings_weight'):      # permutohedral / tcnn / HashNeRF
                if hasattr(e, name):
                    return getattr(e, name)
            raise AttributeError("unknown grid embedder")
        dt = table(self.delta_grid.embedder) if hasattr(self, 'delta_grid') else None
        return table(self.grid.embedder), dt, wts

    def trace_composited(self, coords, ray_d, ridx_rows, deltas, depths, offsets, num_rays, channels, bg_white, lod_idx=None):
        """Decode + composite in one pass: per-ray dict(alpha, hit, rgb, depth, semantics, inst_embedding).
        The panoptic probabilities are composited inside the decoder kernel and never materialised.
        Under torch.no_grad() (rendering / validation) the density pass runs first and everything downstream of the integration
        weights -- colour decoder, delta-grid lookup, panoptic heads -- runs on the samples with a non-zero weight only
        (ops.LIVE_COMPACT_FRAC; exact: a zero weight multiplies whatever the skipped decoders would have produced)."""
        if lod_idx is None:
            lod_idx = len(self.grid.active_lods) - 1
        batch, num_samples, _ = coords.shape
        feats = self._encode(self.grid, coords, lod_idx)
        want_rgb = 'rgb' in channels
        want_sem, want_inst = 'semantics' in channels, 'inst_embedding' in channels
        rows = None
        probe = not torch.is_grad_enabled() and ops.LIVE_COMPACT_FRAC > 0.0 and feats.shape[0] > 0 and (want_rgb or want_sem or want_inst)
        if probe and getattr(self, '_dense_chunks_left', 0) > 0:
            self._dense_chunks_left -= 1          # the last probe found (almost) every sample live: skip the density-first pass for a while
            probe = False
        if probe:
            sigma, _ = self._dc(feats, ray_d, num_samples, False)
            alpha, hit, _, dep_o, _, _, w = ops.composite(sigma, deltas, depths if 'depth' in channels else None, None,
                                                           None, None, offsets, bg_white)
            wf = w.reshape(-1)
            live = torch.nonzero(wf > ops.LIVE_WEIGHT_EPS).reshape(-1)      # host sync on its size (this path already has one per march)
            self.last_live_fraction = live.numel() / wf.numel()
            if live.numel() < ops.LIVE_COMPACT_FRAC * wf.numel():
                rows = live
            else:
                self._dense_chunks_left = 63
        if rows is not None:
            w = wf.index_select(0, rows)
            ridx_rows = ridx_rows.index_select(0, rows)
            rgb_o = None
            if want_rgb:
                rd = ray_d.index_select(0, rows // num_samples) if num_samples > 1 else ray_d.index_select(0, rows)
                _, rgb = self._dc(feats.index_select(0, rows), rd, 1, True)
                acc = ops.SumReduceFn.apply(rgb * w.unsqueeze(-1), ops.ray_offsets(ridx_rows, num_rays))
                rgb_o = (1.0 - alpha) + alpha * acc if bg_white else alpha * acc          # alpha on top, like ops.composite
        else:
            sigma, rgb = self._dc(feats, ray_d, num_samples, want_rgb)
            alpha, hit, rgb_o, dep_o, _, _, w = ops.composite(sigma, deltas, depths if 'depth' in channels else None, rgb,
                                                               None, None, offsets, bg_white)
        out = {'alpha': alpha, 'hit': hit, 'density': sigma}
        if want_rgb:
            out['rgb'] = rgb_o
        if 'depth' in channels:
            out['depth'] = dep_o
        if want_sem or want_inst:
            a, b = self._panoptic_inputs(feats, coords, lod_idx, rows) if rows is not None else self._panoptic_inputs(feats, coords, lod_idx)
            wts = _decoder_tensors(self.decoder_semantics, 1) + _decoder_tensors(self.decoder_inst, 2)
            lodw = self._lodw(feats.device)
            fused = ops.PanCompositeFn.apply if self._use_tc() else ops.pan_composite_f32
            sem_o, inst_o = fused(
                a, b, lodw, w, alpha.detach(), ridx_rows, num_rays, self.num_classes if want_sem else 0,
                self.num_instances if want_inst else 0, bool(self.sem_softmax), bool(self.inst_softmax),
                float(getattr(self, 'inst_soft_temperature', 0.0)), *wts)
            if want_sem:
                out['semantics'] = sem_o
            if want_inst:
                out['inst_embedding'] = inst_o
        return out

    def rgb_semantics(self, coords, ray_d, compute_channels, pidx=None, lod_idx=None):
        """coords [batch, num_samples, 3], ray_d [batch, 3] -> dict with density [batch,S,1], rgb [batch,S,3],
        semantics [batch*S, C], inst_embedding [batch*S, C] (reference shapes, pc_nerf/panoptic_nef.py:253-363)."""
        out_dict = {}
        if not compute_channels:
            return out_dict
        if lod_idx is None:
            lod_idx = len(self.grid.active_lods) - 1
        batch, num_samples, _ = coords.shape
        feats = self._encode(self.grid, coords, lod_idx)
        if any(c in compute_channels for c in ['density', 'rgb']):
            sigma, rgb = self._dc(feats, ray_d, num_samples, 'rgb' in compute_channels)
            if 'density' in compute_channels:
                out_dict['density'] = sigma.reshape(batch, num_samples, 1)
            if 'rgb' in compute_channels:
                out_dict['rgb'] = rgb.reshape(batch, num_samples, 3)
        want_sem, want_inst = 'semantics' in compute_channels, 'inst_embedding' in compute_channels
        if want_inst and self.inst_direct_pos:
            raise NotImplementedError("inst_direct_pos is not served by the fused decoders")
        if want_sem and want_inst and self.sem_detach == self.inst_detach:
            x = feats.detach() if self.sem_detach else feats
            out_dict['semantics'], out_dict['inst_embedding'] = self._pan(x, None, True, True)
        else:
            if want_sem:
                out_dict['semantics'], _ = self._pan(feats.detach() if self.sem_detach else feats, None, True, False)
            if want_inst:
                _, out_dict['inst_embedding'] = self._pan(feats.detach() if self.inst_detach else feats, None, False, True)
        return out_dict
