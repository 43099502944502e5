"""PanopticDDensityNeF: PanopticNeF + delta grid + a delta-DENSITY head; the panoptic channels are integrated with their own
density `panoptic_density = relu(density_pre.detach() + delta_density)` by PanopticDDensityPackedRFTracer
(reference pc_nerf/panoptic_dd_nef.py:21-275; decoder :41-58, grid :60-64, rgb_semantics :130-275).

SURVEY 8(f) rank 2 (used by 7 of the 13 bup20 configs).  Built from the existing kernels on the step-by-step path:
  * density / colour / semantic / instance heads: csrc/decoder*.cu as in PanopticDeltaNeF;
  * the PRE-activation colour density (the reference reads `density_feats[..., 0:1]` before the ReLU, detached) comes from
    the semantic-head kernel run on the density decoder's weights (feat -> 64 -> 16 raw outputs, no gradient needed);
  * the delta-density decoder is a BasicDecoder with activation 'none' (wisp Identity): two Linear layers without a
    nonlinearity are one linear map, collapsed on the host (autograd carries the gradient to both layers) and applied
    by csrc/decoder.cu linear_head_*.
"""
import copy

import torch

from .. import ops
from ..wisp_compat import BasicDecoder, get_activation_class, get_layer_class
from .panoptic_nef import PanopticNeF, _decoder_tensors


class PanopticDDensityNeF(PanopticNeF):
    def __init__(self, delta_num_layers: int = 1, delta_hidden_dim: int = 64, separate_sem_grid: bool = False,
                 inst_soft_temperature: float = 0.0, **kwargs):
        self.delta_num_layers = delta_num_layers
        self.delta_hidden_dim = delta_hidden_dim
        self.separate_sem_grid = separate_sem_grid
        self.inst_soft_temperature = inst_soft_temperature
        super().__init__(**kwargs)

    def init_decoder(self):
        super().init_decoder()
        if self.delta_num_layers == 0:
            self.delta_hidden_dim = self.input_dim_density
        self.decoder_delta_density = BasicDecoder(input_dim=self.input_dim_density, output_dim=1,
                                                  activation=get_activation_class('none'), bias=True,
                                                  layer=get_layer_class(self.layer_type), num_layers=self.delta_num_layers,
                                                  hidden_dim=self.delta_hidden_dim, skip=[])

    def init_grid(self):
        super().init_grid()
        self.delta_grid = copy.deepcopy(self.grid)
        if self.grid_type == "PermutoGrid":
            self.delta_grid.set_capacity(self.kwargs['delta_capacity_log_2'])

    def get_nef_type(self):
        return 'delta_panoptic_nef'

    def _prune_grids(self):
        return [self.grid, self.delta_grid]

    def register_forward_functions(self):
        self._register_forward_function(self.rgb_semantics, ["density", "rgb", "delta_density", "panoptic_density",
                                                             "semantics", "inst_embedding"])

    def fused_panoptic_ok(self, channels):     # the modular fused kernels composite with the detached colour density: not this model
        return False

    def fused_trace_cfg(self, channels, rays, num_steps, bg_color, raymarch_type='ray', max_travel=None, dd=False):
        """Sync-free fused trace with the panoptic density stream (ops.FusedTraceFn, cfg['dd']).  Only for the DD tracer (dd=True):
        PanopticPackedRFTracer would composite the panoptic channels with the detached colour density."""
        if not dd or self.separate_sem_grid or not (self.sem_softmax and self.inst_softmax):
            return None
        if self.sem_sigmoid or self.sem_normalize or self.inst_sigmoid or self.inst_normalize:
            return None
        fused_ok, self.fused_panoptic_ok = self.fused_panoptic_ok, lambda channels: True    # shapes are checked by the base method
        try:
            ok_shapes = (self.effective_feature_dim <= 48 and self.effective_feature_dim % 4 == 0 and self.num_classes <= 16
                         and self.num_instances <= 208)
            cfg = super().fused_trace_cfg(channels, rays, num_steps, bg_color, raymarch_type, max_travel) if ok_shapes else None
        finally:
            del self.fused_panoptic_ok
        if cfg is not None:
            cfg['dd'] = True
        return cfg

    def _pan_src(self):
        return 'delta'

    def _panoptic_inputs(self, feats, coords, lod_idx, rows=None):
        """(a, b) of rgb_semantics (:229): (feats.detach(), delta), or (delta, None) with separate_sem_grid.  rows (int64 [K],
        inference only): evaluate packed samples `rows` only -- the delta grid is looked up for those only."""
        a = feats.detach()
        if rows is not None:
            a = a.index_select(0, rows)
            coords = coords.reshape(-1, 1, 3).index_select(0, rows)
        dfe = self._encode(self.delta_grid, coords.detach(), lod_idx)
        return (a, dfe) if not self.separate_sem_grid else (dfe, None)

    def fused_trace_tensors(self):
        table, dtable, wts = super().fused_trace_tensors()
        dec = self.decoder_delta_density          # Linear(+Identity) layers collapsed into one map (autograd reaches both layers)
        w, bias = dec.lout.weight, dec.lout.bias
        for l in reversed(list(dec.layers)):
            bias = bias + w @ l.bias
            w = w @ l.weight
        return table, dtable, list(wts) + [w, bias]

    def _density_pre(self, feats):
        """density_feats[..., 0:1] BEFORE the ReLU, detached (:243): the semantic-head kernel on the density decoder's weights."""
        wd = _decoder_tensors(self.decoder_density, 1)
        with torch.no_grad():
            w = [t.detach() for t in wd] + [wd[0].detach(), wd[1].detach(), wd[0].detach(), wd[1].detach(), wd[2].detach(), wd[3].detach()]
            y16, _ = ops.DecodePanFn.apply(feats.detach(), None, self._lodw(feats.device), 16, 0, False, False, 0.0, False, *w)
        return y16[:, 0:1]

    def _delta_density(self, a, b):
        """decoder_delta_density on (a + b) * lod_weights: Linear(+Identity) layers collapsed into one map."""
        dec = self.decoder_delta_density
        w, bias = dec.lout.weight, dec.lout.bias                      # [1, h], [1]
        for l in reversed(list(dec.layers)):                          # y = lout(l_n(... l_1(x)))
            bias = bias + w @ l.bias
            w = w @ l.weight
        return ops.LinearHeadFn.apply(a, b, self._lodw(a.device), w, bias)

    def rgb_semantics(self, coords, ray_d, compute_channels, pidx=None, lod_idx=None):
        out_dict = {}
        if not compute_channels:
            return out_dict
        if lod_idx is None:
            lod_idx = len(self.grid.active_lods) - 1
        batch, num_samples, _ = coords.shape
        if self.position_input:
            raise NotImplementedError
        feats = self._encode(self.grid, coords, lod_idx)
        need_density = any(c in compute_channels for c in ('density', 'rgb')) or \
            ('panoptic_density' in compute_channels and not self.separate_sem_grid)          # :187-188
        if need_density:
            sigma, rgb = self._dc(feats, ray_d, num_samples, 'rgb' in compute_channels)
            if 'density' in compute_channels:
                out_dict['density'] = sigma.reshape(batch, num_samples, 1)
            if 'rgb' in compute_channels:
                out_dict['rgb'] = rgb.reshape(batch, num_samples, 3)
        pan = [c for c in ('delta_density', 'panoptic_density', 'semantics', 'inst_embedding') if c in compute_channels]
        if pan:
            dfe = self._encode(self.delta_grid, coords.detach(), lod_idx)                     # :221-222
            a, b = (feats.detach(), dfe) if not self.separate_sem_grid else (dfe, None)      # :229
        if 'delta_density' in compute_channels or 'panoptic_density' in compute_channels:
            dd = self._delta_density(a, b).reshape(batch, num_samples, 1)
            if 'delta_density' in compute_channels:
                out_dict['delta_density'] = dd
            if 'panoptic_density' in compute_channels:
                pre = self._density_pre(feats).reshape(batch, num_samples, 1) if not self.separate_sem_grid else 0.0
                out_dict['panoptic_density'] = torch.relu(pre + dd)                            # :243-245
        want_sem, want_inst = 'semantics' in compute_channels, 'inst_embedding' in compute_channels
        if want_sem or want_inst:
            sem, inst = self._pan(a, b, want_sem, want_inst, self.inst_soft_temperature)
            if want_sem:
                out_dict['semantics'] = sem
            if want_inst:
                out_dict['inst_embedding'] = inst
        return out_dict
