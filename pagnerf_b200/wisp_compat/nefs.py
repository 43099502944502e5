"""wisp.models.nefs.BaseNeuralField stand-in: attribute storage + channel dispatch.

The reference's fields (pc_nerf/panoptic_nef.py:20,70,239-251) rely on this base to (1) store the
constructor arguments as attributes and the rest in `self.kwargs`, (2) call
init_grid / init_embedder / init_decoder / register_forward_functions, and (3) dispatch
`forward(channels, **kwargs)` to the registered function(s), returning a tensor for a str request,
a list for a list, a dict for a set / None.
"""
import inspect

import torch.nn as nn


class _FieldMethod:
    """A forward function that is a method of the field, kept as its plain function and bound to the field again at each call.  The
    bound method would make the field reference itself: a field its owner drops (and its parameters on the device) would then live
    on until the cycle collector runs, which may be at any later allocation."""

    def __init__(self, func):
        self.func = func


class BaseNeuralField(nn.Module):
    def __init__(self, grid_type='OctreeGrid', interpolation_type='linear', multiscale_type='none',
                 as_type='octree', raymarch_type='voxel', decoder_type='none', embedder_type='none',
                 activation_type='relu', layer_type='none', base_lod=2, num_lods=1, sample_tex=False,
                 dilate=None, feature_dim=16, hidden_dim=128, pos_multires=10, view_multires=4,
                 num_layers=1, position_input=False, **kwargs):
        super().__init__()
        self.grid_type = grid_type
        self.interpolation_type = interpolation_type
        self.raymarch_type = raymarch_type
        self.embedder_type = embedder_type
        self.activation_type = activation_type
        self.layer_type = layer_type
        self.decoder_type = decoder_type
        self.multiscale_type = multiscale_type
        self.base_lod = base_lod
        self.num_lods = num_lods
        self.sample_tex = sample_tex
        self.dilate = dilate
        self.feature_dim = feature_dim
        self.hidden_dim = hidden_dim
        self.pos_multires = pos_multires
        self.view_multires = view_multires
        self.num_layers = num_layers
        self.position_input = position_input
        self.kwargs = kwargs

        self.grid = None
        self.decoder = None
        self.init_grid()
        self.init_embedder()
        self.init_decoder()
        self._forward_functions = {}
        self.register_forward_functions()
        self.supported_channels = set(c for cs in self._forward_functions.values() for c in cs)

    # -- hooks the subclasses override -------------------------------------------------------
    def init_embedder(self):
        return

    def init_decoder(self):
        return

    def init_grid(self):
        raise NotImplementedError

    def register_forward_functions(self):
        raise NotImplementedError

    def get_nef_type(self):
        return 'nef'

    def prune(self):
        return

    # -- dispatch ---------------------------------------------------------------------------
    def _register_forward_function(self, fn, channels):
        if isinstance(channels, str):
            channels = [channels]
        if inspect.ismethod(fn) and fn.__self__ is self:
            fn = _FieldMethod(fn.__func__)
        self._forward_functions[fn] = set(channels)

    def get_supported_channels(self):
        return self.supported_channels

    @property
    def device(self):
        return next(self.parameters()).device

    def forward(self, channels=None, **kwargs):
        if not (isinstance(channels, (str, list, set)) or channels is None):
            raise Exception(f"Channels type invalid, got {type(channels)}."
                            "Make sure your arguments for the nef are provided as keyword arguments.")
        if channels is None:
            requested = self.get_supported_channels()
        elif isinstance(channels, str):
            requested = {channels}
        else:
            requested = set(channels)
        unsupported = requested - self.get_supported_channels()
        if unsupported:
            raise Exception(f"Channels {unsupported} are not supported in {type(self)}")

        return_dict = {}
        for fn, out_channels in self._forward_functions.items():
            supported = out_channels & requested
            if not supported:
                continue
            if isinstance(fn, _FieldMethod):
                fn = fn.func.__get__(self, type(self))
            argspec = inspect.getfullargspec(fn)
            ndef = len(argspec.defaults) if argspec.defaults else 0
            required = argspec.args[:len(argspec.args) - ndef][1:]
            optional = argspec.args[len(argspec.args) - ndef:]
            input_args = {}
            for a in required:
                if a not in kwargs:
                    raise Exception(f"Argument {a} not found as input to in {type(self)}.{fn.__name__}()")
                input_args[a] = kwargs[a]
            for a in optional:
                if a in kwargs:
                    input_args[a] = kwargs[a]
            output = fn(**input_args)
            for c in supported:
                return_dict[c] = output[c]

        if isinstance(channels, str):
            return return_dict.get(channels)
        if isinstance(channels, list):
            return [return_dict[c] for c in channels]
        return return_dict
