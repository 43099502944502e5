"""CPU: a neural field its owner drops is freed at once, with its parameters, and not left to the cycle collector (its registered
forward functions must not make it reference itself)."""
import gc
import weakref

import pytest

from tests.util import load_golden, build_cuda_nef


@pytest.mark.parametrize("name", ["trace_delta_permuto_ray", "trace_nef_tcnn_ray", "trace_dd_permuto_ray"])
def test_dropped_field_is_freed_by_reference_counting(name):
    nef = build_cuda_nef(load_golden(name), "cpu")
    field, param = weakref.ref(nef), weakref.ref(next(nef.parameters()))
    channels = nef.get_supported_channels()
    assert {"density", "rgb", "semantics", "inst_embedding"} <= channels
    gc.disable()
    try:
        del nef
        assert field() is None and param() is None
    finally:
        gc.enable()

