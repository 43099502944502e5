"""ctypes binding of libpagnerf_b200.so (the C ABI declared in include/pagnerf_b200.h).

The prototypes are parsed from the header so the binding cannot drift from the declared ABI.
There is NO fallback: if the library is missing or a symbol is absent, loading raises.
"""
import ctypes
import os
import re
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PAGNERF_B200_LIB") or os.path.join(_HERE, "csrc", "libpagnerf_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "pagnerf_b200.h")

_lock = threading.Lock()
_lib = None
_protos = None

# kernels launched per entry point (for bench.py's gpu_launches accounting)
KERNELS_PER_CALL = {
    "pag_march_ray_count": 2, "pag_march_ray_bits_count": 2, "pag_compact_count": 2, "pag_raytrace_count": 2, "pag_voxel_filter_count": 2, "pag_voxel_filter_count_staged": 2, "pag_raytrace_stage": 4, "pag_octree_from_mask": 12, "pag_adam_step": 2, "pag_pan_composite_bwd_tc": 2, "pag_decode_dc_bwd_tc_dyn": 2,
    "pag_pq_update": 3,
}
launch_count = 0


def parse_header(path=HEADER_PATH):
    """-> {name: [ctypes argtypes]} for every `int pag_*(...)` prototype in the header."""
    src = open(path).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    protos = {}
    for m in re.finditer(r"\bint\s+(pag_\w+)\s*\(([^;]*?)\)\s*;", src, flags=re.S):
        name, args = m.group(1), m.group(2)
        types = []
        for a in args.split(","):
            a = a.strip()
            if "*" in a:
                types.append(ctypes.c_void_p)
            elif a.startswith("int64_t"):
                types.append(ctypes.c_int64)
            elif a.startswith("uint32_t"):
                types.append(ctypes.c_uint32)
            elif a.startswith("float"):
                types.append(ctypes.c_float)
            elif a.startswith("int"):
                types.append(ctypes.c_int)
            else:
                raise ValueError(f"unparsed argument '{a}' in {name}")
        protos[name] = types
    return protos


def load():
    global _lib, _protos
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"pagnerf_b200: CUDA library not built ({LIB_PATH} missing). Run `python -m pagnerf_b200.build` "
                "(or __graft_entry__.build()). There is no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        _protos = parse_header()
        for name, argtypes in _protos.items():
            fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
            fn.argtypes = argtypes
            fn.restype = ctypes.c_int
        _lib = lib
        return _lib


def exported_symbols():
    load()
    return sorted(_protos.keys())


def query_i64(name, *args):
    """Host-side size query `int name(args..., int64_t* out)` (no stream, no launch) -> int."""
    out = ctypes.c_int64(0)
    rc = getattr(load(), name)(*args, ctypes.byref(out))
    if rc != 0:
        raise RuntimeError(f"pagnerf_b200: {name} -> {rc}")
    return int(out.value)


def ptr(t):
    """device pointer of a tensor (None -> NULL); asserts contiguity."""
    if t is None:
        return None
    assert t.is_contiguous(), "pagnerf_b200: non-contiguous tensor passed to the C ABI"
    return t.data_ptr()


def ptr_array(tensors):
    """host array of device pointers (for `const float* const*` parameters)."""
    arr = (ctypes.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = ptr(t)
    return arr


def stream():
    return torch.cuda.current_stream().cuda_stream


_timing = False
_events = []   # (name, start_event, end_event)


def timing_reset(enable):
    """Enable / disable per-entry-point CUDA-event timing (bench.py's live roofline measurement)."""
    global _timing, _events
    _timing, _events = bool(enable), []


def timing_report():
    """-> {entry point: {ms_per_launch, launches, ms_total}}; synchronises the device."""
    torch.cuda.synchronize()
    agg = {}
    for name, e0, e1 in _events:
        a = agg.setdefault(name, {"ms_total": 0.0, "launches": 0})
        a["ms_total"] += e0.elapsed_time(e1)
        a["launches"] += 1
    for a in agg.values():
        a["ms_per_launch"] = a["ms_total"] / a["launches"]
    return agg


def call(name, *args):
    """Invoke an entry point on torch's current stream; raises on any non-zero return code."""
    global launch_count
    lib = load()
    if _timing:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = getattr(lib, name)(*args, stream())
        e1.record()
        _events.append((name, e0, e1))
    else:
        rc = getattr(lib, name)(*args, stream())
    if rc != 0:
        kind = {-1: "invalid argument", -2: "unsupported shape/config"}.get(rc, f"cudaError {rc}")
        raise RuntimeError(f"pagnerf_b200.{name} failed: {kind}")
    launch_count += KERNELS_PER_CALL.get(name, 1)
