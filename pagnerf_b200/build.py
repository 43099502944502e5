"""In-tree build of the C-ABI CUDA library (sm_100a only).

    python -m pagnerf_b200.build            # -> pagnerf_b200/csrc/libpagnerf_b200.so

nvcc cross-compiles without a GPU; the .so is git-ignored but travels with the repo snapshot.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libpagnerf_b200.so")
SOURCES = ["octree.cu", "permuto.cu", "hashgrid.cu", "composite.cu", "pose.cu", "adam.cu", "allreduce.cu", "loss.cu", "metrics.cu", "decoder.cu", "decoder_tiled.cu", "decoder_tc.cu", "decoder_tc_fused.cu", "tc_test.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


LAST_BUILD = None


def build(force=False, verbose=False, extra_flags=(), tag=""):
    """tag / extra_flags: an instrumented variant (e.g. tag='_dbg', extra_flags=['-DPAG_PHASE_TIMING']) built beside the
    product library as libpagnerf_b200<tag>.so; select it at load time with PAGNERF_B200_LIB=<path>."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    force = force or os.environ.get("PAGNERF_FORCE_BUILD") == "1"
    lib = LIB.replace(".so", f"{tag}.so")
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(os.path.dirname(HERE), "include", "pagnerf_b200.h"))
    hdrs = [h for h in hdrs if os.path.exists(h)]
    objs = []
    procs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(CSRC, src.replace(".cu", f"{tag}.o"))
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            cmd = [nvcc, *NVCC_FLAGS, *extra_flags, "-c", s, "-o", o] + (["-Xptxas", "-v"] if verbose else [])
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            print(f"--- {src} ---\n{out}")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    linked = bool(force or procs or _stale(lib, objs))
    if linked:
        subprocess.check_call([nvcc, "-shared", "-o", lib, *objs, "-gencode", "arch=compute_100a,code=sm_100a"])
    # what this call did, for the record (the driver's GPU box reuses the .so that travelled with the snapshot unless a source is
    # newer; PAGNERF_FORCE_BUILD=1 or build(force=True) compiles everything from source there)
    global LAST_BUILD
    LAST_BUILD = {"library": lib, "compiled": [src for src, _ in procs], "reused": [s_ for s_ in SOURCES if s_ not in [x for x, _ in procs]],
                  "linked": linked, "forced": bool(force)}
    try:
        import json
        import time
        LAST_BUILD["when"] = time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime())
        with open(os.path.join(CSRC, "build_info.json"), "w") as f:
            json.dump(LAST_BUILD, f, indent=1)
    except OSError:
        pass
    return lib


if __name__ == "__main__":
    if "--phase-timing" in sys.argv:
        print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, extra_flags=["-DPAG_PHASE_TIMING"], tag="_dbg"))
    else:
        print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
