"""ctypes binding of csrc/libkgx.so (the C ABI declared in include/kgx.h).  Fails loudly when the CUDA
library is missing or does not export a declared symbol -- there is no fallback path."""
import ctypes
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_PATH = os.environ.get("KGX_LIB_OVERRIDE") or os.path.join(CSRC, "libkgx.so")   # override: A/B builds in scripts/ experiments
HOSTTEST_PATH = os.path.join(CSRC, "libkgx_hosttest.so")
INGEST_PATH = os.path.join(CSRC, "libkgx_ingest.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


class Item(ctypes.Structure):
    """kgx_item: the 56-byte DP record (GPUEngine.h:31, GPUMath.h:173-188)."""
    _fields_ = [("x", ctypes.c_uint64 * 4), ("d", ctypes.c_uint64 * 2), ("kidx", ctypes.c_uint64)]


_u64p = ctypes.POINTER(ctypes.c_uint64)
_SIGS = {
    "kgx_device_count": (ctypes.c_int, []),
    "kgx_grid_default": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
    "kgx_device_info": (ctypes.c_int, [ctypes.c_int, ctypes.c_char_p, ctypes.c_int]),
    "kgx_create": (ctypes.c_void_p, [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_uint32]),
    "kgx_create_ex": (ctypes.c_void_p, [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_uint32, ctypes.c_int, ctypes.c_int]),
    "kgx_kernel_kind": (ctypes.c_int, [ctypes.c_void_p]),
    "kgx_destroy": (None, [ctypes.c_void_p]),
    "kgx_last_error": (ctypes.c_char_p, [ctypes.c_void_p]),
    "kgx_num_kangaroos": (ctypes.c_uint64, [ctypes.c_void_p]),
    "kgx_memory_bytes": (ctypes.c_uint64, [ctypes.c_void_p]),
    "kgx_set_symmetry": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "kgx_get_symmetry": (ctypes.c_int, [ctypes.c_void_p]),
    "kgx_set_params": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, _u64p, _u64p, _u64p]),
    "kgx_upload": (ctypes.c_int, [ctypes.c_void_p, _u64p, _u64p, _u64p]),
    "kgx_download": (ctypes.c_int, [ctypes.c_void_p, _u64p, _u64p, _u64p]),
    "kgx_patch": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_uint64, _u64p, _u64p, _u64p]),
    "kgx_create_herd": (ctypes.c_int, [ctypes.c_void_p, _u64p, _u64p, _u64p, _u64p, ctypes.c_int]),
    "kgx_snapshot_begin": (ctypes.c_int, [ctypes.c_void_p]),
    "kgx_snapshot_read": (ctypes.c_int, [ctypes.c_void_p, _u64p, _u64p, _u64p]),
    "kgx_launch_async": (ctypes.c_int, [ctypes.c_void_p]),
    "kgx_collect": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(Item), ctypes.c_uint32, ctypes.POINTER(ctypes.c_uint32),
                                   ctypes.POINTER(ctypes.c_uint32), ctypes.c_int, ctypes.c_int]),
    "kgx_sync": (ctypes.c_int, [ctypes.c_void_p]),
    "kgx_dp_slab_device": (ctypes.c_void_p, [ctypes.c_void_p]),
    "kgx_convert_dps": (ctypes.c_int, [ctypes.c_void_p, _u64p, ctypes.POINTER(ctypes.c_void_p)]),
    "kgx_max_found": (ctypes.c_uint32, [ctypes.c_void_p]),
    "kgx_last_launch_ms": (ctypes.c_float, [ctypes.c_void_p]),
    "kgx_set_jumps_per_launch": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "kgx_kernel_launches": (ctypes.c_uint64, [ctypes.c_void_p]),
    "kgx_debug_prof": (ctypes.c_int, [ctypes.c_void_p, _u64p]),
    "kgx_test_field": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, _u64p, _u64p, _u64p]),
    "kgx_bench_raw": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_float),
                                     ctypes.POINTER(ctypes.c_double)]),
}
EXPORTED_SYMBOLS = sorted(_SIGS)

_lib = None


def build_library(verbose=False):
    """Compile every CUDA source for sm_100a into csrc/libkgx.so (nvcc cross-compiles without a GPU), the rank-0 DP table
    csrc/libkgx_ingest.so and the host-only unit-test helper csrc/libkgx_hosttest.so."""
    src = os.path.join(CSRC, "kgx_engine.cu")
    cmd = ["nvcc"] + NVCC_FLAGS + ["-o", LIB_PATH, src]
    if verbose:
        cmd += ["-Xptxas", "-v"]
    subprocess.check_call(cmd, cwd=CSRC)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-o", INGEST_PATH, os.path.join(CSRC, "kgx_ingest.cpp"), "-lpthread"])
    subprocess.check_call(["g++", "-O2", "-frounding-math", "-ffp-contract=off", "-fPIC", "-shared", "-o", HOSTTEST_PATH, os.path.join(CSRC, "kgx_hosttest.cpp")])
    return LIB_PATH


def _needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    for f in os.listdir(CSRC):
        if f.endswith((".cu", ".cuh", ".h")) and os.path.getmtime(os.path.join(CSRC, f)) > t:
            return True
    return os.path.getmtime(os.path.join(HERE, "..", "include", "kgx.h")) > t


def load_library(rebuild_if_stale=True):
    """Load libkgx.so and type every entry point of include/kgx.h.  Raises (never falls back) when the library
    cannot be built/loaded or a declared symbol is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if rebuild_if_stale and _needs_build():
        build_library()
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("kangaroo_b200: CUDA library %s is missing (run __graft_entry__.build())" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGS.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise RuntimeError("kangaroo_b200: %s does not export %s" % (LIB_PATH, name)) from e
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
