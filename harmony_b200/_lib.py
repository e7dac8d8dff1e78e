"""Loader / builder of libharmony_b200.so (the C ABI declared in include/harmony_b200.h).

There is no CPU fallback: if the shared library is missing or no CUDA device is present the
constructors raise.  The library is built IN-TREE (harmony_b200/libharmony_b200.so) with
``nvcc -gencode arch=compute_100a,code=sm_100a`` by ``build()`` / ``__graft_entry__.build()``.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(_HERE)
SO_PATH = os.path.join(_HERE, "libharmony_b200.so")
SOURCES = [os.path.join(_HERE, "csrc", f) for f in ("harmony_b200.cu", "kernels.cuh", "common.cuh", "update_kernel.cuh", "update_kernel4.cuh", "update_kernel5.cuh",
                                                     "umma.cuh", "assign_tc3.cuh", "logits_tc.cuh", "stats_tc3.cuh", "apply_tc3.cuh",
                                                     "setup_device.cuh")]
HEADER = os.path.join(ROOT, "include", "harmony_b200.h")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-shared",
              "-Xcompiler", "-fPIC"]

_LIB = None


def needs_build():
    if not os.path.exists(SO_PATH):
        return True
    t = os.path.getmtime(SO_PATH)
    return any(os.path.exists(s) and os.path.getmtime(s) > t for s in SOURCES + [HEADER])


def build(force=False, verbose=False):
    """Compile the CUDA library for sm_100a (cross-compiles without a GPU)."""
    if not force and not needs_build():
        return SO_PATH
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + ["-o", SO_PATH, SOURCES[0], "-ldl"]
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return SO_PATH


def exported_symbols():
    """Function names declared in include/harmony_b200.h (used by the CPU-side ABI test)."""
    import re
    txt = open(HEADER).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(hb_[a-z_0-9A-Z]+)\s*\(", txt)))


def lib():
    """ctypes handle with argument types set; raises if the library is missing."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(SO_PATH):
        raise RuntimeError(
            f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            f"(harmony_b200 has no CPU fallback)")
    L = ctypes.CDLL(SO_PATH)
    P, I, I64, D = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double
    L.hb_create.argtypes = [ctypes.POINTER(P), I]
    L.hb_destroy.argtypes = [P]
    L.hb_last_error.restype = ctypes.c_char_p
    L.hb_last_error.argtypes = [P]
    L.hb_pop_warning.argtypes = [P, ctypes.c_char_p, ctypes.c_size_t]
    L.hb_comm_unique_id.argtypes = [ctypes.c_char_p]
    L.hb_comm_init.argtypes = [P, I, I, ctypes.c_char_p]
    L.hb_set_shard.argtypes = [P, I64, I64]
    L.hb_setup.argtypes = [P, P, I, I64, P, P, I, P, P, P, D, I, D, D, I, D, D, I]
    L.hb_setup_device.argtypes = [P, P, I, I64, I64, I, I64, P, P, I, P, P, P, D, I, D, D, I, D, D, I, P]
    L.hb_set_seed.argtypes = [P, ctypes.c_uint64]
    L.hb_set_abort_callback.argtypes = [P, P, P]
    L.hb_init_cluster.argtypes = [P, P]
    L.hb_cluster.argtypes = [P, P]
    L.hb_moe_correct_ridge.argtypes = [P]
    L.hb_check_convergence.argtypes = [P, I]
    L.hb_compute_objective.argtypes = [P]
    L.hb_field_size.restype = I64
    L.hb_field_size.argtypes = [P, I]
    L.hb_get_field.argtypes = [P, I, P]
    L.hb_set_field.argtypes = [P, I, P]
    L.hb_get_field_device.argtypes = [P, I, P, I, I64, P]
    L.hb_get_scalar.argtypes = [P, I, ctypes.POINTER(D)]
    L.hb_set_scalar.argtypes = [P, I, D]
    L.hb_get_B_vec.argtypes = [P, P]
    L.hb_trace.restype = I64
    L.hb_trace.argtypes = [P, I, P, I64]
    L.hb_kernel_launches.restype = I64
    L.hb_kernel_launches.argtypes = [P]
    L.hb_stream.restype = P
    L.hb_stream.argtypes = [P]
    L.hb_synchronize.argtypes = [P]
    L.hb_region_time.argtypes = [P, ctypes.c_char_p, ctypes.POINTER(D), ctypes.POINTER(I64)]
    L.hb_enable_timing.argtypes = [P, I]
    L.hb_debug_permute.restype = ctypes.c_uint64
    L.hb_debug_permute.argtypes = [ctypes.c_uint64, ctypes.c_uint64, ctypes.c_uint64, I]
    L.hb_debug_update_geometry.argtypes = [I, I, ctypes.POINTER(I64)]
    L.hb_debug_kmeans_uniform.restype = D
    L.hb_debug_kmeans_uniform.argtypes = [P, ctypes.c_uint64, ctypes.c_uint64]
    L.hb_debug_kmeans_cells.argtypes = [P, P]
    L.hb_debug_sort_perm.argtypes = [P, P]
    L.hb_debug_widen.argtypes = [P, P, I64, I]
    _LIB = L
    return L
