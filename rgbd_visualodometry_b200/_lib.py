"""Loader / builder of the in-tree CUDA library liborbx.so (C-ABI in include/orbx.h).

There is no fallback: if the library is missing, cannot be built, or no sm_100 device is present,
the operators in orb.py raise -- they never run on the CPU.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
SO = os.environ.get("ORBX_LIB") or os.path.join(PKG, "liborbx.so")   # ORBX_LIB: an alternative build of the same sources (A/B experiments)
SOURCES = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h", ".inc")))
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-fmad=false",
              "-Xcompiler", "-fPIC,-O2,-ffp-contract=off", "-shared", "-diag-suppress", "68", "-lpthread"]


def _stale() -> bool:
    if os.environ.get("ORBX_LIB"):
        return not os.path.exists(SO)
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [os.path.join(ROOT, "include", "orbx.h")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    """nvcc-compile csrc/orbx.cu for sm_100a into rgbd_visualodometry_b200/liborbx.so (in-tree)."""
    if not force and not _stale():
        return SO
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found and liborbx.so is missing or stale")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", SO, os.path.join(CSRC, "orbx.cu")]
    subprocess.check_call(cmd, cwd=CSRC)
    return SO


class Keypoint(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("size", C.c_float), ("angle", C.c_float), ("response", C.c_float),
                ("octave", C.c_int32), ("class_id", C.c_int32)]


class Match(C.Structure):
    _fields_ = [("queryIdx", C.c_int32), ("trainIdx", C.c_int32), ("imgIdx", C.c_int32), ("distance", C.c_float)]


# every symbol include/orbx.h declares: name -> (restype, argtypes)
_P = C.c_void_p
SYMBOLS = {
    "orbx_create": (C.c_int, [C.POINTER(_P), C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int]),
    "orbx_destroy": (None, [_P]),
    "orbx_last_error": (C.c_char_p, [_P]),
    "orbx_version": (C.c_char_p, []),
    "orbx_synchronize": (C.c_int, [_P]),
    "orbx_stream": (_P, [_P]),
    "orbx_launch_count": (C.c_uint64, [_P]),
    "orbx_detect_and_compute": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_int, _P, _P, C.c_int, C.POINTER(C.c_int)]),
    "orbx_detect_and_compute_batch": (C.c_int, [_P, C.POINTER(_P), C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_int, _P, _P, C.c_int, _P]),
    "orbx_detect_and_compute_device": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_int, _P, _P, C.c_int, _P]),
    "orbx_match_hamming": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, C.POINTER(C.c_int)]),
    "orbx_match_hamming_knn2": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, C.POINTER(C.c_int)]),
    "orbx_match_hamming_knn": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_int, _P, C.POINTER(C.c_int)]),
    "orbx_match_hamming_device_knn": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, C.c_int, C.c_int, _P]),
    "orbx_match_hamming_device_pairwise_knn": (C.c_int, [_P, _P, C.c_int, _P, _P, C.c_int, _P, C.c_int, C.c_int, _P]),
    "orbx_match_hamming_radius": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_float, _P, C.c_int, _P, C.POINTER(C.c_int)]),
    "orbx_match_hamming_device_radius": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, C.c_int, C.c_float, _P, C.c_int64, _P]),
    "orbx_match_hamming_device_pairwise_radius": (C.c_int, [_P, _P, C.c_int, _P, _P, C.c_int, _P, C.c_int, C.c_float, _P, C.c_int64, _P]),
    "orbx_match_hamming_device": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_int, _P, _P]),
    "orbx_match_hamming_device_ragged": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, C.c_int, _P, _P]),
    "orbx_match_hamming_sets": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, C.c_int, _P, _P]),
    "orbx_match_hamming_crosscheck": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, C.POINTER(C.c_int)]),
    "orbx_match_hamming_device_crosscheck": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, C.c_int, _P, _P]),
    "orbx_match_hamming_device_pairwise": (C.c_int, [_P, _P, C.c_int, _P, _P, C.c_int, _P, C.c_int, _P, _P]),
    "orbx_match_hamming_device_pairwise_crosscheck": (C.c_int, [_P, _P, C.c_int, _P, _P, C.c_int, _P, C.c_int, _P, _P]),
    "orbx_extract_match_batch": (C.c_int, [_P, C.POINTER(_P), C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_int, _P, _P, C.c_int, _P,
                                          C.POINTER(_P), C.POINTER(C.c_int), C.c_int, C.POINTER(_P)]),
    "orbx_host_register": (C.c_int, [_P, _P, C.c_size_t]),
    "orbx_host_unregister": (C.c_int, [_P, _P]),
    "orbx_map_reserve": (C.c_int, [_P, C.c_int]),
    "orbx_map_size": (C.c_int, [_P]),
    "orbx_map_clear": (C.c_int, [_P]),
    "orbx_map_upsert": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, _P]),
    "orbx_map_upsert_from_frame": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, _P, _P]),
    "orbx_map_erase": (C.c_int, [_P, _P, C.c_int]),
    "orbx_track_match": (C.c_int, [_P, _P, C.c_int, _P, _P, C.c_int, C.c_int, _P, C.c_int, C.c_float, _P, C.POINTER(C.c_int), _P,
                                  C.POINTER(C.c_int), C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "orbx_backproject": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.c_int, C.c_size_t, C.c_float, _P, _P, _P, _P]),
    "orbx_submit_frame": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_size_t, C.c_int]),
    "orbx_collect_frame": (C.c_int, [_P, _P, _P, C.c_int, C.POINTER(C.c_int)]),
    "orbx_filter_matches": (C.c_int, [_P, C.c_int, C.c_float]),
    "orbx_level_geometry": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P, _P]),
    "orbx_debug_read_level": (C.c_int, [_P, C.c_int, C.c_int, _P, C.c_size_t]),
    "orbx_debug_read_fast": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P, C.c_int, C.POINTER(C.c_int)]),
    "orbx_debug_stage_times": (C.c_int, [_P, C.POINTER(C.c_char_p), C.POINTER(C.c_float), C.c_int]),
    "orbx_debug_force_kernels": (C.c_int, [_P, C.c_int]),
    "orbx_set_profiling": (C.c_int, [_P, C.c_int]),
}

_lib = None


def load():
    """dlopen liborbx.so (building it first if stale) and bind every declared symbol.  Raises if impossible."""
    global _lib
    if _lib is None:
        build()
        lib = C.CDLL(SO)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)          # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
