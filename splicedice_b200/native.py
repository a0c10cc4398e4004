"""ctypes binding of ``libsplicedice_b200.so`` (the C-ABI declared in include/splicedice_b200.h).

PyTorch is used by callers only to own device memory and streams; this module passes raw
pointers.  There is no CPU fallback: if the library cannot be loaded (or built) every entry
point raises ``NativeLibraryError``.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_int64, c_size_t, c_uint32, c_uint64, c_void_p

from . import build as _build

SD_OK = 0
SD_ERR_INVALID, SD_ERR_CUDA, SD_ERR_WORKSPACE, SD_ERR_OVERFLOW, SD_ERR_UNSUPPORTED = 1, 2, 3, 4, 5
SD_QUANT_AUTO, SD_QUANT_GATHER, SD_QUANT_TILED = 0, 1, 2
SD_QUANT_NARROW_TILES, SD_QUANT_VEC1, SD_QUANT_VEC2, SD_QUANT_GENERAL = 0x10000, 0x20000, 0x40000, 0x80000
SD_RANKSUM_F32, SD_RANKSUM_F64 = 0, 1
SD_RANKSUM_MAX_SAMPLES, SD_KRUSKAL_MAX_GROUPS, SD_SIGNEDRANK_MAX_PAIRS = 16384, 256, 8192
SD_FRIEDMAN_MAX_CONDITIONS = 256
ABI_VERSION = 1


class NativeLibraryError(RuntimeError):
    pass


class QuantFilter(ctypes.Structure):
    """sd_quant_filter of include/splicedice_b200.h"""
    _fields_ = [("max_length", c_int32), ("min_length", c_int32), ("min_overhang", c_int32), ("min_unique", c_int32),
                ("no_multimap", c_int32), ("low_coverage_nan", c_int32), ("motif_mask", c_uint32),
                ("reserved", c_uint32), ("min_entropy", c_double)]


class NativeCallError(RuntimeError):
    def __init__(self, fn, code, msg):
        super().__init__(f"{fn} failed (code {code}): {msg}")
        self.code = code


_P = c_void_p   # every device / host pointer crosses as void*

_SIGNATURES = {
    "sd_version": (c_int, []),
    "sd_last_error": (c_char_p, []),
    "sd_device_info": (c_int, [c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_size_t)]),
    "sd_cluster_workspace_bytes": (c_size_t, [c_int64]),
    "sd_cluster_build": (c_int, [c_int64, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                 POINTER(c_int64), POINTER(c_int64), _P, c_size_t, _P]),
    "sd_cluster_fill_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "sd_cluster_fill": (c_int, [c_int64, c_int64, _P, _P, _P, _P, c_size_t, _P, c_size_t, _P]),
    "sd_quant_ps": (c_int, [c_int64, c_int32, _P, c_int64, _P, _P, _P, c_int64, _P, c_int64,
                            _P, c_int64, _P, c_int64, c_int64, c_int64, c_uint32, _P]),
    "sd_quant_last_launch": (c_char_p, []),
    "sd_quant_ps_host": (c_int, [c_int, c_int64, c_int32, _P, c_int64, _P, _P, _P, c_int64, _P, c_int64]),
    "sd_host_pipeline_trim": (c_int, [c_int]),
    "sd_fisher_pairwise": (c_int, [c_int64, c_int32, _P, c_int64, _P, c_int64, c_int64, _P, _P,
                                   _P, c_int64, c_int64, c_int64, _P]),
    "sd_fisher_pairwise_bounded": (c_int, [c_int64, c_int32, _P, c_int64, _P, c_int64, c_int64, _P, _P,
                                           _P, c_int64, c_int64, c_int64, c_int64, _P]),
    "sd_fisher_pairwise_scatter": (c_int, [c_int64, c_int32, _P, c_int64, _P, c_int64, c_int64, _P, _P,
                                           c_int32, _P, _P, _P, c_int64, c_int64, c_int64, c_int64, _P]),
    "sd_peer_alloc": (c_int, [c_size_t, POINTER(c_void_p), _P]),
    "sd_peer_free": (c_int, [_P]),
    "sd_peer_open": (c_int, [_P, POINTER(c_void_p)]),
    "sd_peer_close": (c_int, [_P]),
    "sd_peer_scatter_rows": (c_int, [_P, c_int64, c_int64, c_int32, _P, _P, _P, c_int64, _P]),
    "sd_fisher_tables": (c_int, [c_int64, _P, _P, _P, _P, _P, _P]),
    "sd_fisher_pairwise_host": (c_int, [c_int, c_int64, c_int32, _P, c_int64, _P, c_int64,
                                        c_int64, _P, _P, _P, c_int64]),
    "sd_pairwise_host": (c_int, [c_int, c_int64, c_int32, _P, c_int64, _P, _P, c_int64, _P, _P, _P, c_int64]),
    "sd_chi2_pairwise": (c_int, [c_int64, c_int32, _P, c_int64, _P, c_int64, c_int64, _P, _P,
                                 _P, c_int64, c_int64, c_int64, _P, _P]),
    "sd_ranksum_rows": (c_int, [c_int64, c_int32, _P, c_int64, c_int, c_int32, _P, c_int32, _P,
                                c_int64, c_int64, _P, c_int64, _P, c_int64, _P]),
    "sd_kruskal_rows": (c_int, [c_int64, c_int32, _P, c_int64, c_int, c_int32, c_int32, _P, _P,
                                c_int64, c_int64, _P, c_int64, _P, c_int64, _P, c_int64, _P]),
    "sd_signedrank_rows": (c_int, [c_int64, c_int32, _P, c_int64, c_int, c_int32, _P, _P,
                                   c_int64, c_int64, _P, c_int64, _P, c_int64, _P]),
    "sd_friedman_rows": (c_int, [c_int64, c_int32, _P, c_int64, c_int, c_int32, c_int32, _P,
                                 c_int64, c_int64, _P, _P, c_int64, _P, c_int64, _P]),
    "sd_bh_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int]),
    "sd_bh_adjust": (c_int, [c_int64, c_int64, _P, c_int64, _P, c_int64, c_int, _P, c_size_t, _P]),
    "sd_ir_ratio": (c_int, [c_int64, c_int32, _P, c_int64, _P, c_int64, _P, _P, _P, c_int64,
                            c_int64, c_int64, _P]),
    "sd_rsd5": (c_int, [c_int64, _P, _P, _P]),
    "sd_host_table_open": (c_void_p, [c_char_p, POINTER(c_int64), POINTER(c_int32), POINTER(c_int64), POINTER(c_int64)]),
    "sd_host_table_close": (None, [_P]),
    "sd_host_table_read": (c_int, [_P, _P, _P, _P, _P, c_int64, c_int32]),
    "sd_ingest_create": (c_void_p, []),
    "sd_ingest_destroy": (None, [_P]),
    "sd_ingest_collect": (c_int, [_P, c_int32, _P, _P, _P, c_int32]),
    "sd_ingest_junction_count": (c_int64, [_P]),
    "sd_ingest_chrom_count": (c_int32, [_P]),
    "sd_ingest_chrom_name": (c_char_p, [_P, c_int32]),
    "sd_ingest_export": (c_int, [_P, _P, _P, _P, _P]),
    "sd_ingest_index": (c_int, [_P, c_int64, _P, _P, _P, _P, _P, _P]),
    "sd_ingest_counts": (c_int, [_P, c_int32, _P, _P, _P, _P, _P, c_int64, _P, c_int64, c_int32]),
    "sd_host_format_rows": (c_int, [c_int, _P, c_int64, c_int32, c_int64, _P, _P, _P, c_size_t,
                                    POINTER(c_size_t), c_int]),
    "sd_host_format_rows_segments": (c_int, [c_int, _P, c_int64, c_int32, c_int64, _P, _P, _P, c_size_t, _P, _P, c_int32,
                                             POINTER(c_int32), POINTER(c_size_t), c_int]),
    "sd_synth_counts": (c_int, [c_uint64, c_int64, c_int64, c_int32, c_int64, c_uint32, _P, c_int64, _P]),
    "sd_probe_fp64": (c_int, [POINTER(c_double), _P]),
    "sd_probe_copy": (c_int, [c_int64, POINTER(c_double), _P]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def library_path() -> str:
    return _build.LIB


def load():
    """Load (building first if the sources are newer and nvcc exists) the shared library."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    override = os.environ.get("SPLICEDICE_B200_LIB")          # experiment builds (build.build_variant)
    try:
        if override:
            path = override
        elif _build.nvcc() is not None:
            path = _build.build()
    except Exception as e:  # build failure is fatal: there is nothing to fall back to
        raise NativeLibraryError(f"cannot build libsplicedice_b200.so: {e}") from e
    if not os.path.isfile(path):
        raise NativeLibraryError(
            f"{path} is missing and nvcc is not available; splicedice_b200 has no CPU fallback")
    try:
        lib = ctypes.CDLL(path)
    except OSError as e:
        raise NativeLibraryError(f"cannot load {path}: {e}") from e
    for name, (res, args) in _SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise NativeLibraryError(f"{path} does not export {name}") from e
        fn.restype = res
        fn.argtypes = args
    if lib.sd_version() != ABI_VERSION:
        raise NativeLibraryError(f"ABI mismatch: library {lib.sd_version()}, binding {ABI_VERSION}")
    _lib = lib
    return lib


def last_error() -> str:
    return load().sd_last_error().decode("utf-8", "replace")


def call(name: str, *args):
    """Call an int-returning entry point and raise on a non-zero status."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != SD_OK:
        raise NativeCallError(name, rc, lib.sd_last_error().decode("utf-8", "replace"))


def ptr(t):
    """Raw pointer of a torch tensor / numpy array / None."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return c_void_p(t.data_ptr())
    return c_void_p(t.ctypes.data)


def stream_ptr(stream=None):
    """cudaStream_t of a torch stream (None -> torch's current stream)."""
    import torch
    if stream is None:
        stream = torch.cuda.current_stream()
    return c_void_p(stream.cuda_stream)
