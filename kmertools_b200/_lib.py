"""ctypes binding of libkmertools_b200.so — the C ABI declared in include/kmertools_b200.h.

The library is the product; there is no Python or CPU fallback.  If the shared object has not been
built (python -m kmertools_b200.build) loading fails loudly.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

HERE = Path(__file__).resolve().parent
LIB_PATH = HERE / "lib" / "libkmertools_b200.so"

KTB_OK, KTB_ERR_ARG, KTB_ERR_CUDA, KTB_ERR_NOMEM, KTB_ERR_NODEVICE, KTB_ERR_IO = range(6)
NORM_COUNTS, NORM_CLI, NORM_PY = 0, 1, 2
OUT_U32, OUT_F32, OUT_F64 = 0, 1, 2
MAX_K = 12


class KtbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"kmertools_b200 error {code}: {msg}")
        self.code = code


class Stats(C.Structure):
    _fields_ = [("kernel_ms", C.c_double), ("h2d_ms", C.c_double), ("d2h_ms", C.c_double),
                ("wall_ms", C.c_double), ("launches", C.c_uint64), ("h2d_bytes", C.c_uint64),
                ("d2h_bytes", C.c_uint64)]


class FileOpts(C.Structure):
    _fields_ = [("in_path", C.c_char_p), ("out_path", C.c_char_p), ("k", C.c_int), ("canonical", C.c_int),
                ("norm", C.c_int), ("delim", C.c_char), ("header", C.c_int), ("threads", C.c_int),
                ("device", C.c_int)]


class FileStats(C.Structure):
    _fields_ = [("records", C.c_uint64), ("bases", C.c_uint64), ("bytes_written", C.c_uint64),
                ("parse_ms", C.c_double), ("gpu_wait_ms", C.c_double), ("write_ms", C.c_double),
                ("total_ms", C.c_double), ("launches", C.c_uint64)]


# every symbol include/kmertools_b200.h declares: name -> (restype, argtypes)
_VP, _U64, _I, _SZ = C.c_void_p, C.c_uint64, C.c_int, C.c_size_t
SYMBOLS = {
    "ktb_device_count": (_I, []),
    "ktb_oligo_create": (_I, [_I, _I, C.POINTER(_VP)]),
    "ktb_oligo_destroy": (None, [_VP]),
    "ktb_oligo_k": (_I, [_VP]),
    "ktb_oligo_dim": (_U64, [_VP, _I]),
    "ktb_oligo_header": (_I, [_VP, _I, C.c_char_p, _SZ]),
    "ktb_oligo_pos_maps": (_I, [_VP, _VP, _VP, C.POINTER(_U64)]),
    "ktb_kmer_pairs": (_I, [_VP, _U64, _I, _I, _VP, _VP, _U64, C.POINTER(_U64)]),
    "ktb_kmer_pairs_device": (_I, [_VP, _U64, _I, _VP, _VP, _U64, _VP, _VP]),
    "ktb_oligo_vectorise": (_I, [_VP, _VP, _VP, _U64, _I, _I, _I, _VP, _VP]),
    "ktb_oligo_vectorise_device": (_I, [_VP, _VP, _VP, _U64, _U64, _I, _I, _I, _VP, _VP, _VP]),
    "ktb_sparse_vectorise": (_I, [_VP, _VP, _U64, _I, _I, _I, _I, _I, _VP, _VP, _VP, _U64, _VP]),
    "ktb_sparse_vectorise_device": (_I, [_VP, _VP, _U64, _U64, _I, _I, _I, _I, _VP, _VP, _VP, _U64, _VP, _VP]),
    "ktb_counter_create": (_I, [_I, _I, _I, C.POINTER(_VP)]),
    "ktb_counter_destroy": (None, [_VP]),
    "ktb_counter_add": (_I, [_VP, _VP, _VP, _U64]),
    "ktb_counter_add_device": (_I, [_VP, _VP, _VP, _U64, _U64, _VP]),
    "ktb_counter_size": (_I, [_VP, C.POINTER(_U64), C.POINTER(_U64)]),
    "ktb_counter_read": (_I, [_VP, _VP, _VP, _U64]),
    "ktb_counter_read_device": (_I, [_VP, _VP, _VP, _U64, _VP]),
    "ktb_counter_coverage": (_I, [_VP, _VP, _VP, _U64, C.c_uint32, C.c_uint32, _I, _I, _VP, _VP]),
    "ktb_counter_coverage_device": (_I, [_VP, _VP, _VP, _U64, _U64, C.c_uint32, C.c_uint32, _I, _I, _VP, _VP, _VP]),
    "ktb_count_file": (_I, [C.POINTER(FileOpts), _I, C.POINTER(FileStats)]),
    "ktb_coverage_file": (_I, [C.POINTER(FileOpts), C.c_char_p, C.c_uint32, C.c_uint32, C.POINTER(FileStats)]),
    "ktb_oligo_last_stats": (_I, [_VP, C.POINTER(Stats)]),
    "ktb_oligo_set_option": (_I, [_VP, C.c_char_p, C.c_int64]),
    "ktb_host_alloc": (_VP, [_SZ]),
    "ktb_host_alloc_near": (_VP, [_SZ, _I]),
    "ktb_host_free": (None, [_VP]),
    "ktb_device_numa_node": (_I, [_I]),
    "ktb_multi_create": (_I, [_I, C.POINTER(_I), _I, C.POINTER(_VP)]),
    "ktb_multi_destroy": (None, [_VP]),
    "ktb_multi_device_count": (_I, [_VP]),
    "ktb_multi_handle": (_VP, [_VP, _I]),
    "ktb_multi_vectorise": (_I, [_VP, _VP, _VP, _U64, _I, _I, _I, _VP, _VP]),
    "ktb_multi_last_stats": (_I, [_VP, _I, C.POINTER(Stats), C.POINTER(_U64), C.POINTER(_U64)]),
    "ktb_multi_alloc_rows": (_VP, [_VP, _VP, _U64, _I, _I]),
    "ktb_shard_bounds": (_I, [_VP, _U64, _I, _VP]),
    "ktb_comp_oligo_file": (_I, [C.POINTER(FileOpts), C.POINTER(FileStats)]),
    "ktb_comp_cgr_file": (_I, [C.POINTER(FileOpts), _I, C.POINTER(FileStats)]),
    "ktb_release_cached_buffers": (None, []),
    "ktb_fastx_load": (_I, [C.c_char_p, _I, C.POINTER(_VP), C.POINTER(_VP), C.POINTER(_U64)]),
    "ktb_debug_fastx_batches": (_I, [C.c_char_p, _I, _U64, _U64, C.POINTER(_VP), C.POINTER(_VP), C.POINTER(_U64)]),
    "ktb_debug_span_write": (_I, [C.c_char_p, _VP, _U64, _U64, _I, _I]),
    "ktb_free": (None, [_VP]),
    "ktb_debug_format6": (_I, [C.c_double, C.c_char_p]),
    "ktb_debug_nt4_table": (_I, [_VP, _VP]),
    "ktb_last_error": (C.c_char_p, []),
    "ktb_abi_version": (_I, []),
}

_lib = None


def load() -> C.CDLL:
    """Load the shared library and type every entry point.  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise ImportError(
                f"{LIB_PATH} is missing: build the CUDA library first (python -m kmertools_b200.build). "
                "kmertools_b200 has no CPU fallback.")
        L = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != KTB_OK:
        raise KtbError(rc, (load().ktb_last_error() or b"").decode())
