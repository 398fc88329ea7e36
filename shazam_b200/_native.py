"""ctypes binding of ``include/sia_b200.h`` (the C ABI in ``_lib/libsia_b200.so``).

There is NO fallback: if the library has not been built (``python -m
shazam_b200.build`` / ``__graft_entry__.build()``) importing the compute path
raises, and every call needs a B200 (the library refuses other devices).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "libsia_b200.so")

SIA_F32, SIA_F64 = 0, 1
NFFT, HOP, NBINS, F_STRIDE, ROW_WORDS, HASH_BYTES = 4096, 2048, 2049, 2080, 65, 10
E_INVALID, E_CUDA, E_CAPACITY, E_NOMEM, E_UNSUPPORTED = -1, -2, -3, -4, -5


class SiaError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"sia_b200 error {code}: {msg}")
        self.code = code


class CapacityError(SiaError):
    pass


class FpParams(C.Structure):
    """``sia_fp_params`` — the arguments of ``fingerprint()`` (``__init__.py:212-217``)
    plus the module constants it reads (``__init__.py:40-51``)."""
    _fields_ = [("Fs", C.c_double), ("wsize", C.c_int32), ("wratio", C.c_double), ("fan_value", C.c_int32),
                ("amp_min", C.c_double), ("connectivity", C.c_int32), ("nbhd", C.c_int32), ("compute", C.c_int32)]


_p = C.c_void_p
_i64p = C.POINTER(C.c_int64)
_i32p = C.POINTER(C.c_int32)

# name -> (restype, argtypes); every function declared in include/sia_b200.h
SIGNATURES = {
    "sia_last_error": (C.c_char_p, []),
    "sia_version": (C.c_int, []),
    "sia_fp_params_default": (None, [C.POINTER(FpParams)]),
    "sia_ctx_create": (C.c_int, [C.c_int, C.c_int64, C.POINTER(_p)]),
    "sia_ctx_destroy": (C.c_int, [_p]),
    "sia_ctx_digest_table": (C.c_int, [_p, C.c_int]),
    "sia_num_frames": (C.c_int64, [C.c_int64]),
    "sia_fp_frames": (C.c_int64, [C.POINTER(FpParams), C.c_int64]),
    "sia_deinterleave_i16": (C.c_int, [_p, C.c_int64, C.c_int32, _p, C.c_int64, _p]),
    "sia_stft_db": (C.c_int, [_p, _p, _i64p, _i64p, C.c_int32, C.POINTER(FpParams), _p, C.c_int32, _i64p, _p]),
    "sia_peaks": (C.c_int, [_p, _p, C.c_int32, _i64p, C.c_int32, C.POINTER(FpParams), _p, _p, C.c_int64, _p, _p, _p]),
    "sia_pairs_sha1": (C.c_int, [_p, _p, _p, _p, C.c_int32, C.c_int32, _p, _p, C.c_int64, _p, _p, _p]),
    "sia_fingerprint_batch": (C.c_int, [_p, _p, _i64p, _i64p, C.c_int32, C.POINTER(FpParams), _p, _p, C.c_int64,
                                        _i64p, _i64p, _p]),
    "sia_fingerprint_batch_host": (C.c_int, [_p, _p, _i64p, _i64p, C.c_int32, C.POINTER(FpParams), _p, _p,
                                             C.c_int64, _i64p, _i64p]),
    "sia_ctx_timing": (C.c_int, [_p, C.c_int, C.POINTER(C.c_double), _i32p, C.c_int32]),
    "sia_stream_create": (C.c_int, [_p, C.c_int32, C.POINTER(FpParams), C.POINTER(_p)]),
    "sia_stream_destroy": (C.c_int, [_p]),
    "sia_stream_push": (C.c_int, [_p, _p, _i64p, _i64p, _p, _p, _p, C.c_int64, _i64p, _i64p, _p]),
    "sia_mix_noise": (C.c_int, [C.c_int, _p, C.c_int64, _p, C.c_int64, C.c_int32, C.c_int64, C.c_double, _p, C.c_int64, _p, _p]),
    "sia_index_create": (C.c_int, [C.c_int, C.c_int64, C.POINTER(_p)]),
    "sia_index_destroy": (C.c_int, [_p]),
    "sia_index_insert": (C.c_int, [_p, C.c_int32, _p, _p, C.c_int64, _p]),
    "sia_index_insert_rows": (C.c_int, [_p, _p, _p, _p, C.c_int64, _p]),
    "sia_index_insert_host": (C.c_int, [_p, C.c_int32, _p, _p, C.c_int64]),
    "sia_index_finalize": (C.c_int, [_p, _i64p]),
    "sia_index_rows": (C.c_int64, [_p]),
    "sia_index_delete_songs": (C.c_int, [_p, _i32p, C.c_int32, _i64p]),
    "sia_index_export": (C.c_int, [_p, C.c_int64, C.c_int64, _p, _p, _p, _p]),
    "sia_index_select_host": (C.c_int, [_p, _p, C.c_int64, _p, _p, _p, C.c_int64, _i64p]),
    "sia_index_query_batch": (C.c_int, [_p, _p, _p, _i64p, C.c_int32, C.c_int32, _p, _p, _p, _p, _p, _i64p, _p]),
    "sia_index_query_apriori": (C.c_int, [_p, _p, _p, _i64p, C.c_int32, C.c_int32, C.c_int32, _p, _p, _p, _p, _p, _p, _p,
                                          _i64p, _p]),
    "sia_index_query_timing": (C.c_int, [_p, C.POINTER(C.c_double)]),
    "sia_index_trim": (C.c_int, [_p]),
    "sia_index_keys": (C.c_int64, [_p]),
    "sia_index_max_song": (C.c_int32, [_p]),
    "sia_vote_tuples": (C.c_int, [C.c_int, _p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _p, _p, _p, _p, _p, _p]),
    "sia_route_entries": (C.c_int, [C.c_int, _p, _p, _p, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int64, _p, _p, _p]),
    "sia_index_expand_slots": (C.c_int, [_p, _p, C.c_int32, C.c_int64, C.c_int32, _p, C.c_int64, _p, _p]),
    "sia_vote_key_slots": (C.c_int, [C.c_int, _p, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _p, _p, _p, _p,
                                     _p, C.c_int32, _p]),
    "sia_vote_finish": (C.c_int, [C.c_int]),
    "sia_peer_alloc": (C.c_int, [C.c_int, C.c_int64, C.POINTER(_p), _p]),
    "sia_peer_open": (C.c_int, [C.c_int, _p, C.POINTER(_p)]),
    "sia_peer_close": (C.c_int, [C.c_int, _p]),
    "sia_peer_free": (C.c_int, [C.c_int, _p]),
    "sia_index_lookup_slots": (C.c_int, [_p, _p, C.c_int32, C.c_int64, C.c_int32, _p, _p, _p]),
    "sia_index_scatter_peers": (C.c_int, [_p, C.c_int32, C.c_int32, C.c_int32, _p, C.POINTER(_p), C.POINTER(_p), C.POINTER(_p),
                                          C.c_int64, C.c_int64, _p, _p]),
    "sia_vote_count_regions": (C.c_int, [C.c_int, _p, C.c_int32, C.c_int32, _p, _p, _p, C.c_int64, C.c_int64, _p, _p, _p, _p,
                                         _p, _p, _p]),
}

_lib = None


def lib() -> C.CDLL:
    """Load the shared library (once).  Raises if it was not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build the CUDA extension first "
                "(python -m shazam_b200.build, or __graft_entry__.build()). There is no CPU fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)   # AttributeError = header/library mismatch: fail loudly
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int) -> None:
    if rc == 0:
        return
    msg = lib().sia_last_error().decode("utf-8", "replace")
    raise (CapacityError if rc == E_CAPACITY else SiaError)(rc, msg)


def default_params() -> FpParams:
    p = FpParams()
    lib().sia_fp_params_default(C.byref(p))
    return p


def hop_of(p: FpParams) -> int:
    """Samples between frame starts: ``wsize - int(wsize * wratio)`` (``__init__.py:235``, ``noverlap``).
    Parameters the library rejects raise its error here."""
    rc = lib().sia_fp_frames(C.byref(p), 0)
    if rc < 0:
        check(rc)
    return int(p.wsize) - int(p.wsize * p.wratio)


def num_frames(n_samples: int, hop: int = HOP) -> int:
    """Frames of a track of ``n_samples`` at ``hop`` (mlab.specgram: a short input is one zero-padded frame)."""
    n = max(int(n_samples), NFFT)
    return 1 + (n - NFFT) // int(hop)
