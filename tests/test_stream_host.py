"""The streaming C ABI rejects NULL and invalid arguments with SIA_E_INVALID before touching a GPU, and the Python
driver refuses to run without CUDA."""
import ctypes as C

import pytest


def test_stream_abi_invalid_arguments(native_lib):
    from shazam_b200 import _native as N
    p = N.default_params()
    h = C.c_void_p()
    assert native_lib.sia_stream_create(None, 4, C.byref(p), C.byref(h)) == N.E_INVALID
    assert b"NULL" in native_lib.sia_last_error()
    assert native_lib.sia_stream_create(None, 4, C.byref(p), None) == N.E_INVALID
    assert native_lib.sia_stream_destroy(None) == N.E_INVALID
    z = (C.c_int64 * 2)()
    total = C.c_int64()
    assert native_lib.sia_stream_push(None, None, z, z, None, None, None, 0, None, C.byref(total), None) == N.E_INVALID
    assert b"NULL" in native_lib.sia_last_error()


def test_stream_fingerprinter_needs_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from shazam_b200.stream import StreamFingerprinter
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        StreamFingerprinter(None, 4)


def test_stream_is_a_lazy_import():
    import shazam_b200
    assert shazam_b200.stream.StreamFingerprinter.__name__ == "StreamFingerprinter"
