"""sia_index_query_apriori rejects invalid arguments with SIA_E_INVALID and a message before touching a GPU."""
import ctypes as C


def _call(lib, ix, topn, batch, outs):
    starts = (C.c_int64 * 2)(0, 4)
    stats = (C.c_int64 * 4)()
    return lib.sia_index_query_apriori(ix, None, None, starts, 1, topn, batch, *outs, stats, None)


def test_query_apriori_invalid_arguments(native_lib):
    from shazam_b200 import _native as N
    fake = [C.c_void_p(0x1000 + 64 * i) for i in range(7)]    # never dereferenced: the checks come first
    assert _call(native_lib, None, 2, 1000, fake) == N.E_INVALID
    assert b"NULL argument" in native_lib.sia_last_error()
    for i in range(7):
        outs = list(fake)
        outs[i] = None
        assert _call(native_lib, None, 2, 1000, outs) == N.E_INVALID
        assert b"NULL output" in native_lib.sia_last_error()
    for topn, batch in ((2, 0), (2, -5), (0, 1000), (-1, 1)):
        assert _call(native_lib, None, topn, batch, fake) == N.E_INVALID
        assert b"batch_hashes >= 1" in native_lib.sia_last_error()
