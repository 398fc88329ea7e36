"""Peak neighbourhood of any size, host side: the parameter checks every sia_fp_params path shares accept
PEAK_NEIGHBORHOOD_SIZE 1..64 with either CONNECTIVITY_MASK and refuse the rest; they need no device."""
import ctypes as C

import pytest


def _params(N, nbhd, conn):
    p = N.default_params()
    p.nbhd = nbhd
    p.connectivity = conn
    return p


@pytest.mark.parametrize("conn", [1, 2])
@pytest.mark.parametrize("nbhd", [1, 10, 16, 17, 20, 32, 63, 64])
def test_nbhd_accepted(native_lib, nbhd, conn):
    from shazam_b200 import _native as N
    p = _params(N, nbhd, conn)
    assert native_lib.sia_fp_frames(C.byref(p), 220500) == N.num_frames(220500)
    assert N.hop_of(p) == 2048


@pytest.mark.parametrize("conn", [1, 2])
@pytest.mark.parametrize("nbhd", [0, -1, 65, 1 << 20])
def test_nbhd_rejected(native_lib, nbhd, conn):
    from shazam_b200 import _native as N
    p = _params(N, nbhd, conn)
    assert native_lib.sia_fp_frames(C.byref(p), 220500) == N.E_INVALID
    assert "nbhd" in native_lib.sia_last_error().decode()
    with pytest.raises(N.SiaError) as e:
        N.hop_of(p)
    assert e.value.code == N.E_INVALID


def test_connectivity_still_checked(native_lib):
    from shazam_b200 import _native as N
    assert native_lib.sia_fp_frames(C.byref(_params(N, 20, 3)), 220500) == N.E_INVALID
