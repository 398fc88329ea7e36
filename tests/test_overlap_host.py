"""Any overlap ratio, host side: the oracle's spectrogram at other noverlap values against scipy, and the library's
frame count (sia_fp_frames) and parameter checks, which need no device."""
import ctypes as C
import math

import numpy as np
import pytest

from oracle import sia_oracle as O


@pytest.mark.parametrize("noverlap", [0, 1, 1024, 1228, 2047, 3072, 4095])
def test_specgram_any_overlap_matches_scipy(wav_fixture, noverlap):
    from scipy.signal import spectrogram
    x = wav_fixture["pcm"][:6000] if noverlap > 3072 else wav_fixture["pcm"]   # hop 1: one frame per sample
    P = O.specgram_psd(x, 22050, noverlap=noverlap)
    _, _, S = spectrogram(x.astype(np.float64), fs=22050, window=np.hanning(4096), nperseg=4096, noverlap=noverlap,
                          detrend=False, scaling="density", mode="psd")
    assert P.shape == S.shape == (2049, O.num_frames(len(x), noverlap=noverlap))
    assert np.max(np.abs(P - S) / S) < 1e-8


def _params(N, wratio=0.5, wsize=4096):
    p = N.default_params()
    p.wratio = wratio
    p.wsize = wsize
    return p


def test_fp_frames_matches_oracle(native_lib):
    from shazam_b200 import _native as N
    rng = np.random.default_rng(5)
    ratios = [0.5, 0.0, -0.0001, 0.25, 0.3, 0.75, 0.9, 0.99, 0.99999] + list(rng.uniform(0, 0.9999, 20))
    for w in ratios:
        noverlap = int(4096 * w)
        hop = 4096 - noverlap
        p = _params(N, w)
        assert N.hop_of(p) == hop
        lens = [0, 1, 3000, 4095, 4096, 4097, 4096 + hop - 1, 4096 + hop, 4096 + hop + 1, 3 * hop + 4096,
                220500] + list(rng.integers(0, 400000, 20))
        for n in lens:
            want = O.num_frames(int(n), 4096, noverlap)
            assert native_lib.sia_fp_frames(C.byref(p), int(n)) == want, (w, n)
            assert N.num_frames(int(n), hop) == want, (w, n)
    # wratio 0.5 is sia_num_frames
    p = _params(N)
    for n in (0, 4096, 8191, 8192, 220500, 7938000):
        assert native_lib.sia_fp_frames(C.byref(p), n) == native_lib.sia_num_frames(n) == N.num_frames(n)


@pytest.mark.parametrize("wsize,wratio,code", [
    (2048, 0.5, -5),              # SIA_E_UNSUPPORTED: the window size sets the spectrogram's shape
    (4096, 1.0, -1),              # SIA_E_INVALID: noverlap 4096, hop 0
    (4096, -0.01, -5),            # noverlap -40: gaps between frames
    (4096, math.nan, -1),
    (4096, math.inf, -1),
])
def test_fp_frames_rejects(native_lib, wsize, wratio, code):
    from shazam_b200 import _native as N
    p = _params(N, wratio, wsize)
    assert native_lib.sia_fp_frames(C.byref(p), 100000) == code
    assert native_lib.sia_last_error()
    with pytest.raises(N.SiaError) as e:
        N.hop_of(p)
    assert e.value.code == code


def test_fp_frames_rejects_negative_length(native_lib):
    from shazam_b200 import _native as N
    assert native_lib.sia_fp_frames(C.byref(_params(N, 0.75)), -1) == N.E_INVALID
    assert native_lib.sia_fp_frames(None, 4096) == N.E_INVALID
