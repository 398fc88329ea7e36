"""The reference's function-level interface, backed by the CUDA path.

Same names, argument meaning and return shapes as the functions the reference scripts
call by bare name (``__init__.py:116-245``, ``recognizer.py:214-338``), so a script's main
flow runs unchanged after ``from shazam_b200.compat import *`` / rebinding its globals.
Everything here calls the C ABI; nothing is computed on the CPU except the conversions
between Python tuples and arrays.
"""
from __future__ import annotations

from time import time
from typing import Optional

import numpy as np
import torch

from . import _native as N
from .fingerprinter import Fingerprinter, as_pcm_int16, digests_to_hex

# module constants, __init__.py:40-51 / recognizer.py:30-68
RATE = 44100
DEFAULT_FS = 44100
DEFAULT_WINDOW_SIZE = 4096
DEFAULT_OVERLAP_RATIO = 0.5
DEFAULT_FAN_VALUE = 5
DEFAULT_AMP_MIN = 10
CONNECTIVITY_MASK = 2
PEAK_NEIGHBORHOOD_SIZE = 10
PEAK_SORT = True
MIN_HASH_TIME_DELTA = 0
MAX_HASH_TIME_DELTA = 200
FINGERPRINT_REDUCTION = 20
TOPN = 2

_default_fp: Optional[Fingerprinter] = None


def get_fingerprinter() -> Fingerprinter:
    """Process-wide context on the current CUDA device (created on first use)."""
    global _default_fp
    if _default_fp is None:
        _default_fp = Fingerprinter(torch.cuda.current_device() if torch.cuda.is_available() else 0,
                                    max_chunk_frames=32768)
    return _default_fp


def set_fingerprinter(fp: Optional[Fingerprinter]) -> None:
    global _default_fp
    _default_fp = fp


def fingerprint(channel_samples, Fs: int = RATE, wsize: int = DEFAULT_WINDOW_SIZE,
                wratio: float = DEFAULT_OVERLAP_RATIO, fan_value: int = DEFAULT_FAN_VALUE,
                amp_min: int = DEFAULT_AMP_MIN):
    """``__init__.py:212-245``: FFT the channel, log transform, local maxima, hashes.
    Returns ``[(hex20, t1), ...]`` in the reference's order.  Any ``wratio`` with
    ``0 <= int(4096 * wratio) <= 4095``; ``t1`` counts frames of that overlap."""
    if wsize != DEFAULT_WINDOW_SIZE:
        raise N.SiaError(N.E_UNSUPPORTED, f"only wsize=4096 is implemented (got {wsize})")
    fp = get_fingerprinter()
    batch = fp.fingerprint_tracks([as_pcm_int16(channel_samples)], Fs=Fs, fan_value=fan_value, amp_min=amp_min,
                                  connectivity=CONNECTIVITY_MASK, nbhd=PEAK_NEIGHBORHOOD_SIZE, wratio=wratio)
    return list(zip(digests_to_hex(batch.hash), batch.t1.tolist()))


def get_2D_peaks(arr2D, plot: bool = False, amp_min=DEFAULT_AMP_MIN):
    """``__init__.py:116-177`` on a caller-supplied ``[freq][time]`` float array (<= 2049
    bins).  Returns ``[(f, t), ...]`` in np.where order (freq-major), like the reference."""
    if plot:
        raise N.SiaError(N.E_UNSUPPORTED, "plot=True is not part of the accelerated path")
    a = np.asarray(arr2D, dtype=np.float64)
    if a.ndim != 2 or a.shape[0] > N.NBINS:
        raise N.SiaError(N.E_UNSUPPORTED, f"arr2D must be [<= {N.NBINS} bins][frames]")
    F, T = a.shape
    if T == 0 or F == 0:
        return []
    fp = get_fingerprinter()
    host = np.full((T, N.F_STRIDE), -np.inf, np.float64)   # rows past F behave as 'outside the array'
    host[:, :F] = a.T
    spec = torch.from_numpy(host).to(fp.tdev)
    p = fp.params(amp_min=amp_min, connectivity=CONNECTIVITY_MASK, nbhd=PEAK_NEIGHBORHOOD_SIZE)
    pt, pf, _ = fp.peaks(spec, np.array([T], np.int64), p, cap_peaks=max(1024, T * F))
    t = pt.cpu().numpy().astype(np.int64)
    f = pf.cpu().numpy().astype(np.int64)
    order = np.lexsort((t, f))
    return list(zip(f[order], t[order]))


def generate_hashes(peaks, fan_value: int = DEFAULT_FAN_VALUE):
    """``__init__.py:179-210``.  ``peaks`` is a list of ``(f, t)``; sorted (stably) by time
    like the reference when PEAK_SORT."""
    if len(peaks) == 0:
        return []
    pk = np.asarray(peaks, dtype=np.int64).reshape(-1, 2)
    if PEAK_SORT:
        pk = pk[np.argsort(pk[:, 1], kind="stable")]
    fp = get_fingerprinter()
    pt = torch.from_numpy(pk[:, 1].astype(np.int32)).to(fp.tdev)
    pf = torch.from_numpy(pk[:, 0].astype(np.int32)).to(fp.tdev)
    tps = torch.tensor([0, len(pk)], dtype=torch.int64, device=fp.tdev)
    h, t1, _ = fp.pairs_sha1(pt, pf, tps, fan_value)
    return list(zip(digests_to_hex(h), t1.cpu().numpy().tolist()))


def generate_fingerprints(samples, Fs=RATE):
    """``recognizer.py:214-220``."""
    t = time()
    hashes = fingerprint(samples, Fs=Fs)
    return hashes, time() - t
