"""Streaming fingerprinting: many concurrent audio streams, fed block by block.

``StreamFingerprinter`` holds ``n_streams`` independent streams on one ``Fingerprinter``'s context (the
``sia_stream_*`` functions of the C ABI).  Every push gives each stream a block of int16 PCM (possibly empty) and
returns, per stream, the hashes that became final during that push.  For any cut of a stream's PCM into blocks, the
concatenation of what it emits up to and including the push that ends it equals ``Fingerprinter`` on the whole PCM
with the same parameters: digests, ``t1`` (frame index from the stream's start) and the reference's list order
(``__init__.py:198-208``).  So a live recording is fingerprinted while it arrives, and recordings longer than the
context workspace (which the batch path refuses) are fingerprinted block by block.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np
import torch

from . import _native as N
from .fingerprinter import FingerprintBatch, Fingerprinter, as_pcm_int16, pack_tracks

N_TIMERS = 6   # stft, peaks(bitmap), peaks(compact), pairs+sha1, scans, stream-state copies


def _i64(a):
    return a.ctypes.data_as(C.POINTER(C.c_int64))


class StreamFingerprinter:
    """``n_streams`` streams with the parameters of ``fingerprint()`` (``__init__.py:212-217``).

    Calls on this object and on its ``Fingerprinter`` are serialised by the caller; close this object before the
    ``Fingerprinter``.  A push that raises (``CapacityError``) leaves every stream as it was, so it can be retried
    with a bigger output buffer or smaller blocks."""

    def __init__(self, fp: Fingerprinter, n_streams: int, Fs=44100, fan_value=5, amp_min=10, connectivity=2,
                 nbhd=10, compute="f64", wratio=0.5):
        if not torch.cuda.is_available():
            raise RuntimeError("sia_b200 needs a CUDA device (B200); there is no CPU fallback")
        self.fp = fp
        self.lib = fp.lib
        self.n_streams = int(n_streams)
        self.p = fp.params(Fs, fan_value, amp_min, connectivity, nbhd, compute, wratio=wratio)
        self.hop = N.hop_of(self.p)
        h = C.c_void_p()
        N.check(self.lib.sia_stream_create(fp._h, self.n_streams, C.byref(self.p), C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self.lib.sia_stream_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _end_flags(self, end) -> np.ndarray:
        if end is None:
            return np.zeros(self.n_streams, np.uint8)
        if isinstance(end, (bool, np.bool_)):
            return np.full(self.n_streams, 1 if end else 0, np.uint8)
        e = np.ascontiguousarray(np.asarray(end, dtype=bool).astype(np.uint8))
        if e.shape != (self.n_streams,):
            raise ValueError(f"end must be a bool or {self.n_streams} flags")
        return e

    def default_cap(self, lens) -> int:
        """Hash rows a push of blocks of these lengths needs at most, with the batch path's allowance per frame."""
        fan = int(self.p.fan_value)
        frames = int(sum(int(n) // self.hop + 2 + int(self.p.nbhd) for n in lens))
        return int(max(4096, (frames * 8 + self.n_streams * fan) * max(fan - 1, 1)))

    def push_device(self, d_pcm: torch.Tensor, starts, lens, end=None, out: Optional[tuple] = None,
                    cap_hashes: Optional[int] = None) -> FingerprintBatch:
        """Blocks already in HBM: stream b gets ``d_pcm[starts[b]:starts[b]+lens[b]]`` (starts multiples of 8).
        Digests stay in HBM; rows of stream b are ``starts[b]:starts[b+1]`` of the result (one host sync)."""
        if self._h is None:
            raise RuntimeError("StreamFingerprinter is closed")
        starts = np.ascontiguousarray(starts, np.int64)
        lens = np.ascontiguousarray(lens, np.int64)
        if starts.shape != (self.n_streams,) or lens.shape != (self.n_streams,):
            raise ValueError(f"starts and lens need one entry per stream ({self.n_streams})")
        flags = self._end_flags(end)
        tdev = self.fp.tdev
        if out is not None:
            hsh, t1 = out
            cap = t1.numel()
        else:
            cap = int(cap_hashes) if cap_hashes is not None else self.default_cap(lens)
            hsh = torch.empty((cap, N.HASH_BYTES), dtype=torch.uint8, device=tdev)
            t1 = torch.empty(cap, dtype=torch.int32, device=tdev)
        ths = np.zeros(self.n_streams + 1, np.int64)
        total = C.c_int64()
        pcm_ptr = d_pcm.data_ptr() if d_pcm is not None and d_pcm.numel() else None
        N.check(self.lib.sia_stream_push(self._h, C.c_void_p(pcm_ptr), _i64(starts), _i64(lens),
                                         C.c_void_p(flags.ctypes.data), C.c_void_p(hsh.data_ptr()),
                                         C.c_void_p(t1.data_ptr()), cap, _i64(ths), C.byref(total),
                                         self.fp._stream()))
        return FingerprintBatch(hsh[:total.value], t1[:total.value], ths)

    def push(self, blocks: Sequence, end=None) -> FingerprintBatch:
        """One int16 array per stream (empty or None: nothing new) -> host digests of the hashes that became final,
        with the capacity retry of ``Fingerprinter.fingerprint_tracks``."""
        if len(blocks) != self.n_streams:
            raise ValueError(f"push needs one block per stream ({self.n_streams})")
        blocks = [np.zeros(0, np.int16) if b is None else as_pcm_int16(b) for b in blocks]
        pcm, starts, lens = pack_tracks(blocks)
        d_pcm = torch.from_numpy(pcm).to(self.fp.tdev)
        cap = self.default_cap(lens)
        for _ in range(6):
            try:
                r = self.push_device(d_pcm, starts, lens, end=end, cap_hashes=cap)
                return FingerprintBatch(r.hash.cpu().numpy(), r.t1.cpu().numpy(), r.starts)
            except N.CapacityError as e:
                if "hash output capacity" not in str(e):
                    raise
                cap *= 4
        raise N.CapacityError(N.E_CAPACITY, "hash output keeps overflowing")

    def timing(self, enable: bool = True):
        """Read and reset the context's per-kernel device timers, including the stream-state copies of the pushes:
        (ms[6], launches[6]) for stft, peaks-bitmap, peaks-compact, pairs+sha1, scans, stream-state copies."""
        ms = (C.c_double * N_TIMERS)()
        ln = (C.c_int32 * N_TIMERS)()
        N.check(self.lib.sia_ctx_timing(self.fp._h, int(enable), ms, ln, N_TIMERS))
        return list(ms), list(ln)
