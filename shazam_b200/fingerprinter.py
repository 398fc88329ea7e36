"""Host side of the fingerprint path: a thin driver over the C ABI.

``Fingerprinter`` owns one ``sia_ctx`` (workspaces, streams) on one GPU.  torch is used
only for device buffers and the current stream.  Array-typed entry points are the fast
path; ``shazam_b200.compat`` wraps them in the reference's tuple-typed signatures.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np
import torch

from . import _native as N


@dataclass
class FingerprintBatch:
    """Digests of a batch of tracks.  ``hash[i]`` is BINARY(10) (``mysql_database.py:49``),
    ``t1[i]`` the anchor frame (the `offset` column); rows of track b are
    ``starts[b]:starts[b+1]`` in the reference's list order (``__init__.py:198-208``)."""
    hash: "np.ndarray | torch.Tensor"   # uint8 [N, 10]
    t1: "np.ndarray | torch.Tensor"     # int32 [N]
    starts: np.ndarray                  # int64 [B+1]

    def track(self, b: int):
        s, e = int(self.starts[b]), int(self.starts[b + 1])
        return self.hash[s:e], self.t1[s:e]

    def __len__(self):
        return len(self.starts) - 1


def digests_to_hex(h) -> list:
    """uint8[N,10] -> list of the reference's 20-char lowercase hex strings."""
    if isinstance(h, torch.Tensor):
        h = h.cpu().numpy()
    h = np.ascontiguousarray(h, dtype=np.uint8)
    hx = h.tobytes().hex()
    return [hx[i:i + 20] for i in range(0, len(hx), 20)]


def hex_to_digests(hexes: Sequence[str]) -> np.ndarray:
    if len(hexes) == 0:
        return np.zeros((0, N.HASH_BYTES), np.uint8)
    b = bytes.fromhex("".join(hexes))
    if len(b) != N.HASH_BYTES * len(hexes):
        raise ValueError("hashes must be 20 hex characters each (FINGERPRINT_REDUCTION)")
    return np.frombuffer(b, np.uint8).reshape(-1, N.HASH_BYTES).copy()


def as_pcm_int16(channel_samples) -> np.ndarray:
    """The reference feeds int16 arrays (``__init__.py:91-95``) or Python lists of int16
    values (``recognizer.py:361-368``).  The CUDA path takes int16 PCM only."""
    a = np.asarray(channel_samples)
    if a.ndim != 1:
        raise ValueError("channel_samples must be 1-D")
    if a.dtype == np.int16:
        return np.ascontiguousarray(a)
    if a.size == 0:
        return np.zeros(0, np.int16)
    if not np.issubdtype(a.dtype, np.integer):
        raise TypeError(f"sia_b200 fingerprints int16 PCM; got dtype {a.dtype}")
    if a.min() < -32768 or a.max() > 32767:
        raise TypeError("sample values outside the int16 range")
    return a.astype(np.int16)


def pack_tracks(tracks: Sequence[np.ndarray], pinned: bool = False):
    """Concatenate int16 tracks with 8-sample aligned starts.  Returns (pcm, starts, lens)."""
    lens = np.array([len(t) for t in tracks], np.int64)
    starts = np.zeros(len(tracks), np.int64)
    off = 0
    for i, n in enumerate(lens):
        starts[i] = off
        off += (int(n) + 7) // 8 * 8
    total = max(off, 8)
    if pinned:
        buf = torch.zeros(total, dtype=torch.int16).pin_memory()
        pcm = buf.numpy()
    else:
        buf = None
        pcm = np.zeros(total, np.int16)
    for t, s, n in zip(tracks, starts, lens):
        pcm[s:s + n] = t
    return (buf if pinned else pcm), starts, lens


def _i64(a):
    return a.ctypes.data_as(C.POINTER(C.c_int64))


class Fingerprinter:
    """One GPU's fingerprinting context.

    Defaults follow the reference's constants (``__init__.py:40-51``): window 4096, overlap
    0.5, fan 5, amp_min 10 dB, square 21x21 footprint (CONNECTIVITY_MASK 2, neighbourhood 10).
    ``wratio`` (the overlap ratio) may be any value with ``0 <= int(4096 * wratio) <= 4095``; peak times
    and ``t1`` then count frames of hop ``4096 - int(4096 * wratio)``, so an index is built and queried
    at one ``wratio``.
    ``compute='f64'`` runs the FFT in double precision (every bin within 1e-3 dB of the
    reference's float64 specgram); ``'f32'`` is the fast mode.
    """

    def __init__(self, device: int = 0, max_chunk_frames: int = 131072):
        if not torch.cuda.is_available():
            raise RuntimeError("sia_b200 needs a CUDA device (B200); there is no CPU fallback")
        self.lib = N.lib()
        self.device = int(device)
        self.tdev = torch.device("cuda", self.device)
        h = C.c_void_p()
        N.check(self.lib.sia_ctx_create(self.device, int(max_chunk_frames), C.byref(h)))
        self._h = h
        self.max_chunk_frames = int(max_chunk_frames)

    def digest_table(self, enable: bool = True) -> None:
        """Build (or free) the 13.5 GB table of every sha1("f1|f2|dt")[:10] the pipeline can produce: K3 becomes a
        gather.  Identical results; worth it when many tracks are fingerprinted with this context."""
        N.check(self.lib.sia_ctx_digest_table(self._h, 1 if enable else 0))

    def close(self):
        if getattr(self, "_h", None):
            self.lib.sia_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ helpers
    @staticmethod
    def params(Fs=44100, fan_value=5, amp_min=10, connectivity=2, nbhd=10, compute="f64",
               wsize=4096, wratio=0.5) -> N.FpParams:
        """``fingerprint()``'s parameters; ``connectivity`` 2 (square) or 1 (diamond) and ``nbhd`` 1..64 set the peak
        footprint (``CONNECTIVITY_MASK``, ``PEAK_NEIGHBORHOOD_SIZE``)."""
        p = N.default_params()
        p.Fs = float(Fs)
        p.wsize = int(wsize)
        p.wratio = float(wratio)
        p.fan_value = int(fan_value)
        p.amp_min = float(amp_min)
        p.connectivity = int(connectivity)
        p.nbhd = int(nbhd)
        p.compute = N.SIA_F64 if compute in ("f64", N.SIA_F64, torch.float64) else N.SIA_F32
        return p

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.tdev).cuda_stream)

    def timing(self, enable: bool = True):
        """Read and reset the per-kernel device timers: (ms[5], launches[5]) for
        stft, peaks-bitmap, peaks-compact, pairs+sha1, scans."""
        ms = (C.c_double * 5)()
        ln = (C.c_int32 * 5)()
        N.check(self.lib.sia_ctx_timing(self._h, int(enable), ms, ln, 5))
        return list(ms), list(ln)

    # ------------------------------------------------------------------ stages
    def stft_db(self, d_pcm: torch.Tensor, starts: np.ndarray, lens: np.ndarray, p: N.FpParams,
                out_dtype=torch.float32) -> torch.Tensor:
        """K1: int16 PCM on the device -> dB spectrogram [frames, F_STRIDE] (time-major)."""
        starts = np.ascontiguousarray(starts, np.int64)
        lens = np.ascontiguousarray(lens, np.int64)
        hop = N.hop_of(p)
        frames = int(sum(N.num_frames(n, hop) for n in lens))
        spec = torch.full((frames, N.F_STRIDE), float("-inf"), dtype=out_dtype, device=self.tdev)
        total = C.c_int64()
        N.check(self.lib.sia_stft_db(self._h, C.c_void_p(d_pcm.data_ptr()), _i64(starts), _i64(lens), len(lens),
                                     C.byref(p), C.c_void_p(spec.data_ptr()),
                                     N.SIA_F64 if out_dtype == torch.float64 else N.SIA_F32, C.byref(total),
                                     self._stream()))
        assert total.value == frames
        return spec

    def peaks(self, spec: torch.Tensor, track_frames: np.ndarray, p: N.FpParams, cap_peaks: Optional[int] = None):
        """K2: spectrogram [frames, F_STRIDE] (float32/float64) -> (peak_t, peak_f, track_peak_starts)."""
        track_frames = np.ascontiguousarray(track_frames, np.int64)
        nt = len(track_frames)
        assert spec.is_contiguous() and spec.shape[1] == N.F_STRIDE and spec.shape[0] == int(track_frames.sum())
        cap = int(cap_peaks) if cap_peaks is not None else max(1024, int(track_frames.sum()) * 64)
        pt = torch.empty(cap, dtype=torch.int32, device=self.tdev)
        pf = torch.empty(cap, dtype=torch.int32, device=self.tdev)
        tps = torch.zeros(nt + 1, dtype=torch.int64, device=self.tdev)
        status = torch.zeros(1, dtype=torch.int32, device=self.tdev)
        N.check(self.lib.sia_peaks(self._h, C.c_void_p(spec.data_ptr()),
                                   N.SIA_F64 if spec.dtype == torch.float64 else N.SIA_F32, _i64(track_frames), nt,
                                   C.byref(p), C.c_void_p(pt.data_ptr()), C.c_void_p(pf.data_ptr()), cap,
                                   C.c_void_p(tps.data_ptr()), C.c_void_p(status.data_ptr()), self._stream()))
        tps_h = tps.cpu().numpy()
        if int(status.item()) & 1:
            raise N.CapacityError(N.E_CAPACITY, f"peak capacity {cap} exceeded ({int(tps_h[-1])} peaks)")
        n = int(tps_h[-1])
        return pt[:n], pf[:n], tps

    def pairs_sha1(self, peak_t: torch.Tensor, peak_f: torch.Tensor, track_peak_starts: torch.Tensor,
                   fan_value: int, cap_hashes: Optional[int] = None):
        """K3: time-ordered peaks -> (hash uint8[N,10], t1 int32[N], track_hash_starts int64[B+1])."""
        nt = track_peak_starts.numel() - 1
        cap = int(cap_hashes) if cap_hashes is not None else max(16, peak_t.numel() * max(fan_value - 1, 1))
        hsh = torch.empty((cap, N.HASH_BYTES), dtype=torch.uint8, device=self.tdev)
        t1 = torch.empty(cap, dtype=torch.int32, device=self.tdev)
        ths = torch.zeros(nt + 1, dtype=torch.int64, device=self.tdev)
        status = torch.zeros(1, dtype=torch.int32, device=self.tdev)
        peak_t = peak_t.contiguous()
        peak_f = peak_f.contiguous()
        N.check(self.lib.sia_pairs_sha1(self._h, C.c_void_p(peak_t.data_ptr()), C.c_void_p(peak_f.data_ptr()),
                                        C.c_void_p(track_peak_starts.data_ptr()), nt, int(fan_value),
                                        C.c_void_p(hsh.data_ptr()), C.c_void_p(t1.data_ptr()), cap,
                                        C.c_void_p(ths.data_ptr()), C.c_void_p(status.data_ptr()), self._stream()))
        ths_h = ths.cpu().numpy()
        st = int(status.item())
        if st & 4:
            raise N.SiaError(N.E_INVALID, "generate_hashes: peak frequency bins must be in 0..99999")
        if st & 2:
            raise N.CapacityError(N.E_CAPACITY, f"hash capacity {cap} exceeded ({int(ths_h[-1])} hashes)")
        n = int(ths_h[-1])
        return hsh[:n], t1[:n], ths

    # ------------------------------------------------------------------ whole path
    def fingerprint_device(self, d_pcm: torch.Tensor, starts: np.ndarray, lens: np.ndarray, p: N.FpParams,
                           cap_hashes: Optional[int] = None, out: Optional[tuple] = None) -> FingerprintBatch:
        """PCM already resident in HBM -> digests in HBM (one host sync at the end)."""
        starts = np.ascontiguousarray(starts, np.int64)
        lens = np.ascontiguousarray(lens, np.int64)
        nt = len(lens)
        if out is not None:
            hsh, t1 = out
            cap = t1.numel()
        else:
            cap = int(cap_hashes) if cap_hashes is not None else self.default_cap(lens, p.fan_value, N.hop_of(p))
            hsh = torch.empty((cap, N.HASH_BYTES), dtype=torch.uint8, device=self.tdev)
            t1 = torch.empty(cap, dtype=torch.int32, device=self.tdev)
        ths = np.zeros(nt + 1, np.int64)
        total = C.c_int64()
        N.check(self.lib.sia_fingerprint_batch(self._h, C.c_void_p(d_pcm.data_ptr()), _i64(starts), _i64(lens), nt,
                                               C.byref(p), C.c_void_p(hsh.data_ptr()), C.c_void_p(t1.data_ptr()), cap,
                                               _i64(ths), C.byref(total), self._stream()))
        return FingerprintBatch(hsh[:total.value], t1[:total.value], ths)

    def fingerprint_host(self, pcm, starts: np.ndarray, lens: np.ndarray, p: N.FpParams,
                         cap_hashes: Optional[int] = None, out: Optional[tuple] = None) -> FingerprintBatch:
        """Host PCM (numpy or pinned torch int16) -> digests in host memory; H2D, kernels and
        D2H are pipelined inside the library."""
        starts = np.ascontiguousarray(starts, np.int64)
        lens = np.ascontiguousarray(lens, np.int64)
        nt = len(lens)
        if isinstance(pcm, torch.Tensor):
            assert pcm.dtype == torch.int16 and pcm.device.type == "cpu" and pcm.is_contiguous()
            pcm_ptr = pcm.data_ptr()
        else:
            pcm = np.ascontiguousarray(pcm, np.int16)
            pcm_ptr = pcm.ctypes.data
        if out is not None:
            hsh, t1 = out
            cap = t1.numel() if isinstance(t1, torch.Tensor) else len(t1)
        else:
            cap = int(cap_hashes) if cap_hashes is not None else self.default_cap(lens, p.fan_value, N.hop_of(p))
            hsh = np.empty((cap, N.HASH_BYTES), np.uint8)
            t1 = np.empty(cap, np.int32)
        hp = hsh.data_ptr() if isinstance(hsh, torch.Tensor) else hsh.ctypes.data
        tp = t1.data_ptr() if isinstance(t1, torch.Tensor) else t1.ctypes.data
        ths = np.zeros(nt + 1, np.int64)
        total = C.c_int64()
        N.check(self.lib.sia_fingerprint_batch_host(self._h, C.c_void_p(pcm_ptr), _i64(starts), _i64(lens), nt,
                                                    C.byref(p), C.c_void_p(hp), C.c_void_p(tp), cap, _i64(ths),
                                                    C.byref(total)))
        return FingerprintBatch(hsh[:total.value], t1[:total.value], ths)

    @staticmethod
    def default_cap(lens, fan_value: int, hop: int = N.HOP) -> int:
        frames = sum(N.num_frames(int(n), hop) for n in lens)
        return int(max(4096, frames * 8 * max(fan_value - 1, 1)))

    def deinterleave(self, d_interleaved: torch.Tensor, n_channels: int):
        """``data[chn::n_channels]`` of ``read()`` (``__init__.py:91-95``) on the device: interleaved int16 PCM
        -> (d_pcm, starts, lens) with one 8-sample-aligned track per channel, ready for ``fingerprint_device``."""
        assert d_interleaved.is_cuda and d_interleaved.dtype == torch.int16 and d_interleaved.is_contiguous()
        n_frames = d_interleaved.numel() // n_channels
        stride = (n_frames + 7) // 8 * 8
        out = torch.zeros(max(stride * n_channels, 8), dtype=torch.int16, device=self.tdev)
        N.check(self.lib.sia_deinterleave_i16(C.c_void_p(d_interleaved.data_ptr()), n_frames, int(n_channels),
                                              C.c_void_p(out.data_ptr()), stride, self._stream()))
        return out, np.arange(n_channels, dtype=np.int64) * stride, np.full(n_channels, n_frames, np.int64)

    def fingerprint_interleaved(self, pcm_interleaved, n_channels: int, Fs=44100, fan_value=5, amp_min=10,
                                connectivity=2, nbhd=10, compute="f64", wratio=0.5) -> FingerprintBatch:
        """All channels of one decoded file as one GPU batch (SURVEY §8f-1): the interleaved samples are copied
        once, split on the device and fingerprinted channel by channel; digests stay in HBM (one track per
        channel), e.g. for ``ingest.union_channels_device``."""
        host = np.ascontiguousarray(pcm_interleaved, np.int16)
        if not host.flags.writeable:                    # np.frombuffer over the decoder's bytes: torch wants a writable array
            host = host.copy()
        x = torch.from_numpy(host).to(self.tdev)
        d_pcm, starts, lens = self.deinterleave(x, n_channels)
        p = self.params(Fs, fan_value, amp_min, connectivity, nbhd, compute, wratio=wratio)
        cap = self.default_cap(lens, fan_value, N.hop_of(p))
        for _ in range(6):
            try:
                return self.fingerprint_device(d_pcm, starts, lens, p, cap_hashes=cap)
            except N.CapacityError as e:
                if "hash output capacity" not in str(e):
                    raise
                cap *= 4
        raise N.CapacityError(N.E_CAPACITY, "hash output keeps overflowing")

    def fingerprint_tracks(self, tracks: Sequence[np.ndarray], Fs=44100, fan_value=5, amp_min=10,
                           connectivity=2, nbhd=10, compute="f64", wratio=0.5) -> FingerprintBatch:
        """Convenience: list of int16 arrays -> host digests (with a capacity retry)."""
        tracks = [as_pcm_int16(t) for t in tracks]
        pcm, starts, lens = pack_tracks(tracks)
        p = self.params(Fs, fan_value, amp_min, connectivity, nbhd, compute, wratio=wratio)
        cap = self.default_cap(lens, fan_value, N.hop_of(p))
        for _ in range(6):
            try:
                return self.fingerprint_host(pcm, starts, lens, p, cap_hashes=cap)
            except N.CapacityError as e:
                if "hash output capacity" not in str(e):
                    raise
                cap *= 4
        raise N.CapacityError(N.E_CAPACITY, "hash output keeps overflowing")
