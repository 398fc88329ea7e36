"""Batch fingerprinting at several overlap ratios on one GPU: prints one JSON line.

The workload is bench.py's M1: --tracks synthetic 3-minute 44.1 kHz tracks (bench.py's generator and seeds),
device-resident, fan 15, amp_min 10, float64 FFT, digest table on.  For every --ratios value (wratio; hop =
4096 - int(4096 * wratio)) it reports the step time over --steps timed steps (median, min, max), audio-s/s, the
per-kernel device time from sia_ctx_timing, and K1 and K2 nanoseconds per spectrogram frame, K1's also as a ratio to
the hop-2048 path.  A lower hop means more frames per second of audio, so audio-s/s falls with it; ns per frame is
what compares the kernels.  The bit-identity check runs K1 on --check-tracks of the tracks: every even row at wratio
0.75 (hop 1024) must equal the row at wratio 0.5 that starts at the same sample.  The device name and power limit
are read in the same run.

    python tools/overlap_bench.py                      # 1000 tracks, wratio 0.5, 0.75, 0.3, 0
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for d in (ROOT, os.path.join(ROOT, "tools")):
    if d not in sys.path:
        sys.path.insert(0, d)

FS, FAN, AMP_MIN = 44100, 15, 10
TIMERS = ["stft", "peaks_bitmap", "peaks_compact", "pairs_sha1", "scan"]


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--tracks", type=int, default=1000)
    ap.add_argument("--track-samples", type=int, default=7_938_000)
    ap.add_argument("--ratios", default="0.5,0.75,0.3,0")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--chunk-frames", type=int, default=262144)
    ap.add_argument("--check-tracks", type=int, default=8)
    ap.add_argument("--compute", default="f64", choices=["f64", "f32"])
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("overlap_bench needs a CUDA device (B200)")
    from bench import synth_tracks_gpu
    from shazam_b200 import _native as N
    from shazam_b200.fingerprinter import Fingerprinter
    from stream_bench import gpu_info

    dev = torch.device("cuda", 0)
    B, L = args.tracks, args.track_samples
    stride = (L + 7) // 8 * 8
    d_pcm = torch.empty(B * stride, dtype=torch.int16, device=dev)
    rows = d_pcm.view(B, stride)
    synth_tracks_gpu(dev, 0, B, L, [rows[i, :L] for i in range(B)])
    starts = np.arange(B, dtype=np.int64) * stride
    lens = np.full(B, L, np.int64)
    audio_s = B * L / FS
    torch.cuda.synchronize()

    fp = Fingerprinter(0, max_chunk_frames=args.chunk_frames)
    fp.digest_table(True)
    out = {"tool": "overlap_bench", **gpu_info(), "tracks": B, "track_samples": L, "audio_s": audio_s,
           "fan_value": FAN, "amp_min": AMP_MIN, "compute": args.compute, "digest_table": True, "steps": args.steps,
           "ratios": {}}

    for wratio in [float(r) for r in args.ratios.split(",")]:
        p = fp.params(Fs=FS, fan_value=FAN, amp_min=AMP_MIN, compute=args.compute, wratio=wratio)
        hop = N.hop_of(p)
        frames = B * N.num_frames(L, hop)
        cap = int(frames * 5.5 * (FAN - 1))               # bench.py's allowance: ~4 peaks per frame on this signal
        d_hash = torch.empty((cap, 10), dtype=torch.uint8, device=dev)
        d_t1 = torch.empty(cap, dtype=torch.int32, device=dev)
        for _ in range(args.warmup):
            res = fp.fingerprint_device(d_pcm, starts, lens, p, out=(d_hash, d_t1))
        torch.cuda.synchronize()
        fp.timing(True)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for a, b in ev:
            a.record()
            res = fp.fingerprint_device(d_pcm, starts, lens, p, out=(d_hash, d_t1))
            b.record()
        torch.cuda.synchronize()
        step_ms = [a.elapsed_time(b) for a, b in ev]
        kms, kl = fp.timing(False)
        kms = [x / args.steps for x in kms]
        med = float(np.median(step_ms))
        out["ratios"][str(wratio)] = {
            "hop": hop, "frames": frames, "hashes": len(res.t1),
            "step_ms_median": round(med, 2), "step_ms_min": round(min(step_ms), 2),
            "step_ms_max": round(max(step_ms), 2), "audio_s_per_s": round(audio_s / (med * 1e-3)),
            "kernel_ms": dict(zip(TIMERS, [round(x, 3) for x in kms])),
            "k1_ns_per_frame": round(kms[0] * 1e6 / frames, 3),
            "k2_ns_per_frame": round((kms[1] + kms[2]) * 1e6 / frames, 3)}
        del d_hash, d_t1, res
    base = out["ratios"].get("0.5")
    if base:
        for r in out["ratios"].values():
            r["k1_ns_per_frame_vs_hop2048"] = round(r["k1_ns_per_frame"] / base["k1_ns_per_frame"], 4)

    # K1 bit identity: even rows at hop 1024 against the hop-2048 rows, on a subset of the tracks
    nc = min(args.check_tracks, B)
    spec = {}
    for wratio in (0.5, 0.75):
        p = fp.params(Fs=FS, compute=args.compute, wratio=wratio)
        spec[wratio] = fp.stft_db(d_pcm, starts[:nc], lens[:nc], p).view(nc, -1, N.F_STRIDE)[:, :, :N.NBINS]
    n = min(spec[0.5].shape[1], (spec[0.75].shape[1] + 1) // 2)
    out["bit_identity_0.75_vs_0.5"] = {"tracks": nc, "rows": nc * n,
                                       "equal": bool(torch.equal(spec[0.75][:, 0:2 * n:2], spec[0.5][:, :n]))}
    fp.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
