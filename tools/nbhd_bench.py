"""Batch fingerprinting at several peak footprints on one GPU: prints one JSON line.

The workload is bench.py's M1: --tracks synthetic 3-minute 44.1 kHz tracks (bench.py's generator and seeds),
device-resident, fan 15, amp_min 10, digest table on, float64 FFT by default (--compute f32 for the float32 one).
For every --nbhd value and both connectivities (2 = square, 1 = diamond) it reports the step time over --steps timed
steps (median, min, max), the per-kernel device time from sia_ctx_timing, K2's bitmap time and nanoseconds per
spectrogram frame, and peaks and hashes per second of audio: a wider neighbourhood keeps fewer peaks, so fewer hashes
and a smaller index.  nbhd 10 with the square footprint is the tuned production kernel; every other footprint runs
the footprint-general kernel.  The device name and power limit are read in the same run.

    python tools/nbhd_bench.py                      # 1000 tracks, nbhd 3, 10, 16, 20, 32, 64
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
    ap.add_argument("--nbhd", default="3,10,16,20,32,64")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--chunk-frames", type=int, default=262144)
    ap.add_argument("--compute", default="f64", choices=["f64", "f32"])
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("nbhd_bench needs a CUDA device (B200)")
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
    frames = B * N.num_frames(L)
    torch.cuda.synchronize()

    fp = Fingerprinter(0, max_chunk_frames=args.chunk_frames)
    fp.digest_table(True)
    out = {"tool": "nbhd_bench", **gpu_info(), "tracks": B, "track_samples": L, "audio_s": audio_s, "frames": frames,
           "fan_value": FAN, "amp_min": AMP_MIN, "compute": args.compute, "digest_table": True, "steps": args.steps,
           "runs": {}}
    per_frame = 5.5                                   # bench.py's hash allowance, raised when a footprint needs more
    for nbhd in [int(v) for v in args.nbhd.split(",")]:
        for conn in (2, 1):
            p = fp.params(Fs=FS, fan_value=FAN, amp_min=AMP_MIN, compute=args.compute, connectivity=conn, nbhd=nbhd)
            while True:
                cap = int(frames * per_frame * (FAN - 1))
                d_hash = torch.empty((cap, 10), dtype=torch.uint8, device=dev)
                d_t1 = torch.empty(cap, dtype=torch.int32, device=dev)
                try:
                    for _ in range(args.warmup):
                        res = fp.fingerprint_device(d_pcm, starts, lens, p, out=(d_hash, d_t1))
                    break
                except N.CapacityError:
                    del d_hash, d_t1
                    per_frame *= 2
            torch.cuda.synchronize()
            fp.timing(True)
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
            for a, b in ev:
                a.record()
                res = fp.fingerprint_device(d_pcm, starts, lens, p, out=(d_hash, d_t1))
                b.record()
            torch.cuda.synchronize()
            step_ms = [a.elapsed_time(b) for a, b in ev]
            kms, _ = fp.timing(False)
            kms = [x / args.steps for x in kms]
            # peaks of the run: one K2 call per track set on a spectrogram of the first 16 tracks
            nc = min(16, B)
            spec = fp.stft_db(d_pcm, starts[:nc], lens[:nc], p)
            _, _, tps = fp.peaks(spec, np.full(nc, N.num_frames(L), np.int64), p)
            peaks_nc = int(tps[-1].item())
            del spec
            med = float(np.median(step_ms))
            out["runs"][f"nbhd{nbhd}_{'square' if conn == 2 else 'diamond'}"] = {
                "nbhd": nbhd, "connectivity": conn, "hashes": len(res.t1),
                "step_ms_median": round(med, 2), "step_ms_min": round(min(step_ms), 2),
                "step_ms_max": round(max(step_ms), 2), "audio_s_per_s": round(audio_s / (med * 1e-3)),
                "kernel_ms": dict(zip(TIMERS, [round(x, 3) for x in kms])),
                "k2_bitmap_ms": round(kms[1], 3), "k2_bitmap_ns_per_frame": round(kms[1] * 1e6 / frames, 3),
                "peaks_per_audio_s": round(peaks_nc / (nc * L / FS), 2),
                "hashes_per_audio_s": round(len(res.t1) / audio_s, 2)}
            del d_hash, d_t1, res
    base = out["runs"].get("nbhd10_square")
    if base:
        for r in out["runs"].values():
            r["k2_bitmap_vs_tuned_nbhd10"] = round(r["k2_bitmap_ms"] / base["k2_bitmap_ms"], 3)
    fp.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
