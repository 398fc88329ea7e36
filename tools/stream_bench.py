"""Streaming fingerprinting on one GPU: prints one JSON line.

  (a) 2 streams pushing 8 192-sample blocks (the reference recogniser's read size, recognizer.py:357-369): device time
      per push, and the time from the last push to its final hashes (the wall time of the push that ends the streams);
  (b) --streams streams x --seconds s of audio pushed in blocks of --block samples: audio-s/s over the pushes, the
      per-kernel split from sia_ctx_timing (a second pass with the timers on) and the K2 rows processed per new row;
  (c) the batch path (sia_fingerprint_batch) on the same audio, one track per stream;
  and whether everything (b) emitted is bit-identical to (c).

The audio is bench.py's synthetic music (6 voices, note changes every 0.25 s, noise): a pool of --pool tracks, each
stream a window of it at its own 8-sample offset.  Parameters are bench.py's: Fs 44100, fan 15, amp_min 10, digest
table on (--no-digest-table to hash with SHA-1).  The device name and power limit are read in the same run.

    python tools/stream_bench.py                       # 10 000 streams x 60 s in 1 s blocks
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FS, FAN, AMP_MIN = 44100, 15, 10


def gpu_info():
    import torch
    info = {"device": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out.splitlines()[0])
    except Exception as e:   # the number is reported as unknown rather than guessed
        info["power_limit_error"] = str(e)
    return info


def k2_rows_per_new_row(block: int, n_blocks: int, nbhd: int = 10) -> float:
    """Rows K2 filters per push (carried min(2*nbhd, F) + new) over the new rows, for one stream."""
    L = F = rows = new = 0
    for _ in range(n_blocks):
        L += block
        Fn = 1 + (L - 4096) // 2048 if L >= 4096 else 0
        if Fn > F:
            rows += min(2 * nbhd, F) + Fn - F
            new += Fn - F
        F = Fn
    return rows / max(new, 1)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--streams", type=int, default=10000)
    ap.add_argument("--seconds", type=int, default=60)
    ap.add_argument("--block", type=int, default=44096, help="samples per push and stream (multiple of 8; 1 s = 44096)")
    ap.add_argument("--pool", type=int, default=1000, help="distinct synthetic tracks the streams are windows of")
    ap.add_argument("--small-block", type=int, default=8192)
    ap.add_argument("--small-pushes", type=int, default=26)
    ap.add_argument("--small-rounds", type=int, default=20)
    ap.add_argument("--compute", default="f64", choices=["f64", "f32"])
    ap.add_argument("--no-digest-table", action="store_true")
    args = ap.parse_args()
    if args.block % 8:
        ap.error("--block must be a multiple of 8 samples")

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("stream_bench needs a CUDA device (B200)")
    from bench import synth_tracks_gpu
    from shazam_b200 import _native as N
    from shazam_b200.fingerprinter import Fingerprinter
    from shazam_b200.stream import StreamFingerprinter

    dev = torch.device("cuda", 0)
    S, nb, blk = args.streams, args.seconds * FS // args.block, args.block
    L = nb * blk
    # pool of synthetic tracks; stream b reads L samples at its own 8-aligned offset
    pool_len = args.pool * L
    pool = torch.empty(pool_len, dtype=torch.int16, device=dev)
    synth_tracks_gpu(dev, 7_000_000, args.pool, L, [pool[i * L:(i + 1) * L] for i in range(args.pool)])
    span = pool_len - L
    offs = (np.arange(S, dtype=np.int64) * 1_000_003 * 8) % (span // 8 * 8 + 8)
    offs = np.minimum(offs // 8 * 8, span // 8 * 8)
    lens = np.full(S, L, np.int64)
    torch.cuda.synchronize()

    fp = Fingerprinter(0)
    if not args.no_digest_table:
        fp.digest_table(True)
    p = fp.params(Fs=FS, fan_value=FAN, amp_min=AMP_MIN, compute=args.compute)
    out = {"tool": "stream_bench", **gpu_info(), "fan_value": FAN, "amp_min": AMP_MIN, "compute": args.compute,
           "digest_table": not args.no_digest_table}

    # ---- (c) batch path, one track per stream --------------------------------------------------------------
    cap_c = int(S * N.num_frames(L) * 8 * (FAN - 1))
    c_hash = torch.empty((cap_c, 10), dtype=torch.uint8, device=dev)
    c_t1 = torch.empty(cap_c, dtype=torch.int32, device=dev)
    for _ in range(2):
        res_c = fp.fingerprint_device(pool, offs, lens, p, out=(c_hash, c_t1))
    reps = 3
    torch.cuda.synchronize()
    fp.timing(True)
    t0 = time.perf_counter()
    for _ in range(reps):
        res_c = fp.fingerprint_device(pool, offs, lens, p, out=(c_hash, c_t1))
    torch.cuda.synchronize()
    ms_c = (time.perf_counter() - t0) * 1e3 / reps
    kms_c, _ = fp.timing(False)
    audio_s = S * L / FS
    c_starts = res_c.starts.copy()
    out["c_batch"] = {"tracks": S, "audio_s": audio_s, "ms": round(ms_c, 2), "audio_s_per_s": audio_s / (ms_c * 1e-3),
                      "hashes": int(c_starts[-1]),
                      "kernel_ms": dict(zip(["stft", "peaks_bitmap", "peaks_compact", "pairs_sha1", "scan"],
                                            [round(x / reps, 3) for x in kms_c]))}

    # ---- (b) S streams in blocks ----------------------------------------------------------------------------
    cap_b = int(S * (blk // 2048 + 2 + 10) * 8 * (FAN - 1) + S * FAN * FAN)
    b_hash = torch.empty((cap_b, 10), dtype=torch.uint8, device=dev)
    b_t1 = torch.empty(cap_b, dtype=torch.int32, device=dev)

    def run_b(sf, verify, n_push):
        emitted = np.zeros(S, np.int64)
        ok = True
        wall = 0.0
        c_base = torch.from_numpy(c_starts[:-1]).to(dev)
        for k in range(n_push):
            end = k == nb - 1
            t0 = time.perf_counter()
            r = sf.push_device(pool, offs + k * blk, np.full(S, blk, np.int64), end=end, out=(b_hash, b_t1))
            wall += time.perf_counter() - t0
            cnt = np.diff(r.starts)
            if verify:
                ok &= bool(np.all(emitted + cnt <= np.diff(c_starts)))
                n = int(r.starts[-1])
                if n and ok:
                    seg = torch.repeat_interleave(torch.arange(S, device=dev), torch.from_numpy(cnt).to(dev))
                    base = c_base + torch.from_numpy(emitted - r.starts[:-1]).to(dev)
                    idx = base[seg] + torch.arange(n, device=dev)
                    ok &= bool(torch.equal(c_hash[idx], r.hash)) and bool(torch.equal(c_t1[idx], r.t1))
            emitted += cnt
        if verify:
            ok &= bool(np.array_equal(emitted, np.diff(c_starts)))
        return wall, ok, int(emitted.sum())

    sf = StreamFingerprinter(fp, S, Fs=FS, fan_value=FAN, amp_min=AMP_MIN, compute=args.compute)
    run_b(sf, False, min(3, nb))                      # warm-up, then end every stream with an empty push
    sf.push_device(pool, offs, np.zeros(S, np.int64), end=True, out=(b_hash, b_t1))
    wall_b, ok, n_b = run_b(sf, True, nb)
    fp.timing(True)
    wall_b2, _, _ = run_b(sf, False, nb)
    kms_b, kl_b = sf.timing(False)
    sf.close()
    out["b_stream"] = {"streams": S, "seconds": L / FS, "block_samples": blk, "pushes": nb, "audio_s": audio_s,
                       "ms": round(wall_b * 1e3, 2), "ms_per_push": round(wall_b * 1e3 / nb, 3),
                       "audio_s_per_s": audio_s / wall_b, "hashes": n_b,
                       "ms_with_timers": round(wall_b2 * 1e3, 2),
                       "kernel_ms": dict(zip(["stft", "peaks_bitmap", "peaks_compact", "pairs_sha1", "scan",
                                              "stream_state_copies"], [round(x, 3) for x in kms_b])),
                       "launches": dict(zip(["stft", "peaks_bitmap", "peaks_compact", "pairs_sha1", "scan",
                                             "stream_state_copies"], kl_b)),
                       "k2_rows_per_new_row": round(k2_rows_per_new_row(blk, nb), 3)}
    out["b_over_c"] = round(out["b_stream"]["audio_s_per_s"] / out["c_batch"]["audio_s_per_s"], 3)
    out["identical_b_vs_c"] = ok

    # ---- (a) 2 streams, 8192-sample blocks -------------------------------------------------------------------
    sb, npush = args.small_block, args.small_pushes
    sf = StreamFingerprinter(fp, 2, Fs=FS, fan_value=FAN, amp_min=AMP_MIN, compute=args.compute)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(npush)]
    dev_ms, end_wall = [], []
    a_hash = torch.empty((1 << 20, 10), dtype=torch.uint8, device=dev)
    a_t1 = torch.empty(1 << 20, dtype=torch.int32, device=dev)
    two = offs[:2]
    for rnd in range(args.small_rounds + 2):
        for k in range(npush):
            end = k == npush - 1
            ev[k][0].record()
            t0 = time.perf_counter()
            sf.push_device(pool, two + k * sb, np.full(2, sb, np.int64), end=end, out=(a_hash, a_t1))
            w = time.perf_counter() - t0
            ev[k][1].record()
            if end and rnd >= 2:
                end_wall.append(w * 1e3)
        torch.cuda.synchronize()
        if rnd >= 2:
            dev_ms += [a.elapsed_time(b) for a, b in ev]
    sf.close()
    out["a_two_streams"] = {"block_samples": sb, "pushes_per_stream": npush, "rounds": args.small_rounds,
                            "device_ms_per_push_median": round(float(np.median(dev_ms)), 4),
                            "device_ms_per_push_p90": round(float(np.percentile(dev_ms, 90)), 4),
                            "last_push_to_final_hashes_ms_median": round(float(np.median(end_wall)), 4),
                            "k2_rows_per_new_row": round(k2_rows_per_new_row(sb, npush), 3)}
    fp.close()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
