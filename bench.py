#!/usr/bin/env python
"""bench.py — BASELINE.json's metric, both halves, in ONE JSON line.

M1 (top level): fingerprinted audio-seconds per second.  Workload = BASELINE.json configs[1]: batch fingerprinting of
1,000 synthetic 3-minute 44.1 kHz mono int16 tracks per GPU, fan 15, amp_min 10, 4096-point window, 50 % overlap.
A "step" is one pass of the whole path (K1 STFT->dB, K2 peaks, K3 pairs+SHA-1) over the batch.

  value : PCM already resident in HBM, digests left in HBM (CUDA events, max over ranks)
  e2e   : the same call through the public host API — pinned host PCM in, digests out to
          pinned host memory, H2D and D2H inside the timed region (+ the bare-copy ceiling of the same bytes)
  roofline : the dominant kernel (K1) against the measured HBM copy peak
  cpu_baseline / --impl reference : the reference's CPU algorithm (oracle port: numpy FFT + scipy.ndimage + hashlib,
          one process per track like fingerprint_directory's Pool) on this box's host cores, bounded sample.

M2 ("match"): match queries per second.  Workload = configs[3]/[4]: a 100,000-track synthetic index (~8e9 fingerprints)
and 10,000 concurrent 5 s queries, on N = 1/2/4/8 GPUs ("scaling": "strong": index and query set are fixed).  N = 1: one
index on one GPU.  N > 1: the index is sharded by HASH PREFIX (north_star: query hashes routed to their owning GPU over
NCCL, every vote tuple delivered to the query's owner, exact vote there) in two exact variants — `match.peer_memory`: the
shard scatters the tuples straight into the owner's HBM over NVLink peer memory (the exchange fused into the kernel);
`match.key_exchange`: vote keys through a second NCCL all-to-all — `match.value` is the faster one, and, next to it, by
TRACK (`match.track_sharded`, SURVEY §8e's alternative).  Identity is checked inside the run: hash-prefix == track-sharded for
every query, a 256-query subsample against ONE index holding all rows on rank 0, and a checksum of all results that is
the same number at every N.

Launch: python bench.py [--gpus N --steps K --warmup W --dump-outputs DIR]; for N>1 under torchrun.
"""
from __future__ import annotations

import argparse
import datetime
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FS = 44100
TRACK_SAMPLES = 7_938_000          # 3 min
FAN, AMP_MIN = 15, 10
K1_BYTES_PER_AUDIO_S = 264_684     # SURVEY §8d: 88 200 B PCM read + 176 484 B float32 spectrogram write
FRAMES_PER_TRACK = 3874            # 3 min @ 44.1 kHz
CLIP_FRAMES = 106                  # 5 s


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--tracks", type=int, default=1000, help="tracks per GPU per step")
    ap.add_argument("--track-samples", type=int, default=TRACK_SAMPLES)
    ap.add_argument("--compute", default="f64", choices=["f64", "f32"])
    ap.add_argument("--chunk-frames", type=int, default=262144)
    ap.add_argument("--host-pool-tracks", type=int, default=250)
    ap.add_argument("--cpu-sample-tracks", type=int, default=0, help="0 = 4 per host core")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-digest-table", action="store_true", help="K3 hashes every pair instead of gathering from the table")
    ap.add_argument("--no-fingerprint", action="store_true", help="skip M1 (development runs of the match leg)")
    # M2
    ap.add_argument("--no-match", action="store_true")
    ap.add_argument("--match-tracks", type=int, default=100_000, help="tracks in the whole index")
    ap.add_argument("--match-rows-per-track", type=int, default=80_000)
    ap.add_argument("--match-queries", type=int, default=10_000, help="queries per step over all ranks")
    ap.add_argument("--match-topn", type=int, default=3)
    ap.add_argument("--match-gen-batch", type=int, default=500, help="tracks generated per batch")
    ap.add_argument("--match-flush-rows", type=int, default=250_000_000, help="pending rows per finalize (merge)")
    ap.add_argument("--match-pass-keys", type=int, default=600_000_000, help="N>1: vote keys a rank receives per pass")
    ap.add_argument("--match-check-queries", type=int, default=256, help="N>1: subsample checked against one full index")
    ap.add_argument("--match-cpu-tracks", type=int, default=2714, help="index size of the CPU baseline (configs[2])")
    ap.add_argument("--no-peer", action="store_true", help="N>1: skip the peer-memory (fused exchange) variant of the hash-prefix path")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float32/float64, "
                         "a fixed seeded sample where the whole does not fit 64 MB; N>1: rank 0's tracks, every query)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
    return args


# ------------------------------------------------------------------------------------------
# synthetic tracks (SURVEY.md §8d Config 2 recipe), generated on the GPU
# ------------------------------------------------------------------------------------------
def synth_tracks_gpu(dev, first_seed: int, n_tracks: int, n_samples: int, out):
    """6 voices, note change every 11 025 samples, pitch 110*2^(U{0..59}/12), amplitude
    U(500, 4000), harmonics (1, 1/2, 1/4), + N(0, 200^2) noise, clipped to int16."""
    import torch
    seg = 11025
    nseg = -(-n_samples // seg)
    t = torch.arange(n_samples, device=dev, dtype=torch.float64) / FS
    seg_idx = torch.arange(n_samples, device=dev) // seg
    for i in range(n_tracks):
        g = torch.Generator(device=dev)
        g.manual_seed(first_seed + i)
        x = torch.zeros(n_samples, device=dev, dtype=torch.float64)
        semis = torch.randint(0, 60, (6, nseg), device=dev, generator=g)
        amps = torch.rand((6, nseg), device=dev, generator=g, dtype=torch.float64) * 3500 + 500
        for v in range(6):
            f = 110.0 * torch.pow(2.0, semis[v].double() / 12.0)
            ph = (2 * np.pi) * f[seg_idx] * t
            a = amps[v][seg_idx]
            x += a * (torch.sin(ph) + 0.5 * torch.sin(2 * ph) + 0.25 * torch.sin(3 * ph))
        x += torch.randn(n_samples, device=dev, generator=g, dtype=torch.float64) * 200
        out[i].copy_(torch.clamp(torch.round(x), -32768, 32767).to(torch.int16))


# ------------------------------------------------------------------------------------------
# CPU baseline: the oracle port, one process per track (fingerprint_directory's Pool)
# ------------------------------------------------------------------------------------------
_CPU_TRACKS = None
_CPU_TABLE = None
_CPU_QUERIES = None


def _cpu_worker(i):
    from oracle import sia_oracle as O
    hs = O.fingerprint(_CPU_TRACKS[i], Fs=FS, fan_value=FAN, amp_min=AMP_MIN)
    return len(hs)


def cpu_reference_run(tracks, procs: int, steps: int = 1, warmup: int = 0):
    """Returns (audio_s_per_s, seconds_per_step, hashes) timing `steps` passes over `tracks`."""
    import multiprocessing as mp
    global _CPU_TRACKS
    _CPU_TRACKS = tracks
    ctx = mp.get_context("fork")
    audio_s = sum(len(t) for t in tracks) / FS
    with ctx.Pool(procs) as pool:
        for _ in range(warmup):
            list(pool.imap_unordered(_cpu_worker, range(min(len(tracks), procs))))
        t0 = time.perf_counter()
        nh = 0
        for _ in range(steps):
            nh = sum(pool.imap_unordered(_cpu_worker, range(len(tracks))))
        dt = (time.perf_counter() - t0) / max(steps, 1)
    return audio_s / dt, dt, nh


def _cpu_match_worker(i):
    """return_matches + align_matches of the reference (recognizer.py:222-338, oracle port) for one query."""
    from oracle import sia_oracle as O
    q = _CPU_QUERIES[i]
    matches, dedup = O.return_matches(_CPU_TABLE, q)
    res = O.align_matches(_CPU_TABLE, matches, dedup, len(q), 3) if matches else []
    return len(matches), (res[0]["song_id"] if res else 0)


def cpu_match_run(table, queries, procs: int):
    """queries/s of the oracle port over `queries` (sets of (hex20, offset)) with a Pool of `procs` forked workers that
    share the table copy-on-write (the reference opens one DB connection per process)."""
    import multiprocessing as mp
    global _CPU_TABLE, _CPU_QUERIES
    _CPU_TABLE, _CPU_QUERIES = table, queries
    ctx = mp.get_context("fork")
    with ctx.Pool(procs) as pool:
        list(pool.imap_unordered(_cpu_match_worker, range(min(len(queries), procs))))     # warm the workers
        t0 = time.perf_counter()
        out = list(pool.imap_unordered(_cpu_match_worker, range(len(queries))))
        dt = time.perf_counter() - t0
    return len(queries) / dt, dt, out


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        """Start of the timed region: only samples taken from here on are reported."""
        self.first = len(self.lines)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for ln in self.lines[getattr(self, "first", 0):]:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def bind_to_gpu_numa(gpu_index: int):
    """Multi-GPU runs: pin this rank to the CPUs NVML lists as local to its GPU, so the pinned host buffers of
    the e2e leg are first-touched on the GPU's own NUMA node (8 ranks sharing one socket's memory and PCIe
    root halve each other's copy bandwidth).  Returns the number of CPUs bound, or None if NVML cannot tell."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, m in enumerate(words) for b in range(64) if (int(m) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def per_kernel_roofline(kernel_ms, audio_s, n_hashes, peak_gbs, digest_table):
    """north_star: achieved HBM GB/s of EVERY kernel of the fingerprint path against the measured peak, from the
    event-timed kernel times of the timed region.  Algorithmic bytes are SURVEY §8(d)'s (K1 264 684 B and K2 176 484 B per
    audio-second, K3 14 B written per hash); K3 is not bound by its algorithmic bytes (SHA-1 mode: integer ALU; table
    mode: one random 32-byte sector per hash), so its sector-granular rate is given next to it.  Pure arithmetic:
    ``kernel_ms`` = {name: ms per step}, ``audio_s`` / ``n_hashes`` per step and GPU."""
    frames = audio_s * FS / 2048.0
    rows = [
        ("stft_db(K1)", K1_BYTES_PER_AUDIO_S * audio_s, "fp64 pipe (float64 butterflies); bytes are streamed once"),
        ("peaks_bitmap(K2)", 176_484 * audio_s, "latency / ALU (FMNMX on the half-rate pipe at 8 warps per SM)"),
        ("peaks_compact(K2)", 352.0 * frames, "trivial: 88-word bitmap row per frame -> ordered peak lists"),
        ("pairs_sha1(K3)", 14.0 * n_hashes,
         "random 32-byte sectors of the digest table" if digest_table else "integer ALU (80 SHA-1 rounds per hash)"),
    ]
    out = {}
    for name, nbytes, bound in rows:
        ms = float(kernel_ms.get(name) or 0.0)
        gbs = nbytes / (ms * 1e-3) / 1e9 if ms > 0 else None
        out[name] = {"ms_per_step": ms, "algorithmic_bytes_per_step": nbytes, "achieved_gbs": gbs,
                     "frac_of_hbm_peak": (gbs / peak_gbs) if gbs else None, "limited_by": bound}
    k3 = out["pairs_sha1(K3)"]
    if k3["achieved_gbs"]:
        ms = k3["ms_per_step"]
        k3["hashes_per_second"] = n_hashes / (ms * 1e-3)
        if digest_table:
            sect = (14.0 + 32.0) * n_hashes
            k3["sector_granular_bytes_per_step"] = sect
            k3["sector_granular_gbs"] = sect / (ms * 1e-3) / 1e9
            k3["sector_granular_frac_of_hbm_peak"] = k3["sector_granular_gbs"] / peak_gbs
    return out


# --dump-outputs: bytes of data per group of row-aligned outputs; 63 MB in all, so that with the .npy headers the files
# stay under 64 MB
DUMP_BYTES = {"fingerprint": 44_000_000, "fingerprint_tracks": 4_000_000, "match": 15_000_000}


def dump_rows(out_dir, group, columns, seed):
    """Writes ``out_dir/<group>_<name>.npy`` for every column (a numpy array or a tensor, rows first, all with the same
    number of rows) and ``<group>_index.npy``, the row numbers written: every row when they fit the group's share of
    DUMP_BYTES, else a fixed sample (``seed``) of as many rows as fit, in row order.  8- and 16-bit integers are
    written as float32, everything else as float64: both hold the values exactly."""
    def out_dtype(c):
        return np.float32 if c.dtype.itemsize <= 2 else np.float64

    def row_bytes(c):
        return int(np.prod(c.shape[1:], dtype=np.int64)) * np.dtype(out_dtype(c)).itemsize

    n = len(next(iter(columns.values())))
    k = max(1, DUMP_BYTES[group] // (8 + sum(row_bytes(c) for c in columns.values())))
    idx = np.arange(n) if n <= k else np.sort(np.random.default_rng(seed).choice(n, k, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"{group}_index.npy"), idx.astype(np.float64))
    for name, c in columns.items():
        if isinstance(c, np.ndarray):
            rows = c[idx]
        else:
            import torch
            rows = c[torch.from_numpy(idx).to(c.device)].cpu().numpy()
        np.save(os.path.join(out_dir, f"{group}_{name}.npy"), rows.astype(out_dtype(c)))


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ==========================================================================================
# M1: fingerprinting
# ==========================================================================================
def fingerprint_leg(args, rank, world, local_rank, dev, config):
    import torch
    import torch.distributed as dist
    from shazam_b200 import _native as N
    from shazam_b200.fingerprinter import Fingerprinter
    audio_s_per_track = args.track_samples / FS
    host_cpus = bind_to_gpu_numa(local_rank) if world > 1 else None

    B, L = args.tracks, args.track_samples
    stride = (L + 7) // 8 * 8
    d_pcm = torch.empty(B * stride, dtype=torch.int16, device=dev)
    rows = d_pcm.view(B, stride)
    t_gen = time.perf_counter()
    synth_tracks_gpu(dev, 1_000_000 * rank, B, L, [rows[i, :L] for i in range(B)])
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t_gen
    starts = np.arange(B, dtype=np.int64) * stride
    lens = np.full(B, L, np.int64)

    fp = Fingerprinter(local_rank, max_chunk_frames=args.chunk_frames)
    if not args.no_digest_table:
        fp.digest_table(True)
    p = fp.params(Fs=FS, fan_value=FAN, amp_min=AMP_MIN, compute=args.compute)
    frames_per_track = N.num_frames(L)
    cap = int(B * frames_per_track * 5.5 * (FAN - 1))           # ~4 peaks/frame on this signal class
    d_hash = torch.empty((cap, 10), dtype=torch.uint8, device=dev)
    d_t1 = torch.empty(cap, dtype=torch.int32, device=dev)
    audio_s = B * audio_s_per_track

    def step_device():
        return fp.fingerprint_device(d_pcm, starts, lens, p, out=(d_hash, d_t1))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        res = step_device()
    n_hashes = len(res.t1)
    fp.timing(True)                                   # reset + enable per-kernel CUDA-event timers
    barrier()
    sampler.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        last = step_device()
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop()
    kms, klaunch = fp.timing(False)
    if args.dump_outputs and rank == 0:
        dump_rows(args.dump_outputs, "fingerprint", {"hash": last.hash, "t1": last.t1}, seed=1)
        dump_rows(args.dump_outputs, "fingerprint_tracks", {"starts": last.starts}, seed=2)
    t_dev = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
    ms_step = float(t_dev.item()) / args.steps
    value = world * audio_s / (ms_step * 1e-3)

    # ---- end to end through the host API ------------------------------------------------
    e2e = None
    if not args.no_e2e:
        pool = min(args.host_pool_tracks, B)
        h_pcm = torch.empty(pool * stride, dtype=torch.int16).pin_memory()
        h_pcm.copy_(d_pcm[: pool * stride])
        h_starts = (np.arange(B, dtype=np.int64) % pool) * stride      # the batch cycles over the pinned pool
        h_hash = torch.empty((cap, 10), dtype=torch.uint8).pin_memory()
        h_t1 = torch.empty(cap, dtype=torch.int32).pin_memory()

        def step_host():
            return fp.fingerprint_host(h_pcm, h_starts, lens, p, out=(h_hash, h_t1))
        for _ in range(max(min(args.warmup, 2), 1)):
            r = step_host()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            r = step_host()
        barrier()
        dt = (time.perf_counter() - t0) / args.steps
        n_out = len(r.t1)
        # the ceiling of this leg: the same bytes as bare concurrent copies (H2D of the PCM on one stream, D2H of the
        # digests on another), every rank at once — what the host's PCIe / memory complex gives N GPUs together
        s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        d_in = torch.empty(pool * stride, dtype=torch.int16, device=dev)
        out_bytes = n_out * 14
        h_out = h_hash.view(-1)[:min(out_bytes, h_hash.numel())]
        d_out = d_hash.view(-1)[:h_out.numel()]
        reps_in = -(-B // pool)

        def copy_step():
            with torch.cuda.stream(s_in):
                for _ in range(reps_in):
                    d_in.copy_(h_pcm, non_blocking=True)
            with torch.cuda.stream(s_out):
                h_out.copy_(d_out, non_blocking=True)
            s_in.synchronize(); s_out.synchronize()
        copy_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            copy_step()
        barrier()
        dt_copy = (time.perf_counter() - t0) / args.steps
        t_e = torch.tensor([dt, dt_copy], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
        dt, dt_copy = (float(x) for x in t_e.tolist())
        copied = reps_in * pool * stride * 2 + h_out.numel()
        e2e = {"value": world * audio_s / dt, "unit": "audio-s/s", "ms_per_step": dt * 1e3,
               "h2d_bytes_per_step": int(B * L * 2), "d2h_bytes_per_step": int(n_out * 14 + (B + 1) * 8),
               "api": "Fingerprinter.fingerprint_host -> sia_fingerprint_batch_host (pinned host PCM in, "
                      "digests + offsets out to pinned host memory)",
               "host_pool_tracks": pool,
               "copy_ceiling": {"value": world * audio_s / dt_copy, "unit": "audio-s/s", "ms_per_step": dt_copy * 1e3,
                                "gb_per_s_per_gpu": copied / dt_copy / 1e9,
                                "what": "bare concurrent cudaMemcpyAsync of the same H2D + D2H bytes on two streams, all "
                                        "ranks at once, max over ranks"},
               "frac_of_copy_ceiling": dt_copy / dt}
        if host_cpus:
            e2e["host_cpus_bound_per_rank"] = host_cpus
        del h_pcm, h_hash, h_t1, d_in

    out = None
    if rank == 0:
        # ---- roofline of the dominant kernel (K1) ----------------------------------------------
        peak, peak_src = measured_peak_gbs()
        k1_ms = kms[0]
        k1_launches = max(klaunch[0], 1)
        algo_bytes_per_launch = K1_BYTES_PER_AUDIO_S * audio_s * args.steps / k1_launches
        achieved = algo_bytes_per_launch / (k1_ms / k1_launches * 1e-3) / 1e9 if k1_ms > 0 else None
        names = ["stft_db(K1)", "peaks_bitmap(K2)", "peaks_compact(K2)", "pairs_sha1(K3)", "scans"]
        kernel_ms = {n: round(m / args.steps, 4) for n, m in zip(names, kms)}
        roofline = {"bound": "hbm", "kernel": "stft_db_kernel<%s>" % ("double" if args.compute == "f64" else "float"),
                    "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": (achieved / peak) if achieved else None, "traffic": None, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": algo_bytes_per_launch, "launches_timed": k1_launches,
                    "avg_launch_ms": k1_ms / k1_launches, "kernel_ms_per_step": kernel_ms,
                    "share_of_step": round(k1_ms / max(sum(kms), 1e-9), 4)}
        try:
            roofline["per_kernel"] = per_kernel_roofline(kernel_ms, audio_s, n_hashes, peak, not args.no_digest_table)
        except Exception as e:      # an explanatory table must never cost the line
            roofline["per_kernel"] = {"error": f"{type(e).__name__}: {e}"}
        if args.compute == "f64" and k1_ms > 0:
            # what actually bounds K1: the FP64 pipe (+ the integer pipe, DESIGN.md §5).  854 DP arithmetic instructions
            # per thread and frame (static SASS count: 455 DADD, 249 DFMA, 150 DMUL) x 4 warps = 3 416 DP warp
            # instructions per frame; a B200 SM sub-partition issues one DP warp instruction every 2 cycles
            # (tools/ubench/fp64_rate.cu: 2.13) -> 148 x 4 / 2 per clock at the sampled SM clock
            dp_warp_inst = 3416.0 * B * frames_per_track * args.steps
            clk = (clocks or {}).get("sm_mhz") or 1965.0
            dp_peak = 148 * 4 / 2 * clk * 1e6
            roofline["fp64_pipe"] = {"achieved_warp_inst_per_s": dp_warp_inst / (k1_ms * 1e-3), "peak_warp_inst_per_s": dp_peak,
                                     "frac": dp_warp_inst / (k1_ms * 1e-3) / dp_peak,
                                     "note": "K1 computes in float64 (1e-3 dB bound on every bin); 3416 DP warp instructions "
                                             "per frame (SASS), DP issue rate 1 per 2 cycles per sub-partition (tools/ubench)"}
        prof = os.path.join(ROOT, "profiles", "k1_traffic.json")
        if os.path.exists(prof):
            try:
                per_frame = json.load(open(prof)).get("dram_bytes_per_frame")
                frames = B * frames_per_track * args.steps / k1_launches
                roofline["traffic"] = per_frame * frames if per_frame else None
                roofline["traffic_source"] = "profiles/k1_traffic.json (ncu --set full, dram read+write per frame) x frames per launch"
            except Exception:
                pass

        # ---- CPU baseline on a bounded sample of the same tracks ----------------------------------
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            procs = os.cpu_count() or 1
            ntr = args.cpu_sample_tracks or min(B, 4 * procs)
            tracks = [rows[i, :L].cpu().numpy() for i in range(ntr)]
            v, dt, nh = cpu_reference_run(tracks, procs)
            cpu = {"value": v, "unit": "audio-s/s", "cores": procs, "kind": "port",
                   "sample": f"first {ntr} of the {B} tracks ({ntr * audio_s_per_track:.0f} audio-s, {dt:.1f} s wall), "
                             f"oracle port of the reference CPU path, Pool({procs}) one task per track"}
            try:                    # SURVEY §8(d): the one-process figure next to the Pool's
                v1, dt1, _ = cpu_reference_run(tracks[:2], 1)
                cpu["one_process"] = {"value": v1, "unit": "audio-s/s", "cores": 1,
                                      "sample": f"first {len(tracks[:2])} tracks, {dt1:.1f} s wall"}
            except Exception as e:
                cpu["one_process"] = {"error": f"{type(e).__name__}: {e}"}

        out = {"metric": "fingerprint_audio_seconds_per_second", "value": value, "unit": "audio-s/s", "n_gpus": world,
               "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
               "scaling": "weak", "vs_baseline": None, "dtype": args.compute, "data": "synthetic",
               "config": config, "clocks": clocks, "e2e": e2e,
               "gpu_launches": int(sum(klaunch)), "hashes_per_step_per_gpu": int(n_hashes),
               "roofline": roofline, "cpu_baseline": cpu, "synth_seconds": round(t_gen, 1)}
    fp.close()
    del d_pcm, rows, d_hash, d_t1
    torch.cuda.empty_cache()
    return out


# ==========================================================================================
# M2: matching
# ==========================================================================================
def batch_peaks(dev, batch_id: int, n_tracks: int, peaks_per_track: int):
    """Deterministic peak lists of the tracks of one generation batch: (t[B,P], f[B,P]) sorted by (t, f); the bins are
    skewed towards low frequencies, so the hash popularity has the skew of the 8.4e8-value pre-image space."""
    import torch
    g = torch.Generator(device=dev)
    g.manual_seed(77_000 + batch_id)
    t = torch.randint(0, FRAMES_PER_TRACK, (n_tracks, peaks_per_track), device=dev, generator=g)
    u = torch.rand((n_tracks, peaks_per_track), device=dev, generator=g)
    f = torch.clamp((2049 * u * u).long(), max=2048)
    key, _ = torch.sort(t * 4096 + f, dim=1)
    return (key // 4096).to(torch.int32), (key % 4096).to(torch.int32)


def batch_queries(dev, batch_id: int, pt, pf, rows, t0s):
    """5 s windows (106 frames) of indexed tracks with 30 % of the peaks dropped and as many random peaks added, all
    queries of one generation batch at once.  rows / t0s: track row inside the batch and window start per query.
    Returns (peak_t, peak_f, lengths) with every query's peaks in (t, f) order, times relative to the window."""
    import torch
    g = torch.Generator(device=dev)
    g.manual_seed(4_321_000 + batch_id)
    rows_t = torch.as_tensor(rows, device=dev, dtype=torch.long)
    t0 = torch.as_tensor(t0s, device=dev, dtype=torch.int32)[:, None]
    nq = rows_t.numel()
    qt, qf = pt[rows_t], pf[rows_t]                                   # [nq, P]
    inwin = (qt >= t0) & (qt < t0 + CLIP_FRAMES)
    keep = inwin & (torch.rand(qt.shape, device=dev, generator=g) < 0.7)
    n_drop = (inwin & ~keep).sum(1)
    width = int(n_drop.max().item()) if nq else 0
    nt_ = torch.randint(0, CLIP_FRAMES, (nq, width), device=dev, generator=g, dtype=torch.int32)
    nf_ = torch.randint(0, 2049, (nq, width), device=dev, generator=g, dtype=torch.int32)
    nvalid = torch.arange(width, device=dev)[None, :] < n_drop[:, None]
    qid = torch.arange(nq, device=dev, dtype=torch.long)[:, None]
    k1 = (qid << 32) | ((qt - t0).long() << 12) | qf.long()
    k2 = (qid << 32) | (nt_.long() << 12) | nf_.long()
    key = torch.unique(torch.cat([k1[keep], k2[nvalid]]))             # sorted by (query, t, f), duplicates dropped
    lens = torch.bincount(key >> 32, minlength=nq)
    return ((key >> 12) & 0xfffff).to(torch.int32), (key & 0xfff).to(torch.int32), lens


def results_digest(qids, res, topn):
    """sha256 over (query id, nres, song, diff, count, rows) of all queries in query-id order."""
    order = np.argsort(qids, kind="stable")
    cols = [np.asarray(qids, np.int64)[order], res[4][order].astype(np.int64)]
    cols += [res[k][order].astype(np.int64).reshape(len(order), topn) for k in range(4)]
    blob = np.concatenate([c.reshape(len(order), -1) for c in cols], axis=1)
    return hashlib.sha256(np.ascontiguousarray(blob).tobytes()).hexdigest()


def match_leg(args, rank, world, local_rank, dev):
    import torch
    import torch.distributed as dist
    from shazam_b200.database import FingerprintIndex
    from shazam_b200.distributed import CudaShard, ShardedIndex, TrackShardedIndex
    from shazam_b200.fingerprinter import Fingerprinter

    T, R, Q, topn, GB = args.match_tracks, args.match_rows_per_track, args.match_queries, args.match_topn, args.match_gen_batch
    P = max(2, R // (FAN - 1))
    n_batches = -(-T // GB)
    os.environ["SIA_PEAKS_PER_FRAME_CAP"] = str(max(32, -(-(GB * P) // 4096) + 1))    # K3 workspace: one batch of peaks
    fp = Fingerprinter(local_rank, max_chunk_frames=4096)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- the query set (fixed for every N): track + window start per query ---------------------------------------
    rng = np.random.default_rng(5)
    q_tracks = rng.integers(0, T, Q)
    q_start = rng.integers(0, FRAMES_PER_TRACK - CLIP_FRAMES, Q)
    by_batch = {}
    for qi in range(Q):
        by_batch.setdefault(int(q_tracks[qi]) // GB, []).append(qi)

    rows_est = T * R
    own_batches = [b for b in range(n_batches) if b % world == rank]
    own_tracks = sum(min(GB, T - b * GB) for b in own_batches)
    if world == 1:
        single = FingerprintIndex(local_rank, int(rows_est * 1.01) + (1 << 20))
        hashed = tracked = None
    else:
        single = None
        hashed = ShardedIndex(CudaShard(local_rank, int(rows_est / world * 1.06) + (1 << 22)), rank=rank, world=world)
        tracked = TrackShardedIndex(CudaShard(local_rank, int(own_tracks * R * 1.01) + (1 << 20)), rank=rank, world=world)

    # ---- build (and the queries of the batches this rank generates) ---------------------------------------------
    barrier()
    t_build = time.perf_counter()
    q_pt, q_pf, q_len, q_ids = [], [], [], []
    gen_rows = pending = 0
    rounds = -(-n_batches // world)
    for rnd in range(rounds):
        b = rnd * world + rank
        if b < n_batches:
            nt = min(GB, T - b * GB)
            pt, pf = batch_peaks(dev, b, nt, P)
            tps = torch.arange(nt + 1, device=dev, dtype=torch.int64) * P
            h, t1, ths = fp.pairs_sha1(pt.reshape(-1), pf.reshape(-1), tps, FAN)
            songs = torch.repeat_interleave(torch.arange(nt, device=dev, dtype=torch.int32) + (b * GB + 1), ths[1:] - ths[:-1])
            gen_rows += h.shape[0]
            if b in by_batch:
                qis = by_batch[b]
                a, c, ln = batch_queries(dev, b, pt, pf, [int(q_tracks[i]) - b * GB for i in qis], [int(q_start[i]) for i in qis])
                q_pt.append(a); q_pf.append(c); q_len.append(ln); q_ids += qis
        else:
            h = torch.empty((0, 10), dtype=torch.uint8, device=dev)
            t1 = torch.empty(0, dtype=torch.int32, device=dev)
            songs = torch.empty(0, dtype=torch.int32, device=dev)
        if world == 1:
            single.insert_rows(songs, h, t1)
        else:
            tracked.insert(songs, h, t1)
            hashed.insert(songs, h, t1)         # collective: rows travel to the shard that owns their hash
        pending += GB * R                        # the same on every rank, so the collective finalizes line up
        del h, t1, songs
        if pending >= args.match_flush_rows or rnd == rounds - 1:
            pending = 0
            if world == 1:
                rows_total = single.finalize()
            else:
                tracked.finalize()
                rows_total = hashed.finalize()
    barrier()
    t_build = time.perf_counter() - t_build
    if world == 1:
        n_keys = single.keys
    else:
        kk = torch.tensor([hashed.backend.index.keys], dtype=torch.int64, device=dev)
        dist.all_reduce(kk)
        n_keys = int(kk.item())

    # ---- this rank's queries -> hashes (K3) -------------------------------------------------------------------
    n_q_local = len(q_ids)
    if n_q_local:
        lens = torch.cat(q_len)
        tps = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), torch.cumsum(lens, 0)])
        qh, qt1, qths = fp.pairs_sha1(torch.cat(q_pt), torch.cat(q_pf), tps, FAN)
        q_starts = qths.cpu().numpy()
    else:
        qh = torch.empty((0, 10), dtype=torch.uint8, device=dev); qt1 = torch.empty(0, dtype=torch.int32, device=dev)
        q_starts = np.zeros(1, np.int64)
    fp.close()
    del q_pt, q_pf, q_len
    torch.cuda.empty_cache()

    # ---- N > 1: size the passes of the hash-prefix path (vote keys a rank receives per pass) ---------------------
    qp = 4096
    if world > 1:
        cal = 32
        sub = min(cal, n_q_local)
        hashed.query(qh[:q_starts[sub]], qt1[:q_starts[sub]], q_starts[:sub + 1], topn, queries_per_pass=cal)
        per_q_slot = max(1.0, hashed.key_cap / cal)
        qp = int(max(8, min(4096, args.match_pass_keys / (world * per_q_slot))))
        hashed.key_cap = int(per_q_slot * qp * 1.1) + 64
        hashed.retries = 0

    def step_main():
        if world == 1:
            return single.query_batch(qh, qt1, q_starts, topn)
        return hashed.query(qh, qt1, q_starts, topn, queries_per_pass=qp)

    def timed(fn, steps, warmup):
        for _ in range(max(warmup, 1)):
            r = fn()
        barrier()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        evs[0].record()
        for i in range(steps):
            r = fn()
            evs[i + 1].record()
        barrier()
        per = [evs[i].elapsed_time(evs[i + 1]) for i in range(steps)]
        timed.last_per_step = [round(x, 2) for x in per]
        ms = torch.tensor([evs[0].elapsed_time(evs[-1]) / steps, float(np.median(per))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return r, float(ms[0].item()), float(ms[1].item())

    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.mark()
    res, ms_step, ms_med = timed(step_main, args.steps, max(args.warmup, 3))
    per_step_ms = timed.last_per_step
    clocks = sampler.stop()
    lookup_ms = vote_ms = None
    qstats = None
    if world == 1:
        lookup_ms, vote_ms = single.query_timing()
        qstats = single.query_batch(qh, qt1, q_starts, topn, want_stats=True)[5]
    res_np = [t.cpu().numpy() for t in res]

    track_line, hash_eq_track = None, None
    pass_ms = None
    peer_line = None
    hp = None
    if world > 1:
        retries = hashed.retries
        os.environ["SIA_DIST_TIMING"] = "1"           # stage times of one more step (synchronising: not a timed one)
        step_main()
        pass_ms = hashed.last_pass_ms
        os.environ.pop("SIA_DIST_TIMING", None)
        # ---- the same hash-prefix pass with the second exchange fused into the scatter kernel (NVLink peer memory) ----
        if not args.no_peer:
            try:
                del res
                hashed.backend.index.trim()       # the key path's scratch (vote tables, key buffers of the build): tens of GB
                torch.cuda.empty_cache()
                hp = ShardedIndex(hashed.backend, rank=rank, world=world, exchange="peer")
                hp._max_song, hp.entry_cap = hashed._max_song, hashed.entry_cap
                cal = 32
                sub = min(cal, n_q_local)
                hp.query(qh[:q_starts[sub]], qt1[:q_starts[sub]], q_starts[:sub + 1], topn, queries_per_pass=cal)   # sizes the regions
                hp.region_cap = int(hp.region_cap / cal * qp * 1.1) + (1 << 20)
                hp.retries = 0
                res_p, ms_p, ms_p_med = timed(lambda: hp.query(qh, qt1, q_starts, topn, queries_per_pass=qp), args.steps, max(args.warmup, 3))
                eqp = torch.tensor([int(all(np.array_equal(a, b.cpu().numpy()) for a, b in zip(res_np, res_p)))], device=dev)
                dist.all_reduce(eqp, op=dist.ReduceOp.MIN)
                os.environ["SIA_DIST_TIMING"] = "1"
                hp.query(qh, qt1, q_starts, topn, queries_per_pass=qp)
                os.environ.pop("SIA_DIST_TIMING", None)
                peer_line = {"value": Q / (ms_p * 1e-3), "unit": "queries/s", "ms_per_step": ms_p, "ms_per_step_median": ms_p_med,
                             "equals_key_exchange_results": bool(eqp.item()), "retries_in_timed_steps": hp.retries,
                             "passes_redone_with_the_key_exchange": hp.peer_fallbacks, "region_slots_per_rank": hp.region_cap,
                             "last_pass_stage_ms_rank0": hp.last_pass_ms,
                             "what": "hash prefix, second exchange fused into the scatter kernel: the shard owning the hashes writes "
                                     "the vote tuples of its posting runs straight into the (query, partition) regions in the query "
                                     "owner's HBM (peer stores + peer atomicAdd over NVLink, CUDA IPC mappings); collectives left: "
                                     "all-to-all of the query entries, one all-reduce of the per-query tuple counts, two tiny "
                                     "all-reduces (barrier + flags)"}
            except Exception as e:      # e.g. no peer access on this box: keep the key-exchange line
                import traceback
                traceback.print_exc()
                peer_line = {"error": f"{type(e).__name__}: {str(e)[:300]}"}
        res_t, ms_t, ms_t_med = timed(lambda: tracked.query(qh, qt1, q_starts, topn), args.steps, max(args.warmup, 3))
        res_t_np = [t.cpu().numpy() for t in res_t]
        del res_t
        tracked.backend.index.trim()
        torch.cuda.empty_cache()
        eq = torch.tensor([int(all(np.array_equal(a, b) for a, b in zip(res_np, res_t_np)))], device=dev)
        dist.all_reduce(eq, op=dist.ReduceOp.MIN)
        hash_eq_track = bool(eq.item())
        track_line = {"value": Q / (ms_t * 1e-3), "unit": "queries/s", "ms_per_step": ms_t, "ms_per_step_median": ms_t_med,
                      "what": "index sharded by track (every rank holds all rows of its songs), queries all-gathered, exact "
                              "local vote, G x topn candidates merged"}

    # ---- end to end: query hashes start in pinned host memory, results end in host memory, every step ----------
    h_qh = qh.cpu().pin_memory(); h_qt1 = qt1.cpu().pin_memory()

    # N > 1: through the variant of the hash-prefix path that gives `value` (every rank takes the same branch: the
    # comparison is made on all-reduced times)
    use_peer = bool(world > 1 and peer_line and peer_line.get("equals_key_exchange_results") and peer_line.get("ms_per_step", 1e30) < ms_step)
    sharded_q = hp if use_peer else hashed

    def step_host():
        d_h = h_qh.to(dev, non_blocking=True); d_t = h_qt1.to(dev, non_blocking=True)
        r = single.query_batch(d_h, d_t, q_starts, topn) if world == 1 else sharded_q.query(d_h, d_t, q_starts, topn, queries_per_pass=qp)
        return [x.cpu() for x in r[:5]]
    step_host()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res_host = step_host()
    barrier()
    e2e_s = torch.tensor([(time.perf_counter() - t0) / args.steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_s = float(e2e_s.item())
    io = torch.tensor([h_qh.numel() + 4 * h_qt1.numel(), sum(x.numel() * 4 for x in res_host)], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(io)
    if hp is not None:
        hp.close_peers()
        hp = None
        torch.cuda.empty_cache()
    e2e = {"value": Q / e2e_s, "unit": "queries/s", "ms_per_step": e2e_s * 1e3,
           "h2d_bytes_per_step": int(io[0].item()), "d2h_bytes_per_step": int(io[1].item()),
           "api": "pinned host (digest, offset) arrays -> FingerprintIndex.query_batch / ShardedIndex.query -> results in host memory",
           "variant": "one index" if world == 1 else ("hash prefix over peer memory" if use_peer else "hash prefix, key exchange")}

    # ---- gather every rank's results (small) for the accuracy, the checksum and the n-th-count statistics ----------
    mine = {"qids": q_ids, "res": res_np, "hashes": int(qt1.numel()), "rows": gen_rows}
    if world > 1:
        allr = [None] * world
        dist.all_gather_object(allr, mine)
    else:
        allr = [mine]

    # ---- N > 1: a subsample of rank 0's queries against ONE index holding every row -----------------------------
    subsample = None
    if world > 1 and args.match_check_queries > 0:
        tracked.backend.close()
        del tracked
        hashed.backend.index.trim()              # build / vote scratch of the shard: rank 0 needs the room
        torch.cuda.empty_cache()
        if rank == 0:
            try:
                os.environ["SIA_PEAKS_PER_FRAME_CAP"] = str(max(32, -(-(GB * P) // 4096) + 1))
                fp2 = Fingerprinter(local_rank, max_chunk_frames=4096)
                full = FingerprintIndex(local_rank, int(rows_est * 1.01) + (1 << 20))
                pend = 0
                for b in range(n_batches):
                    nt = min(GB, T - b * GB)
                    pt, pf = batch_peaks(dev, b, nt, P)
                    tps = torch.arange(nt + 1, device=dev, dtype=torch.int64) * P
                    h, t1, ths = fp2.pairs_sha1(pt.reshape(-1), pf.reshape(-1), tps, FAN)
                    songs = torch.repeat_interleave(torch.arange(nt, device=dev, dtype=torch.int32) + (b * GB + 1), ths[1:] - ths[:-1])
                    full.insert_rows(songs, h, t1)
                    pend += h.shape[0]
                    del h, t1, songs
                    if pend >= args.match_flush_rows // 2:
                        full.finalize(); pend = 0
                n_full = full.finalize()
                fp2.close()
                k = min(args.match_check_queries, n_q_local)
                want = [t.cpu().numpy() for t in full.query_batch(qh[:q_starts[k]], qt1[:q_starts[k]], q_starts[:k + 1], topn)]
                subsample = {"queries": k, "single_index_rows": n_full, "rows_equal": bool(n_full == rows_total),
                             "equal": bool(all(np.array_equal(a[:k], b) for a, b in zip(res_np, want)))}
                full.close()
                del full
            except Exception as e:      # e.g. out of memory next to the shard: say so instead of dying
                subsample = {"skipped": f"{type(e).__name__}: {str(e)[:200]}"}
        barrier()

    if rank != 0:
        return None

    qids = np.concatenate([np.asarray(r["qids"], np.int64) for r in allr])
    cat = [np.concatenate([r["res"][k] for r in allr]) for k in range(5)]
    song, diff, cnt = cat[0], cat[1], cat[2]
    ok = (song[:, 0] == q_tracks[qids] + 1) & (diff[:, 0] == q_start[qids])
    nth = cnt[:, topn - 1]
    nth_hist = {str(int(v)): int(c) for v, c in zip(*np.unique(np.minimum(nth, 16), return_counts=True))}
    total_hashes = sum(r["hashes"] for r in allr)
    if args.dump_outputs:
        order = np.argsort(qids, kind="stable")          # row q = query q
        dump_rows(args.dump_outputs, "match", {name: a[order] for name, a in zip(("song", "diff", "count", "rows", "nres"), cat)},
                  seed=3)

    out = {"metric": "match_queries_per_second", "value": Q / (ms_step * 1e-3), "unit": "queries/s", "n_gpus": world,
           "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "ms_per_step_median": ms_med,
           "ms_of_each_step_rank0": per_step_ms,
           "higher_is_better": True, "scaling": "strong", "dtype": "u64", "data": "synthetic",
           "sharding": ("one index on one GPU" if world == 1 else
                        "hash prefix: query entries routed to the shard owning their hash, vote keys exchanged (2 equal-split "
                        "NCCL all-to-alls per pass), exact vote at the query's owner"),
           "config": {"workload": f"configs[3]/[4]: {Q} concurrent 5 s queries (topn {topn}) against a {T}-track synthetic index "
                                  f"(~{R} fingerprints per track) on {world} GPU(s)",
                      "index_rows": int(rows_total), "distinct_hashes": int(n_keys),
                      "index_bytes": int(rows_total) * 8 + int(n_keys) * 16,
                      "rows_generated": int(sum(r["rows"] for r in allr)), "query_hashes_per_step": int(total_hashes),
                      "mean_hashes_per_query": total_hashes / max(1, Q), "queries_per_pass_per_rank": qp if world > 1 else None,
                      "l2": "index (GBs of postings) and per-step vote tables are far larger than L2"},
           "clocks": clocks, "e2e": e2e,
           "accuracy_top1_song_and_offset": float(ok.mean()),
           "index_build": {"seconds": round(t_build, 2), "rows_per_second": rows_total / t_build,
                           "finalize": "incremental merge every %d pending rows" % args.match_flush_rows},
           "identity": {"results_sha256": results_digest(qids, cat, topn),
                        "note": "the same query set at every N: equal checksums at N = 1/2/4/8 mean results identical to the "
                                "single-GPU index for all queries, tie-breaks included"},
           "nth_result_count_histogram": {"topn": topn, "counts": nth_hist,
                                          "note": "aligned matches of each query's n-th result: a threshold top-k merge needs "
                                                  "this to exceed the number of shards to prune anything"}}
    if world > 1:
        out["key_exchange"] = {"value": out["value"], "unit": "queries/s", "ms_per_step": ms_step, "ms_per_step_median": ms_med}
        out["peer_memory"] = peer_line
        if use_peer:
            # the headline of the hash-prefix design is its faster exact variant; both are printed
            out["value"], out["ms_per_step"], out["ms_per_step_median"] = peer_line["value"], peer_line["ms_per_step"], peer_line["ms_per_step_median"]
            out["sharding"] = ("hash prefix: query entries routed to the shard owning their hash (NCCL all-to-all), vote tuples "
                               "scattered by that shard straight into the query owner's regions over NVLink peer memory "
                               "(exchange fused into the kernel), exact vote at the query's owner")
        out["track_sharded"] = track_line
        out["identity"]["hash_prefix_equals_track_sharded"] = hash_eq_track
        out["identity"]["subsample_vs_single_index"] = subsample
        out["exchange"] = {"retries_in_timed_steps": retries, "key_slot_capacity": hashed.key_cap,
                           "entry_slot_capacity": hashed.entry_cap, "passes_per_step": -(-max(len(r["qids"]) for r in allr) // qp),
                           "last_pass_stage_ms_rank0": pass_ms, "collective": "all_to_all_single (NCCL), equal splits"}
    if qstats:
        tuples = qstats[2]
        out["per_step"] = {"query_pairs": qstats[0], "db_rows_matched": qstats[1], "vote_tuples": tuples,
                           "distinct_bins": qstats[3], "mean_postings_per_query_hash": qstats[1] / max(1, qstats[0])}
        # vote roofline: per query hash 8 B directory + 16 B key entry, per vote tuple 8 B posting + 16 B of vote traffic
        # (SURVEY §8d's figure with the 8-byte posting of this layout)
        peak, peak_src = measured_peak_gbs()
        algo = qstats[0] * 24 + tuples * 24
        ach = algo / (vote_ms * 1e-3) / 1e9 if vote_ms else None
        traffic, traffic_src = None, None
        prof = os.path.join(ROOT, "profiles", "vote_traffic.json")
        if os.path.exists(prof):
            try:
                vt = json.load(open(prof))
                traffic = vt["dram_bytes_per_tuple"] * tuples
                traffic_src = "profiles/vote_traffic.json (ncu --set full: dram read + write of pv_scatter_kernel + pv_count_kernel per tuple) x tuples per step"
            except Exception:
                pass
        out["roofline"] = {"bound": "hbm", "kernel": "pv_scatter_kernel + pv_count_kernel (partitioned vote: posting runs -> (query, song "
                                                     "partition) regions -> shared-memory duplicate filter + exact table) + pv_merge_kernel",
                           "achieved": ach, "peak": peak, "unit": "GB/s", "frac": (ach / peak) if ach else None,
                           "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes_per_step": algo,
                           "formula": "H*(8+16) + T*(8+16): H query (hash, offset) pairs (8 B directory + 16 B key entry), T vote tuples "
                                      "(8 B posting read + 8 B tuple written to its region + 8 B read back by the count)",
                           "vote_ms_per_step": vote_ms, "lookup_ms_per_step": lookup_ms,
                           "vote_tuples_per_second": tuples / (vote_ms * 1e-3) if vote_ms else None}
    # ---- CPU baseline: the reference's return_matches + align_matches on a 2,714-track table (configs[2]'s size) ----
    if world == 1 and not args.no_cpu_baseline and args.match_cpu_tracks > 0:
        try:
            out["cpu_baseline"] = cpu_match_baseline(args, dev, local_rank, P, q_tracks, q_ids, qh, qt1, q_starts)
        except Exception as e:
            out["cpu_baseline"] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
    return out


def cpu_match_baseline(args, dev, local_rank, P, q_tracks, q_ids, qh, qt1, q_starts):
    """Oracle port of return_matches + align_matches (recognizer.py:222-338) over an in-memory stand-in for the MySQL
    table holding the first `--match-cpu-tracks` tracks of the same index (the 100k-track table does not fit a host);
    the rows come out of a GPU index export (already unique, in (hash, song, offset) order)."""
    import torch
    from oracle import sia_oracle as O
    from shazam_b200.database import FingerprintIndex
    from shazam_b200.fingerprinter import Fingerprinter
    GB, R = args.match_gen_batch, args.match_rows_per_track
    ntr = min(args.match_cpu_tracks, args.match_tracks)
    os.environ["SIA_PEAKS_PER_FRAME_CAP"] = str(max(32, -(-(GB * P) // 4096) + 1))
    fp = Fingerprinter(local_rank, max_chunk_frames=4096)
    ix = FingerprintIndex(local_rank, int(ntr * R * 1.02) + (1 << 20))
    for b in range(-(-ntr // GB)):
        nt = min(GB, args.match_tracks - b * GB)
        pt, pf = batch_peaks(dev, b, nt, P)
        keep = min(nt, ntr - b * GB)
        tps = torch.arange(keep + 1, device=dev, dtype=torch.int64) * P
        h, t1, ths = fp.pairs_sha1(pt[:keep].reshape(-1), pf[:keep].reshape(-1), tps, FAN)
        songs = torch.repeat_interleave(torch.arange(keep, device=dev, dtype=torch.int32) + (b * GB + 1), ths[1:] - ths[:-1])
        ix.insert_rows(songs, h, t1)
    n = ix.finalize()
    fp.close()
    d, s, o = ix.export()
    hi = torch.zeros(n, dtype=torch.int64, device=dev)
    for k in range(8):
        hi |= d[:, k].to(torch.int64) << (8 * (7 - k))
    lo = (d[:, 8].to(torch.int64) << 8) | d[:, 9].to(torch.int64)
    table = O.ArrayFingerprintTable.from_sorted(hi.cpu().numpy().view(np.uint64), lo.cpu().numpy(), s.cpu().numpy(), o.cpu().numpy())
    ix.close()
    del d, s, o, hi, lo
    for sid in range(1, ntr + 1):
        table.songs[sid] = {"song_name": f"t{sid}", "file_sha1": "AB" * 20, "total_hashes": R, "fingerprinted": 1}
    procs = os.cpu_count() or 1
    picks = [k for k, qi in enumerate(q_ids) if q_tracks[qi] < ntr][: max(4 * procs, 16)]
    queries = []
    for k in picks:
        a, b = int(q_starts[k]), int(q_starts[k + 1])
        hx = qh[a:b].cpu().numpy().tobytes().hex()
        queries.append(set((hx[20 * i:20 * i + 20], int(t)) for i, t in enumerate(qt1[a:b].cpu().tolist())))
    v, dt, outs = cpu_match_run(table, queries, procs)
    hit = sum(1 for nm, _ in outs if nm > 0)
    return {"value": v, "unit": "queries/s", "cores": procs, "kind": "port",
            "sample": f"{len(queries)} of the step's 5 s queries ({dt:.1f} s wall) against the first {ntr} tracks of the index "
                      f"({n} rows) in an in-memory stand-in for the MySQL table; oracle port of return_matches + align_matches, "
                      f"Pool({procs}); mean {np.mean([o[0] for o in outs]):.0f} (song, diff) tuples per query — the 100k-track "
                      "table does not fit the host, and postings per hash grow with the index",
            "queries_with_matches": hit}


# ==========================================================================================
def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    audio_s_per_track = args.track_samples / FS
    config = {"workload": f"configs[1]: batch fingerprinting of {args.tracks} synthetic {audio_s_per_track:.0f}-s "
                          f"44.1 kHz mono int16 tracks per GPU (fan {FAN}, amp_min {AMP_MIN}, wsize 4096, overlap 0.5)",
              "tracks_per_gpu": args.tracks, "track_samples": args.track_samples, "fan_value": FAN,
              "amp_min": AMP_MIN, "sharding": "by track, no collective", "l2": "inputs larger than L2 (15.9 GB PCM per step)",
              "k3": "sha1 per pair" if args.no_digest_table else "digest table (13.5 GB, built once per context by the SHA-1 kernel)"}

    # ---------------------------------------------------------------- reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import sia_oracle as O
        procs = os.cpu_count() or 1
        ntr = args.cpu_sample_tracks or max(procs, 8)
        tracks = [O.synth_track(10_000 + i, args.track_samples) for i in range(ntr)]
        v, dt, nh = cpu_reference_run(tracks, procs, steps=max(args.steps, 1), warmup=min(args.warmup, 1))
        sample = (f"{ntr} of the {args.tracks} tracks per step ({ntr * audio_s_per_track:.0f} audio-s), "
                  f"Pool({procs}) one task per track like fingerprint_directory (__init__.py:341,357)")
        v1, dt1, _ = cpu_reference_run(tracks[:2], 1)            # SURVEY §8(d): the one-process figure, outside the timed steps
        one = {"value": v1, "unit": "audio-s/s", "cores": 1, "sample": f"first {len(tracks[:2])} tracks, {dt1:.1f} s wall"}
        print(json.dumps({
            "impl": "reference", "metric": "fingerprint_audio_seconds_per_second", "value": v, "unit": "audio-s/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config,
            "cpu_baseline": {"value": v, "unit": "audio-s/s", "cores": procs, "kind": "port", "sample": sample,
                             "one_process": one},
            "e2e": {"value": v, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "hashes_per_step_sample": nh}))
        return

    # ---------------------------------------------------------------- B200 arm
    import torch
    import torch.distributed as dist

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL on high-priority streams: its few CTAs are dispatched ahead of the pending CTAs of the big vote kernels, so
        # the exchange of pass i+1 really overlaps the vote of pass i
        opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(minutes=8), pg_options=opts)

    out = None
    if not args.no_fingerprint:
        out = fingerprint_leg(args, rank, world, local_rank, dev, config)
    match = None
    if not args.no_match:
        try:
            match = match_leg(args, rank, world, local_rank, dev)
        except Exception as e:      # keep the M1 line whatever happens to M2 (and say what happened)
            import traceback
            traceback.print_exc()
            match = {"error": f"{type(e).__name__}: {str(e)[:300]}"}
    if rank == 0:
        if out is None:
            out = {"metric": "fingerprint_audio_seconds_per_second", "value": None, "note": "--no-fingerprint"}
        out["match"] = match
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
