"""The a-priori early exit (FingerprintIndex.query_batch_apriori) against the full vote (query_batch) on bench.py's
match workload, one GPU: prints one JSON line.

The index and the queries are built the way bench.py's match leg builds them (batch_peaks / batch_queries, fan 15):
--tracks tracks x --rows rows, --queries 5 s queries.  After warm-up the two calls alternate for --steps
device-synchronised steps each.  Reported: ms per step of both, the tuples the a-priori path read as a share of all
tuples, the histogram of batches read, the exit rate, the share of queries whose top-1 (song, diff) equals the full
vote's, an exact check of --check queries against query_batch run on their prefix queries (batches 0..k), the
query_batch results checksum (bench.py's results_digest) and the per-kernel device time of one a-priori call
(torch.profiler).  The device name and power limit are read in the same run.

    python tools/apriori_bench.py                      # 100 000 tracks x 80 000 rows, 10 000 queries, topn 3, B 1000
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

from bench import CLIP_FRAMES, FAN, FRAMES_PER_TRACK, batch_peaks, batch_queries, results_digest   # noqa: E402


def gpu_info():
    import torch
    info = {"device": torch.cuda.get_device_name(0), "power_limit_w": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_w"] = float(out.splitlines()[0])
    except Exception as e:        # noqa: BLE001 - reported, not fatal
        info["power_limit_error"] = str(e)[:200]
    return info


def prefix_check(ix, qh, qt1, q_starts, qsel, topn, B, got):
    """query_batch over every prefix (batches 0..k, distinct hashes in ascending digest order) of the queries qsel,
    the exit rule applied here; True if every output of `got` (the a-priori call) equals it."""
    import torch
    h = qh.cpu().numpy()
    t = qt1.cpu().numpy()
    L = max(topn, 2)
    pd, po, starts, owner = [], [], [0], []
    nb = {}
    for q in qsel:
        d, o = h[q_starts[q]:q_starts[q + 1]], t[q_starts[q]:q_starts[q + 1]]
        keys = [bytes(r) for r in d]
        uniq = sorted(set(keys))
        nb[q] = -(-len(uniq) // B)
        rank = {k: i for i, k in enumerate(uniq)}
        r = np.array([rank[k] for k in keys], np.int64)
        for k in range(nb[q]):
            sel = r < (k + 1) * B
            pd.append(d[sel]); po.append(o[sel]); starts.append(starts[-1] + int(sel.sum())); owner.append((q, k))
    dev = qh.device
    res = [x.cpu().numpy() for x in ix.query_batch(torch.from_numpy(np.concatenate(pd)).to(dev),
                                                   torch.from_numpy(np.concatenate(po)).to(dev), np.array(starts, np.int64), L)]
    pick = {}
    for p, (q, k) in enumerate(owner):
        if q in pick and pick[q][2]:
            continue
        rows, nres = res[3][p], res[4][p]
        pick[q] = (p, k + 1, bool(nres >= 2 and rows[0] > 2 * rows[1]))
    for q in qsel:
        if q not in pick:
            if got[4][q] != 0 or got[5][q] != nb[q] or got[6][q] != 0:
                return False
            continue
        p, b, fired = pick[q]
        for i in range(4):
            if not np.array_equal(got[i][q], res[i][p][:topn]):
                return False
        if got[4][q] != min(int(res[4][p]), topn) or got[5][q] != b or got[6][q] != int(fired):
            return False
    return True


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--tracks", type=int, default=100_000)
    ap.add_argument("--rows", type=int, default=80_000, help="rows per track")
    ap.add_argument("--queries", type=int, default=10_000)
    ap.add_argument("--topn", type=int, default=3)
    ap.add_argument("--batch", type=int, default=1000, help="distinct hashes per a-priori batch (B)")
    ap.add_argument("--gen-batch", type=int, default=500, help="tracks generated per batch")
    ap.add_argument("--flush-rows", type=int, default=250_000_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--check", type=int, default=64, help="queries of the prefix-query exact check")
    ap.add_argument("--profile-dir", default=None, help="write the torch.profiler table of one a-priori call here")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("apriori_bench needs a CUDA device")
    from shazam_b200.database import FingerprintIndex
    from shazam_b200.fingerprinter import Fingerprinter
    dev = torch.device("cuda", 0)
    info = gpu_info()
    T, R, Q, topn, GB, B = args.tracks, args.rows, args.queries, args.topn, args.gen_batch, args.batch
    P = max(2, R // (FAN - 1))
    n_batches = -(-T // GB)
    os.environ["SIA_PEAKS_PER_FRAME_CAP"] = str(max(32, -(-(GB * P) // 4096) + 1))
    fp = Fingerprinter(0, max_chunk_frames=4096)
    rng = np.random.default_rng(5)
    q_tracks = rng.integers(0, T, Q)
    q_start = rng.integers(0, FRAMES_PER_TRACK - CLIP_FRAMES, Q)
    by_batch = {}
    for qi in range(Q):
        by_batch.setdefault(int(q_tracks[qi]) // GB, []).append(qi)
    ix = FingerprintIndex(0, int(T * R * 1.01) + (1 << 20))
    t_build = time.perf_counter()
    q_pt, q_pf, q_len, q_ids = [], [], [], []
    pending = 0
    for b in range(n_batches):
        nt = min(GB, T - b * GB)
        pt, pf = batch_peaks(dev, b, nt, P)
        tps = torch.arange(nt + 1, device=dev, dtype=torch.int64) * P
        h, t1, ths = fp.pairs_sha1(pt.reshape(-1), pf.reshape(-1), tps, FAN)
        songs = torch.repeat_interleave(torch.arange(nt, device=dev, dtype=torch.int32) + (b * GB + 1), ths[1:] - ths[:-1])
        if b in by_batch:
            qis = by_batch[b]
            a, c, ln = batch_queries(dev, b, pt, pf, [int(q_tracks[i]) - b * GB for i in qis], [int(q_start[i]) for i in qis])
            q_pt.append(a); q_pf.append(c); q_len.append(ln); q_ids += qis
        ix.insert_rows(songs, h, t1)
        pending += GB * R
        del h, t1, songs
        if pending >= args.flush_rows or b == n_batches - 1:
            pending = 0
            rows_total = ix.finalize()
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t_build
    lens = torch.cat(q_len)
    tps = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), torch.cumsum(lens, 0)])
    qh, qt1, qths = fp.pairs_sha1(torch.cat(q_pt), torch.cat(q_pf), tps, FAN)
    q_starts = qths.cpu().numpy()
    fp.close()
    del q_pt, q_pf, q_len
    torch.cuda.empty_cache()

    full = lambda: ix.query_batch(qh, qt1, q_starts, topn)                          # noqa: E731
    apri = lambda: ix.query_batch_apriori(qh, qt1, q_starts, topn, B)               # noqa: E731
    for _ in range(max(args.warmup, 1)):
        r_full, r_apri = full(), apri()
    torch.cuda.synchronize()
    ms = {"query_batch": [], "query_batch_apriori": []}
    for _ in range(args.steps):
        for name, fn in (("query_batch", full), ("query_batch_apriori", apri)):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = fn()
            torch.cuda.synchronize()
            ms[name].append((time.perf_counter() - t0) * 1e3)
            if name == "query_batch":
                r_full = r
            else:
                r_apri = r
    s_full = ix.query_batch(qh, qt1, q_starts, topn, want_stats=True)[5]
    s_apri = ix.query_batch_apriori(qh, qt1, q_starts, topn, B, want_stats=True)[7]
    f = [x.cpu().numpy() for x in r_full]
    a = [x.cpu().numpy() for x in r_apri]
    top1_eq = (a[4] > 0) & (f[4] > 0) & (a[0][:, 0] == f[0][:, 0]) & (a[1][:, 0] == f[1][:, 0])
    top1_eq |= (a[4] == 0) & (f[4] == 0)
    hist = np.bincount(a[5])
    qsel = list(np.random.default_rng(9).choice(len(q_ids), min(args.check, len(q_ids)), replace=False))
    equal = prefix_check(ix, qh, qt1, q_starts, qsel, topn, B, a)

    stage = None
    if args.profile_dir:
        from torch.profiler import ProfilerActivity, profile
        os.makedirs(args.profile_dir, exist_ok=True)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            apri()
            torch.cuda.synchronize()
        stage = {}
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
            if t > 0:
                stage[e.key[:80]] = round(t / 1e3, 2)
        stage = dict(sorted(stage.items(), key=lambda kv: -kv[1])[:12])
        with open(os.path.join(args.profile_dir, "apriori_kernels.txt"), "w") as fh:
            fh.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=40))

    med = {k: round(float(np.median(v)), 2) for k, v in ms.items()}
    out = {
        "tool": "apriori_bench", **info,
        "index_rows": int(rows_total), "index_keys": int(ix.keys), "tracks": T, "queries": Q, "topn": topn, "batch_hashes": B,
        "build_s": round(t_build, 1),
        "ms_per_step_median": med, "ms_per_step": {k: [round(x, 2) for x in v] for k, v in ms.items()},
        "apriori_over_full_time": round(med["query_batch_apriori"] / med["query_batch"], 3),
        "tuples_full": int(s_full[2]), "tuples_apriori": int(s_apri[2]),
        "tuples_read_fraction": round(s_apri[2] / max(1, s_full[2]), 4),
        "rows_read_fraction": round(s_apri[1] / max(1, s_full[1]), 4),
        "batches_read_histogram": {str(k): int(v) for k, v in enumerate(hist) if v},
        "exit_rate": round(float(a[6].mean()), 4),
        "top1_equals_full_vote": round(float(top1_eq.mean()), 4),
        "prefix_check": {"queries": len(qsel), "equal": bool(equal)},
        "query_batch_results_sha256": results_digest(q_ids, f, topn),
        "apriori_kernel_ms_one_call": stage,
    }
    print(json.dumps(out))
    ix.close()


if __name__ == "__main__":
    main()
