"""Host-side pieces of bench.py that need no GPU: the per-kernel roofline arithmetic, the results checksum, and the
reference arm (the CPU path of M1 through the oracle port) printing the contract's JSON line."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def test_per_kernel_roofline_arithmetic():
    # the r02f line: 1000 tracks x 180 s, 2.0e8 hashes per step
    km = {"stft_db(K1)": 35.7225, "peaks_bitmap(K2)": 13.7721, "peaks_compact(K2)": 1.6989, "pairs_sha1(K3)": 3.8078,
          "scans": 0.6665}
    t = bench.per_kernel_roofline(km, 180_000.0, 200_056_346, 6541.1, True)
    assert set(t) == {"stft_db(K1)", "peaks_bitmap(K2)", "peaks_compact(K2)", "pairs_sha1(K3)"}
    k1 = t["stft_db(K1)"]
    assert k1["algorithmic_bytes_per_step"] == 264_684 * 180_000.0
    assert abs(k1["achieved_gbs"] - 264_684 * 180_000.0 / 35.7225e-3 / 1e9) < 1e-6
    assert abs(k1["frac_of_hbm_peak"] - k1["achieved_gbs"] / 6541.1) < 1e-12
    k3 = t["pairs_sha1(K3)"]
    assert abs(k3["hashes_per_second"] - 200_056_346 / 3.8078e-3) < 1.0
    assert k3["sector_granular_bytes_per_step"] == 46.0 * 200_056_346
    # SHA-1 mode: no sector figure; a kernel that did not run reports None, not a division by zero
    t2 = bench.per_kernel_roofline({"stft_db(K1)": 0.0, "pairs_sha1(K3)": 7.9}, 180_000.0, 200_056_346, 6541.1, False)
    assert t2["stft_db(K1)"]["achieved_gbs"] is None and t2["stft_db(K1)"]["frac_of_hbm_peak"] is None
    assert "sector_granular_gbs" not in t2["pairs_sha1(K3)"]


def test_results_digest_is_order_independent():
    rng = np.random.default_rng(0)
    Q, topn = 50, 3
    qids = rng.permutation(Q)
    res = [rng.integers(0, 1000, (Q, topn)).astype(np.int32) for _ in range(4)] + [rng.integers(0, 4, Q).astype(np.int32)]
    d0 = bench.results_digest(qids, res, topn)
    perm = rng.permutation(Q)
    d1 = bench.results_digest(qids[perm], [r[perm] for r in res], topn)
    assert d0 == d1
    res[1][7, 2] += 1
    assert bench.results_digest(qids, res, topn) != d0


def test_dump_rows_exact_values_fixed_sample_and_size(tmp_path):
    rng = np.random.default_rng(1)
    n = 2_000_000                                       # 56 bytes per row: more than the group's 44 MB
    h = rng.integers(0, 256, (n, 10)).astype(np.uint8)
    t1 = rng.integers(0, 1 << 31, n).astype(np.int32)
    for d in ("a", "b"):
        bench.dump_rows(str(tmp_path / d), "fingerprint", {"hash": h, "t1": t1}, seed=1)
    idx = np.load(tmp_path / "a" / "fingerprint_index.npy")
    assert idx.dtype == np.float64 and len(idx) == 44_000_000 // 56 and np.all(np.diff(idx) > 0)
    k = idx.astype(np.int64)
    got_h, got_t1 = np.load(tmp_path / "a" / "fingerprint_hash.npy"), np.load(tmp_path / "a" / "fingerprint_t1.npy")
    assert got_h.dtype == np.float32 and np.array_equal(got_h, h[k]) and got_t1.dtype == np.float64 and np.array_equal(got_t1, t1[k])
    for f in os.listdir(tmp_path / "a"):
        assert open(tmp_path / "a" / f, "rb").read() == open(tmp_path / "b" / f, "rb").read(), f
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 44_000_000 + 3 * 128
    bench.dump_rows(str(tmp_path / "c"), "match", {"song": t1[:10].reshape(5, 2)}, seed=3)     # small: every row
    assert np.array_equal(np.load(tmp_path / "c" / "match_index.npy"), np.arange(5))
    assert np.array_equal(np.load(tmp_path / "c" / "match_song.npy"), t1[:10].reshape(5, 2))


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and "--steps must be at least 1" in out.stderr


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--track-samples", "220500", "--cpu-sample-tracks", "2"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "fingerprint_audio_seconds_per_second"
    assert line["unit"] == "audio-s/s" and line["higher_is_better"] is True and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["one_process"]["cores"] == 1 and line["cpu_baseline"]["one_process"]["value"] > 0
    assert line["e2e"] == {"value": line["value"], "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_do_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
