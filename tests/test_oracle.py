"""The oracle against the committed golden vectors (made by executing the reference's own
functions, tests/golden/make_golden.py) and against scipy for the restated specgram."""
import hashlib
import os

import numpy as np
import pytest

from oracle import sia_oracle as O


def test_sha1_kats():
    # SURVEY.md §8 a-5 known answers
    for msg, want in [("253|422|0", "987a1bcc49e707cb9e6a"), ("253|577|0", "0f34024f21634bf6fbb0"),
                      ("2048|0|200", "a8b1bf935e7453ba6aef"), ("0|0|0", "bcd8195eb61a41102f4c")]:
        assert hashlib.sha1(msg.encode()).hexdigest()[:20] == want
    assert O.generate_hashes([(253, 0), (422, 0), (577, 0)], 5)[0:2] == \
        [("987a1bcc49e707cb9e6a", 0), ("0f34024f21634bf6fbb0", 0)]


def test_specgram_matches_scipy(wav_fixture):
    from scipy.signal import spectrogram
    x = wav_fixture["pcm"]
    for fs in (22050, 44100):
        P = O.specgram_psd(x, fs)
        _, _, S = spectrogram(x.astype(np.float64), fs=fs, window=np.hanning(4096), nperseg=4096, noverlap=2048,
                              detrend=False, scaling="density", mode="psd")
        assert P.shape == S.shape == (2049, 106)
        assert np.max(np.abs(P - S) / S) < 1e-8
    assert O.num_frames(220500) == 106 and O.num_frames(3000) == 1 and O.num_frames(4096) == 1
    assert O.num_frames(8191) == 2 and O.num_frames(0) == 1


def test_specgram_against_a_direct_dft_in_extended_precision(wav_fixture):
    """SURVEY.md §8 a-2 / Appendix A written out from first principles — a direct O(N^2) DFT in numpy longdouble (no FFT
    library, no scipy) of a few frames, including the weakest bins (the 1e-3 dB bound of north_star is on EVERY bin, and
    the oracle is what the kernel is measured against): frames x[2048k : 2048k+4096], symmetric Hann, |X|^2, bins
    1..2047 doubled, / Fs, / sum(win^2)."""
    x = wav_fixture["pcm"].astype(np.longdouble)
    fs = 22050
    P = O.specgram_psd(wav_fixture["pcm"], fs)
    n = np.arange(4096, dtype=np.longdouble)
    win = (0.5 - 0.5 * np.cos(2 * np.pi * n / 4095)).astype(np.longdouble)          # np.hanning(4096)
    k = np.arange(2049, dtype=np.int64)
    # exp(-2 pi i k n / N) with the phase reduced mod N in integers before the multiplication
    phase = (np.outer(k, np.arange(4096, dtype=np.int64)) % 4096).astype(np.longdouble) * (2 * np.pi / 4096)
    C, S = np.cos(phase), np.sin(phase)
    worst = 0.0
    for t in (0, 57, 105):
        f = x[2048 * t: 2048 * t + 4096] * win
        re, im = C @ f, -(S @ f)
        p = re * re + im * im
        p[1:2048] *= 2
        p = p / fs / (win * win).sum()
        rel = np.abs(P[:, t].astype(np.longdouble) - p) / p
        worst = max(worst, float(rel.max()))
        db = np.abs(10 * np.log10(P[:, t].astype(np.longdouble)) - 10 * np.log10(p))
        assert float(db.max()) < 1e-9, (t, float(db.max()))          # measured 5e-11 dB
    assert worst < 1e-9, worst          # measured 1.1e-11: float64 FFT rounding on bins 113 dB under the frame maximum


def test_wav_fixture_pins(wav_fixture):
    g = wav_fixture
    arr = O.spectrogram_db(g["pcm"], 22050)
    assert arr.shape == (2049, 106)
    assert abs(arr.min() + 74.795) < 2e-3 and abs(arr.max() - 69.344) < 2e-3
    for conn in (2, 1):
        pk = np.array(O.get_2D_peaks(arr, 10, conn), np.int32).reshape(-1, 2)
        assert np.array_equal(pk, g[f"peaks_c{conn}"])
    assert len(g["peaks_c2"]) == 409 and len(g["peaks_c1"]) == 663
    for conn in (2, 1):
        for fan in (5, 15):
            for fs in (22050, 44100):
                h, t = O.fingerprint_arrays(g["pcm"], fs, fan, 10, conn)
                assert np.array_equal(h, g[f"hash_c{conn}_fan{fan}_fs{fs}"])
                assert np.array_equal(t, g[f"t1_c{conn}_fan{fan}_fs{fs}"])
    assert len(g["hash_c2_fan5_fs22050"]) == 1626 and len(g["hash_c2_fan15_fs22050"]) == 5621
    h, t = O.fingerprint_arrays([int(v) for v in g["pcm"][:50000]], 44100)
    assert np.array_equal(h, g["hash_list50k"]) and np.array_equal(t, g["t1_list50k"])


def test_synth_cases(synth_cases):
    g = synth_cases
    for kind in g["kinds"]:
        x = g[f"{kind}_pcm"]
        for fan, amp in ((5, 10), (15, 10), (15, 0), (15, -5)):
            h, t = O.fingerprint_arrays(x, 44100, fan, amp)
            assert np.array_equal(h, g[f"{kind}_hash_fan{fan}_amp{amp}"]), (kind, fan, amp)
            assert np.array_equal(t, g[f"{kind}_t1_fan{fan}_amp{amp}"]), (kind, fan, amp)


def test_peaks_cases_and_clipped_window_statement(peaks_cases):
    g = peaks_cases
    for name in g["names"]:
        arr = g[f"{name}_arr"]
        for conn in (2, 1):
            for amp in (10, 0, -5, -100):
                want = g[f"{name}_c{conn}_amp{amp}"]
                got = np.array(O.get_2D_peaks(arr, amp, conn), np.int32).reshape(-1, 2)
                assert np.array_equal(got, want), (name, conn, amp)
                if arr.size <= 8000:   # the statement the CUDA kernel implements
                    bf = np.array(O.peaks_bruteforce(arr, amp, conn), np.int32).reshape(-1, 2)
                    assert np.array_equal(bf, want), ("bruteforce", name, conn, amp)


def test_match_cases(match_cases):
    for case in match_cases:
        if case["case"] == "kat":
            r = case["results"]
            assert [(x["song_id"], x["offset"], x["offset_seconds"]) for x in r] == \
                [(2, -4, -0.18576), (7, 3, 0.13932), (9, 1, 0.04644)]
            continue
        table = O.FingerprintTable()
        for sid, s in sorted(case["songs"].items(), key=lambda kv: int(kv[0])):
            assert table.insert_song(s["song_name"], s["file_sha1"], s["total_hashes"]) == int(sid)
        for sid, h, o in case["rows"]:
            table.insert_hashes(sid, [(h, o)])
        q = [tuple(x) for x in case["query"]]
        matches, dedup = O.return_matches(table, q)
        assert len(matches) == case["n_matches"]
        assert hashlib.sha256(repr(sorted(matches)).encode()).hexdigest() == case["matches_sorted_sha"]
        assert {str(k): v for k, v in dedup.items()} == case["dedup"]
        for topn, want in case["results_by_topn"].items():
            got = O.align_matches(table, matches, dedup, len(q), int(topn)) if q else []
            got = [{k: (v.decode() if isinstance(v, bytes) else v) for k, v in r.items()} for r in got]
            assert got == want


def test_mix_noise_equals_the_reference_mixer():
    """``get_noise_from_sound`` (recognizer_test.py:426-435, executed from the reference's source by make_golden.py)
    + the addition of :554: the oracle's mixer — what the GPU mixer ``sia_mix_noise`` is checked against — gives the
    reference's scaled noise to the last bit, and the mix has the requested SNR."""
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "noise_cases.npz"))
    for k in range(2):
        signal, noise = g[f"signal_{k}"], g[f"noise_{k}"]
        for j, snr in enumerate(g["snrs"]):
            want = g[f"scaled_{k}_{j}"]
            mixed = O.mix_noise(signal, noise, float(snr))
            assert np.array_equal(mixed, signal + want), (k, j)
            got_snr = 20 * np.log10(np.sqrt(np.mean(signal ** 2)) / np.sqrt(np.mean(want ** 2)))
            assert abs(got_snr - snr) < 1e-9


def test_synth_track_is_deterministic():
    a = O.synth_track(5, 50000)
    b = O.synth_track(5, 50000)
    assert a.dtype == np.int16 and np.array_equal(a, b) and a.std() > 1000
    s = O.mix_noise(a.astype(np.float64), np.random.default_rng(0).normal(0, 1, 50000), 10.0)
    n = s - a
    assert abs(20 * np.log10(np.sqrt(np.mean(a.astype(float) ** 2)) / np.sqrt(np.mean(n ** 2))) - 10.0) < 1e-6


@pytest.mark.skipif(not os.path.isdir(os.environ.get("SIA_REFERENCE_DIR", "")),
                    reason="needs a checkout of the reference project, named by SIA_REFERENCE_DIR")
def test_committed_golden_vectors_regenerate_from_the_reference(tmp_path):
    """The pin of the pin: tests/golden/make_golden.py executes the reference's OWN functions (AST-extracted from the
    checkout named by SIA_REFERENCE_DIR) and must reproduce every committed fixture bit for bit.  No other test reads
    the reference: they compare with the committed fixtures."""
    import importlib.util
    import json
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(here, "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    mg.main(str(tmp_path))
    for name in ("wav_fixture.npz", "synth_cases.npz", "peaks_cases.npz", "noise_cases.npz"):
        a, b = np.load(os.path.join(here, name)), np.load(tmp_path / name)
        assert set(a.files) == set(b.files), name
        for k in a.files:
            assert np.array_equal(a[k], b[k]), (name, k)
    for name in ("match_cases.json", "apriori_cases.json", "csv_cases.json"):
        assert json.load(open(os.path.join(here, name))) == json.load(open(tmp_path / name)), name
