"""Peak neighbourhood of any size (PEAK_NEIGHBORHOOD_SIZE 1..64, CONNECTIVITY_MASK 1 or 2): K2's footprint kernel
bit-exact against the oracle's get_2D_peaks on float64 and float32 input, per track of a multi-track chunk, end to
end through compat and both pipelines, and through the streaming path."""
import numpy as np
import pytest

from oracle import sia_oracle as O
from tests.test_fingerprint_gpu import _gpu_peaks
from tests.test_stream_gpu import _cuts, run_streams

pytestmark = pytest.mark.gpu


def _arr(rng, F, T):
    """Values rounded to 0.1 (ties and plateaus) with a zero block (the erosion term)."""
    a = np.round(rng.normal(6, 9, (F, T)), 1)
    a[F // 3:F // 3 + max(F // 4, 1), T // 4:T // 4 + max(T // 3, 1)] = 0.0
    return a


@pytest.mark.parametrize("nbhd", [1, 2, 5, 9, 11, 16, 17, 20, 31, 32, 33, 64])
def test_float64_against_oracle(fpr, nbhd):
    rng = np.random.default_rng(100 + nbhd)
    shapes = [(300, 140), (5, 40), (40, 5), (1, 1), (2049, 3)]   # smaller than the window in one or both axes
    for F, T in shapes:
        arr = _arr(rng, F, T)
        for conn in (1, 2):
            for amp in (5, 0, -5):
                got = _gpu_peaks(fpr, arr, amp, conn, nbhd)
                want = np.array(O.get_2D_peaks(arr, amp, conn, nbhd), np.int32).reshape(-1, 2)
                assert np.array_equal(got, want), (F, T, nbhd, conn, amp, len(got), len(want))


@pytest.mark.parametrize("nbhd", [20, 64])
@pytest.mark.parametrize("conn", [1, 2])
def test_float32_tracks_do_not_leak(fpr, nbhd, conn):
    """Tracks of 1, 7, 2*nbhd and 300 frames in one chunk: each equals the oracle on that track alone."""
    import torch
    rng = np.random.default_rng(7 * nbhd + conn)
    frames = [1, 7, 2 * nbhd, 300, 7]
    arrs = [_arr(rng, 2049, T).astype(np.float32) for T in frames]
    arrs[3][500:520, 100:140] = 60.0                       # a plateau wider than the window at nbhd 20
    host = np.zeros((sum(frames), 2080), np.float32)
    host[:, :2049] = np.concatenate([a.T for a in arrs])
    spec = torch.from_numpy(host).to(fpr.tdev)
    for amp in (10, -3):
        p = fpr.params(amp_min=amp, connectivity=conn, nbhd=nbhd)
        pt, pf, tps = fpr.peaks(spec, np.array(frames, np.int64), p, cap_peaks=host.size)
        pt, pf, tps = pt.cpu().numpy(), pf.cpu().numpy(), tps.cpu().numpy()
        for k, a in enumerate(arrs):
            want = sorted((int(t), int(f)) for f, t in O.get_2D_peaks(a.astype(np.float64), amp, conn, nbhd))
            got = list(zip(pt[tps[k]:tps[k + 1]].tolist(), pf[tps[k]:tps[k + 1]].tolist()))
            assert got == want, (amp, k, len(got), len(want))


def _oracle_hex(x, fs, fan, conn, nbhd, wratio=0.5):
    arr = O.spectrogram_db(x, fs, 4096, int(4096 * wratio))
    return O.generate_hashes(O.get_2D_peaks(arr, 10, conn, nbhd), fan)


@pytest.mark.parametrize("nbhd,conn", [(20, 2), (20, 1), (64, 2), (64, 1)])
def test_compat_end_to_end(fpr, wav_fixture, synth_cases, monkeypatch, nbhd, conn):
    from shazam_b200 import compat
    from shazam_b200.fingerprinter import pack_tracks
    import torch
    monkeypatch.setattr(compat, "PEAK_NEIGHBORHOOD_SIZE", nbhd)
    monkeypatch.setattr(compat, "CONNECTIVITY_MASK", conn)
    compat.set_fingerprinter(fpr)
    try:
        x = wav_fixture["pcm"]
        for fs in (22050, 44100):
            for fan in (5, 15):
                want = _oracle_hex(x, fs, fan, conn, nbhd)
                assert len(want) > 0 and compat.fingerprint(x, Fs=fs, fan_value=fan) == want, (fs, fan)
        want = _oracle_hex(x, 22050, 15, conn, nbhd, 0.75)
        assert compat.fingerprint(x, Fs=22050, fan_value=15, wratio=0.75) == want
        for kind in synth_cases["kinds"]:
            y = synth_cases[f"{kind}_pcm"]
            assert compat.fingerprint(y, fan_value=15) == _oracle_hex(y, 44100, 15, conn, nbhd), kind
    finally:
        compat.set_fingerprinter(None)
    # the host pipeline and the device pipeline agree
    tracks = [O.synth_track(900 + i, n) for i, n in enumerate([30 * 44100, 4096, 0, 200000, 12 * 44100 + 5])]
    p = fpr.params(fan_value=15, connectivity=conn, nbhd=nbhd)
    pcm, starts, lens = pack_tracks(tracks)
    a = fpr.fingerprint_host(pcm, starts, lens, p)
    b = fpr.fingerprint_device(torch.from_numpy(pcm).to(fpr.tdev), starts, lens, p)
    assert len(a.t1) > 0 and np.array_equal(a.starts, b.starts)
    assert np.array_equal(a.hash, b.hash.cpu().numpy()) and np.array_equal(a.t1, b.t1.cpu().numpy())


def _rule_counts(fpr, x, fan, nbhd, conn, lengths):
    """Cumulative hash counts the emission rule of DESIGN §11 gives after pushes ending at these sample counts."""
    import torch
    from shazam_b200.fingerprinter import pack_tracks
    pcm, starts, lens = pack_tracks([x])
    p = fpr.params(fan_value=fan, nbhd=nbhd, connectivity=conn)
    spec = fpr.stft_db(torch.from_numpy(pcm).to(fpr.tdev), starts, lens, p)
    pt, _, _ = fpr.peaks(spec, np.array([spec.shape[0]], np.int64), p)
    t = pt.cpu().numpy().astype(np.int64)
    m = np.zeros(len(t), np.int64)
    for i in range(len(t)):
        for j in range(1, fan):
            if i + j >= len(t) or t[i + j] - t[i] > 200:
                break
            m[i] += 1
    out = []
    for L in lengths:
        F = 1 + (L - 4096) // 2048 if L >= 4096 else 0
        H = F - 1 - nbhd
        n = int(np.searchsorted(t, H, side="right"))
        k = max(n - fan + 1, int(np.searchsorted(t, H - 200, side="right")), 0)
        out.append(int(m[:k].sum()))
    return out


@pytest.mark.parametrize("nbhd", [20, 64])
@pytest.mark.parametrize("conn", [1, 2])
def test_streaming_equals_batch(fpr, wav_fixture, nbhd, conn):
    from shazam_b200.stream import StreamFingerprinter
    x = wav_fixture["pcm"]
    fan = 15
    cut_sets = [_cuts(len(x), 997), _cuts(len(x), 2048), _cuts(len(x), 8192), _cuts(len(x), 30000),
                [4096] + [2048] * 40 + _cuts(len(x) - 4096 - 40 * 2048, 50000), [len(x)]]
    sf = StreamFingerprinter(fpr, len(cut_sets), fan_value=fan, connectivity=conn, nbhd=nbhd)
    try:
        # push() sizes its output with default_cap: a push it did not cover would raise CapacityError
        got, counts = run_streams(sf, [x] * len(cut_sets), cut_sets)
    finally:
        sf.close()
    want = fpr.fingerprint_tracks([x], fan_value=fan, connectivity=conn, nbhd=nbhd)
    assert len(want.t1) > 0
    for i, (cuts, cnt, (h, t)) in enumerate(zip(cut_sets, counts, got)):
        assert np.array_equal(h, want.hash) and np.array_equal(t, want.t1), (i, len(t), len(want.t1))
        assert cnt == _rule_counts(fpr, x, fan, nbhd, conn, np.cumsum(cuts)[:-1]) + [len(t)], i


def test_streaming_capacity_at_nbhd_64(fpr):
    """At nbhd 64 a stream carries 128 rows: a push whose carried + new rows exceed a small workspace is
    SIA_E_CAPACITY and leaves every stream as it was."""
    from shazam_b200 import _native as N
    from shazam_b200.fingerprinter import Fingerprinter
    from shazam_b200.stream import StreamFingerprinter
    fp = Fingerprinter(0, max_chunk_frames=256)
    try:
        y = O.synth_track(31, 40 * 44100)
        z = O.synth_track(32, 20 * 44100)
        want = [fpr.fingerprint_tracks([t], nbhd=64).track(0) for t in (y, z)]
        sf = StreamFingerprinter(fp, 2, nbhd=64)
        try:
            r0 = sf.push([y[:200 * 2048], z[:100000]])            # 128 carried rows after this push
            with pytest.raises(N.CapacityError, match="rows"):
                sf.push([y[200 * 2048:200 * 2048 + 140 * 2048], z[100000:110000]])  # 128 + 140 > 256
            rest = [y[200 * 2048:], z[100000:]]
            (gy, gz), _ = run_streams(sf, rest, [_cuts(len(rest[0]), 100 * 2048), _cuts(len(rest[1]), 100 * 2048)])
        finally:
            sf.close()
        for b, (g, w) in enumerate(zip((gy, gz), want)):
            h0, t0 = r0.track(b)
            assert np.array_equal(np.concatenate([h0, g[0]]), w[0]) and np.array_equal(np.concatenate([t0, g[1]]), w[1])
    finally:
        fp.close()


def test_full_size_track_nbhd_20(fpr):
    """A 3-minute track: as in test_full_size_track_properties, K2 compares the float32-stored dB, so a few peaks
    differ from the float64 oracle where rounding creates or breaks ties; print how many."""
    from shazam_b200.fingerprinter import digests_to_hex
    n = 7_938_000
    x = O.synth_track(1000, n)
    b = fpr.fingerprint_tracks([x], fan_value=15, nbhd=20)
    h, t1 = b.track(0)
    want = _oracle_hex(x, 44100, 15, 2, 20)
    sa = set(zip(digests_to_hex(h), t1.tolist()))
    sb = set((hx, int(t)) for hx, t in want)
    jacc = len(sa & sb) / len(sa | sb)
    print(f"full-size track at nbhd 20: {len(sa)} GPU / {len(sb)} oracle hashes, {len(sa - sb)} only GPU, "
          f"{len(sb - sa)} only oracle, Jaccard {jacc:.5f}")
    assert len(sa) > 1000 and jacc >= 0.99, (jacc, len(sa - sb), len(sb - sa))
