"""Fingerprinting at any overlap ratio (wratio, hop = 4096 - int(4096 * wratio)): K1's any-hop staging against the
tuned hop-2048 path bit for bit and against the float64 oracle, hashes against the oracle's fingerprint() at the same
wratio, and the batch, host-pipeline, streaming, compat and index paths at non-default ratios."""
import numpy as np
import pytest

from oracle import sia_oracle as O
from tests.test_fingerprint_gpu import DB_TOL, _check_spec
from tests.test_stream_gpu import _cuts, run_streams

pytestmark = pytest.mark.gpu


def _hop(wratio):
    return 4096 - int(4096 * wratio)


def _spec(fpr, tracks, wratio, compute, out_dtype, fs=44100):
    """K1 rows of a batch of tracks, split per track (each [T_b, 2049])."""
    import torch
    from shazam_b200 import _native as N
    from shazam_b200.fingerprinter import pack_tracks
    pcm, starts, lens = pack_tracks(tracks)
    p = fpr.params(Fs=fs, compute=compute, wratio=wratio)
    spec = fpr.stft_db(torch.from_numpy(pcm).to(fpr.tdev), starts, lens, p, out_dtype=out_dtype)
    rows = spec[:, :2049].cpu().numpy()
    counts = [N.num_frames(n, _hop(wratio)) for n in lens]
    assert rows.shape[0] == sum(counts)
    return np.split(rows, np.cumsum(counts)[:-1])


K1_TRACKS = [(11, 100003), (12, 5000), (13, 3000), (14, 50001), (15, 4096)]


@pytest.fixture(scope="module")
def k1_tracks():
    return [O.synth_track(seed, n) for seed, n in K1_TRACKS]


@pytest.mark.parametrize("compute", ["f64", "f32"])
@pytest.mark.parametrize("out", ["f32", "f64"])
def test_k1_any_hop_bit_identical_to_tuned_path(fpr, k1_tracks, compute, out):
    import torch
    out_dtype = torch.float64 if out == "f64" else torch.float32
    half = _spec(fpr, k1_tracks, 0.5, compute, out_dtype)
    # hop 1024: frame 2k starts where frame k of hop 2048 does
    for a, b in zip(_spec(fpr, k1_tracks, 0.75, compute, out_dtype), half):
        n = min((len(a) + 1) // 2, len(b))
        assert np.array_equal(a[0:2 * n:2], b[:n])
    # hop 4096: frame k starts where frame 2k of hop 2048 does
    for a, b in zip(_spec(fpr, k1_tracks, 0.0, compute, out_dtype), half):
        n = min(len(a), (len(b) + 1) // 2)
        assert np.array_equal(a[:n], b[0:2 * n:2])
    # hop 2868 (frame starts = 0, 4 mod 8) and hop 1229 (odd: every residue mod 8): frame k equals frame 0 of the tuned
    # path on a copy of samples [k hop, k hop + 4096) at an aligned start
    x = k1_tracks[0]
    for wratio in (0.3, 0.7):
        hop = _hop(wratio)
        rows = _spec(fpr, [x], wratio, compute, out_dtype)[0]
        ks = list(range(0, 16)) + list(range(len(rows) - 9, len(rows)))
        assert len({(k * hop) % 8 for k in ks}) == (8 if hop % 2 else 2)
        copies = _spec(fpr, [x[k * hop:k * hop + 4096] for k in ks], 0.5, compute, out_dtype)
        for k, c in zip(ks, copies):
            assert c.shape[0] == 1 and np.array_equal(rows[k], c[0]), (wratio, k)


@pytest.mark.parametrize("wratio", [0.0, 0.3, 0.7, 0.75, 0.9])
def test_k1_any_hop_against_oracle(fpr, wav_fixture, wratio):
    import torch
    x = wav_fixture["pcm"]
    ref = O.spectrogram_db(x, 22050, 4096, int(4096 * wratio)).T          # [T][F]
    got = _spec(fpr, [x], wratio, "f64", torch.float64, fs=22050)[0]
    assert got.shape == ref.shape
    assert _check_spec(got.T, ref.T, floor_db=230.0) < 1e-6
    got32 = _spec(fpr, [x], wratio, "f64", torch.float32, fs=22050)[0]
    assert np.abs(got32 - ref).max() < DB_TOL                            # every bin, no floor


def _hex_list(batch, b=0):
    from shazam_b200.fingerprinter import digests_to_hex
    h, t = batch.track(b)
    return list(zip(digests_to_hex(h), [int(v) for v in t]))


def _oracle_fp(x, fs, wratio, fan, amp=10, conn=2, arr=None):
    arr = O.spectrogram_db(x, fs, 4096, int(4096 * wratio)) if arr is None else arr
    return O.generate_hashes(O.get_2D_peaks(arr, amp, conn), fan)


RATIOS = [0.0, 0.25, 0.3, 0.75, 0.9]


@pytest.mark.parametrize("wratio", RATIOS)
@pytest.mark.parametrize("fs", [22050, 44100])
def test_hashes_wav_against_oracle(fpr, wav_fixture, wratio, fs):
    x = wav_fixture["pcm"]
    arr = O.spectrogram_db(x, fs, 4096, int(4096 * wratio))
    for fan in (5, 15):
        for conn in (1, 2):
            got = _hex_list(fpr.fingerprint_tracks([x], Fs=fs, fan_value=fan, connectivity=conn, wratio=wratio))
            want = _oracle_fp(x, fs, wratio, fan, conn=conn, arr=arr)
            assert len(want) > 0 and got == want, (wratio, fs, fan, conn, len(got), len(want))


@pytest.mark.parametrize("wratio", RATIOS)
def test_hashes_synth_batch_against_oracle(fpr, synth_cases, wratio):
    """Bit-exact against the oracle, with one explained exception.  K2 compares the float32-stored dB (the
    mechanism of test_full_size_track_properties).  The 'periodic' case repeats a 2048-sample period, so at a hop
    that is not a multiple of 2048 its neighbouring frames differ only in the last bits of float64.  Rounding to
    float32 turns those near-ties into plateaus, and a plateau keeps every tied maximum.  There the GPU must equal,
    bit for bit, the oracle run on its own float64 dB rounded to float32."""
    kinds = list(synth_cases["kinds"])
    tracks = [synth_cases[f"{k}_pcm"] for k in kinds]
    batch = fpr.fingerprint_tracks(tracks, fan_value=15, wratio=wratio)
    for b, k in enumerate(kinds):
        arr = O.spectrogram_db(tracks[b], 44100, 4096, int(4096 * wratio))
        want64 = _oracle_fp(tracks[b], 44100, wratio, 15, arr=arr)
        want32 = _oracle_fp(tracks[b], 44100, wratio, 15, arr=arr.astype(np.float32).astype(np.float64))
        assert (want32 != want64) == (k == "periodic" and _hop(wratio) % 2048 != 0), (k, wratio)
        assert _hex_list(batch, b) == want32, (k, wratio)


@pytest.mark.parametrize("wratio", [0.0, 0.3, 0.75])
def test_chunking_host_and_device_paths_agree(fpr, wratio):
    import torch
    from shazam_b200.fingerprinter import Fingerprinter, pack_tracks
    tracks = [O.synth_track(60 + i, n) for i, n in enumerate([90000, 30000, 5000, 250000, 44100, 3000, 120000, 66001])]
    small = Fingerprinter(0, max_chunk_frames=256)          # 241 frames for the longest track at hop 1024
    try:
        a = small.fingerprint_tracks(tracks, fan_value=15, wratio=wratio)
        b = fpr.fingerprint_tracks(tracks, fan_value=15, wratio=wratio)
        pcm, starts, lens = pack_tracks(tracks)
        p = fpr.params(fan_value=15, wratio=wratio)
        c = fpr.fingerprint_device(torch.from_numpy(pcm).to(fpr.tdev), starts, lens, p)
        d = small.fingerprint_device(torch.from_numpy(pcm).to(small.tdev), starts, lens, p)
        for r in (b, c, d):
            assert np.array_equal(a.starts, r.starts)
            h, t = (r.hash, r.t1) if r is b else (r.hash.cpu().numpy(), r.t1.cpu().numpy())
            assert np.array_equal(a.hash, h) and np.array_equal(a.t1, t)
        assert _hex_list(a, 3) == _oracle_fp(tracks[3], 44100, wratio, 15)
    finally:
        small.close()


def test_host_pipeline_tracks_of_a_full_workspace_at_hop_4096(fpr):
    """Tracks of exactly max_chunk_frames frames at hop 4096 hold twice the samples of such tracks at hop 2048: the
    host pipeline's staging buffer has to take them."""
    import torch
    from shazam_b200.fingerprinter import Fingerprinter, pack_tracks
    mcf = 128
    n = 4096 * mcf + 4095                     # 1 + (n - 4096) // 4096 = 128 frames
    tracks = [O.synth_track(80 + i, n - 8 * i) for i in range(3)]
    small = Fingerprinter(0, max_chunk_frames=mcf)
    try:
        a = small.fingerprint_tracks(tracks, wratio=0.0)
        for i, x in enumerate(tracks):
            assert _hex_list(a, i) == _oracle_fp(x, 44100, 0.0, 5), i
        pcm, starts, lens = pack_tracks(tracks)
        b = fpr.fingerprint_device(torch.from_numpy(pcm).to(fpr.tdev), starts, lens, fpr.params(wratio=0.0))
        assert np.array_equal(a.starts, b.starts)
        assert np.array_equal(a.hash, b.hash.cpu().numpy()) and np.array_equal(a.t1, b.t1.cpu().numpy())
    finally:
        small.close()


def test_compat_fingerprint_wratio(fpr, wav_fixture):
    from shazam_b200 import _native as N
    from shazam_b200 import compat
    from shazam_b200.fingerprinter import digests_to_hex
    compat.set_fingerprinter(fpr)
    try:
        x = wav_fixture["pcm"]
        assert compat.fingerprint(x, Fs=22050, wratio=0.75) == O.fingerprint(x, 22050, 4096, 0.75)
        want = list(zip(digests_to_hex(wav_fixture["hash_c2_fan5_fs22050"]),
                        [int(v) for v in wav_fixture["t1_c2_fan5_fs22050"]]))
        assert compat.fingerprint(x, Fs=22050) == want
        with pytest.raises(N.SiaError, match="wsize") as e:
            compat.fingerprint(x, wsize=2048)
        assert e.value.code == N.E_UNSUPPORTED and "wratio" not in str(e.value)
        with pytest.raises(N.SiaError) as e:
            compat.fingerprint(x, wratio=1.0)
        assert e.value.code == N.E_INVALID
    finally:
        compat.set_fingerprinter(None)


def _rule_counts(fpr, x, fan, nbhd, wratio, lengths):
    """Cumulative hash counts the emission rule of DESIGN §11 gives after pushes ending at the given sample counts,
    with F = complete frames at this hop."""
    import torch
    from shazam_b200.fingerprinter import pack_tracks
    hop = _hop(wratio)
    pcm, starts, lens = pack_tracks([x])
    p = fpr.params(fan_value=fan, nbhd=nbhd, wratio=wratio)
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
        F = 1 + (L - 4096) // hop if L >= 4096 else 0
        H = F - 1 - nbhd
        n = int(np.searchsorted(t, H, side="right"))
        k = max(n - fan + 1, int(np.searchsorted(t, H - 200, side="right")), 0)
        out.append(int(m[:k].sum()))
    return out


@pytest.mark.parametrize("wratio", [0.0, 0.3, 0.75])
def test_streaming_any_hop_equals_batch(fpr, wav_fixture, wratio):
    from shazam_b200.stream import StreamFingerprinter
    x = wav_fixture["pcm"]
    hop = _hop(wratio)
    with_empty = [c for s in _cuts(len(x), 5000) for c in (s, 0)]
    cut_sets = [_cuts(len(x), 997), _cuts(len(x), hop), _cuts(len(x), 3 * hop + 5), _cuts(len(x), 8192), with_empty,
                [4095, 1, hop - 1, 1, 1] + _cuts(len(x) - 4097 - hop, 20000), [len(x)]]
    fan = 15
    sf = StreamFingerprinter(fpr, len(cut_sets), fan_value=fan, wratio=wratio)
    try:
        got, counts = run_streams(sf, [x] * len(cut_sets), cut_sets)
    finally:
        sf.close()
    want = fpr.fingerprint_tracks([x], fan_value=fan, wratio=wratio)
    assert len(want.t1) > 0
    for i, (cuts, cnt, (h, t)) in enumerate(zip(cut_sets, counts, got)):
        assert np.array_equal(h, want.hash) and np.array_equal(t, want.t1), (i, len(t), len(want.t1))
        ends = np.cumsum(cuts)
        assert cnt == _rule_counts(fpr, x, fan, 10, wratio, ends[:-1]) + [len(t)], i


def test_index_round_trip_at_hop_1024(fpr):
    import torch
    from shazam_b200.database import FingerprintIndex
    wratio, hop = 0.75, 1024
    songs = [O.synth_track(700 + i, 20 * 44100) for i in range(50)]
    ix = FingerprintIndex(0, capacity_rows=1 << 24)
    try:
        ref = fpr.fingerprint_tracks(songs, wratio=wratio)
        for s in range(len(songs)):
            h, t = ref.track(s)
            ix.insert(s + 1, h, t)
        rng = np.random.default_rng(3)
        picks = [(int(s), int(j)) for s, j in zip(rng.integers(0, 50, 40), rng.integers(0, (15 * 44100) // hop, 40))]
        clips = [songs[s][hop * j:hop * j + 5 * 44100] for s, j in picks]
        q = fpr.fingerprint_tracks(clips, wratio=wratio)
        song, diff, _, _, nres = ix.query_batch(torch.from_numpy(q.hash).to(fpr.tdev), torch.from_numpy(q.t1).to(fpr.tdev),
                                                q.starts, 2)
        song, diff, nres = song.cpu().numpy(), diff.cpu().numpy(), nres.cpu().numpy()
        for i, (s, j) in enumerate(picks):
            assert nres[i] >= 1 and song[i, 0] == s + 1 and diff[i, 0] == j, (i, s, j, song[i], diff[i])
    finally:
        ix.close()
