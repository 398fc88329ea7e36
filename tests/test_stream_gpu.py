"""Streaming fingerprinting (StreamFingerprinter / sia_stream_*): whatever the cut of a stream into blocks, what it
emits up to its end push is bit-identical to the whole-track path, and every hash is emitted as soon as the emission
rule allows."""
import numpy as np
import pytest

from oracle import sia_oracle as O

pytestmark = pytest.mark.gpu


def _cuts(n, size):
    return [size] * (n // size) + ([n % size] if n % size else [])


def _fine_cuts(n):
    """1-sample steps around the first frame boundaries, the rest in one block."""
    cuts, pos = [], 0
    for lo, hi in ((4090, 4100), (6138, 6150)):
        if lo > pos:
            cuts.append(lo - pos)
            pos = lo
        while pos < min(hi, n):
            cuts.append(1)
            pos += 1
    if n > pos:
        cuts.append(n - pos)
    return cuts


def run_streams(sf, tracks, cuts, end_at=None):
    """Push track b in blocks of cuts[b] (ending with its last block); returns per-stream (hash, t1) of everything
    emitted and the cumulative hash counts after every push."""
    S = len(tracks)
    bounds = [np.concatenate([[0], np.cumsum(c)]).astype(np.int64) for c in cuts]
    n_push = max(len(c) for c in cuts) if end_at is None else max(end_at) + 1
    last = [len(c) - 1 for c in cuts] if end_at is None else list(end_at)
    out_h = [[] for _ in range(S)]
    out_t = [[] for _ in range(S)]
    counts = [[] for _ in range(S)]
    for k in range(n_push):
        blocks, end = [], np.zeros(S, bool)
        for b in range(S):
            if k < len(cuts[b]) and k <= last[b]:
                blocks.append(tracks[b][bounds[b][k]:bounds[b][k + 1]])
            else:
                blocks.append(None)
            end[b] = k == last[b]
        r = sf.push(blocks, end=end)
        for b in range(S):
            h, t = r.track(b)
            if k <= last[b]:
                out_h[b].append(h)
                out_t[b].append(t)
                counts[b].append(sum(len(x) for x in out_t[b]))
            else:
                assert len(t) == 0
    cat = [(np.concatenate(out_h[b]).reshape(-1, 10), np.concatenate(out_t[b])) for b in range(S)]
    return cat, counts


def _stream_fp(fp, n, **kw):
    from shazam_b200.stream import StreamFingerprinter
    return StreamFingerprinter(fp, n, **kw)


@pytest.mark.parametrize("fs", [22050, 44100])
@pytest.mark.parametrize("fan", [5, 15])
@pytest.mark.parametrize("conn", [1, 2])
def test_wav_fixture_any_cut_equals_golden(fpr, wav_fixture, fs, fan, conn):
    x = wav_fixture["pcm"]
    cut_sets = [_cuts(len(x), s) for s in (997, 2048, 4096, 8192, 44100)] + [_fine_cuts(len(x)), [len(x)]]
    sf = _stream_fp(fpr, len(cut_sets), Fs=fs, fan_value=fan, connectivity=conn)
    try:
        got, _ = run_streams(sf, [x] * len(cut_sets), cut_sets)
    finally:
        sf.close()
    want_h, want_t = wav_fixture[f"hash_c{conn}_fan{fan}_fs{fs}"], wav_fixture[f"t1_c{conn}_fan{fan}_fs{fs}"]
    for i, (h, t) in enumerate(got):
        assert np.array_equal(h, want_h) and np.array_equal(t, want_t), (i, len(t), len(want_t))


def _rule_counts(fpr, x, fan, nbhd, lengths):
    """Cumulative hash counts the emission rule gives after pushes ending at the given sample counts, from the
    whole-track GPU peaks."""
    import torch
    from shazam_b200.fingerprinter import pack_tracks
    pcm, starts, lens = pack_tracks([x])
    p = fpr.params(fan_value=fan, nbhd=nbhd)
    spec = fpr.stft_db(torch.from_numpy(pcm).to(fpr.tdev), starts, lens, p)
    pt, pf, _ = fpr.peaks(spec, np.array([spec.shape[0]], np.int64), p)
    t = pt.cpu().numpy().astype(np.int64)
    n_all = len(t)
    m = np.zeros(n_all, np.int64)
    for i in range(n_all):
        for j in range(1, fan):
            if i + j >= n_all or t[i + j] - t[i] > 200:
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


@pytest.mark.parametrize("fan", [5, 15])
def test_emission_timing(fpr, wav_fixture, fan):
    x = wav_fixture["pcm"]
    cut_sets = [_cuts(len(x), 997), _cuts(len(x), 8192), _fine_cuts(len(x))]
    sf = _stream_fp(fpr, len(cut_sets), fan_value=fan)
    try:
        got, counts = run_streams(sf, [x] * len(cut_sets), cut_sets)
    finally:
        sf.close()
    for cuts, cnt, (h, t) in zip(cut_sets, counts, got):
        ends = np.cumsum(cuts)
        want = _rule_counts(fpr, x, fan, 10, ends[:-1]) + [len(t)]
        assert cnt == want


def test_ragged_streams_one_handle(fpr, synth_cases):
    rng = np.random.default_rng(7)
    totals = [0, 100, 4095, 4096, 4097, 6143, 6144, 441000, 2646000]
    tracks = [O.synth_track(100 + i, totals[i % len(totals)] + (0 if i < 2 * len(totals) else int(rng.integers(0, 5000))))
              for i in range(56)]
    kinds = list(synth_cases["kinds"])
    tracks += [synth_cases[f"{k}_pcm"] for k in kinds]
    cuts = []
    for x in tracks:
        c, pos = [], 0
        while pos < len(x) or not c:
            r = rng.random()
            size = 0 if r < 0.15 else int(rng.integers(1, 9000)) if r < 0.6 else int(rng.integers(9000, 200000))
            size = min(size, len(x) - pos)
            c.append(size)
            pos += size
        c += [0] * int(rng.integers(0, 3))           # empty blocks, the last one ends the stream
        cuts.append(c)
    sf = _stream_fp(fpr, len(tracks))
    try:
        got, _ = run_streams(sf, tracks, cuts)
    finally:
        sf.close()
    want = fpr.fingerprint_tracks(tracks)
    for b, (h, t) in enumerate(got):
        wh, wt = want.track(b)
        assert np.array_equal(h, wh) and np.array_equal(t, wt), (b, len(tracks[b]), len(t), len(wt))
    for i, k in enumerate(kinds):
        h, t = got[56 + i]
        assert np.array_equal(h, synth_cases[f"{k}_hash_fan5_amp10"]) and np.array_equal(t, synth_cases[f"{k}_t1_fan5_amp10"]), k


@pytest.mark.parametrize("kw", [dict(amp_min=0), dict(amp_min=-5, fan_value=15), dict(nbhd=3), dict(nbhd=16),
                                dict(compute="f32"), dict(connectivity=1, nbhd=7), dict(digest_table=True)])
def test_parameters_match_batch(fpr, kw):
    kw = dict(kw)
    table = kw.pop("digest_table", False)
    tracks = [O.synth_track(300 + i, n) for i, n in enumerate([30000, 4095, 250000, 600000])]
    cut_sets = [_cuts(len(tracks[0]), 3000), [len(tracks[1])], _cuts(len(tracks[2]), 8192), _cuts(len(tracks[3]), 44100)]
    if table:
        fpr.digest_table(True)
    try:
        sf = _stream_fp(fpr, len(tracks), **kw)
        try:
            got, _ = run_streams(sf, tracks, cut_sets)
        finally:
            sf.close()
        want = fpr.fingerprint_tracks(tracks, **kw)
    finally:
        if table:
            fpr.digest_table(False)
    for b, (h, t) in enumerate(got):
        wh, wt = want.track(b)
        assert np.array_equal(h, wh) and np.array_equal(t, wt), (b, kw)


@pytest.fixture(scope="module")
def fp_small(native_lib):
    from shazam_b200.fingerprinter import Fingerprinter
    f = Fingerprinter(0, max_chunk_frames=1024)
    yield f
    f.close()


def test_stream_longer_than_workspace(fp_small):
    from shazam_b200 import _native as N
    x = O.synth_track(11, 180 * 44100)
    with pytest.raises(N.CapacityError, match="frames"):
        fp_small.fingerprint_tracks([x])
    sf = _stream_fp(fp_small, 1)
    try:
        (got,), _ = run_streams(sf, [x], [_cuts(len(x), 441000)])
    finally:
        sf.close()
    wh, wt = O.fingerprint_arrays(x)
    assert np.array_equal(got[0], wh) and np.array_equal(got[1], wt)


def test_failure_leaves_state_untouched(fpr, fp_small):
    import torch
    from shazam_b200 import _native as N
    from shazam_b200.fingerprinter import pack_tracks
    x = O.synth_track(12, 30 * 44100)
    want = fpr.fingerprint_tracks([x]).track(0)
    # hash output too small, then a retry
    sf = _stream_fp(fpr, 1)
    try:
        hs, ts, pos = [], [], 0
        for c in _cuts(len(x), 100000):
            blk = x[pos:pos + c]
            pos += c
            pcm, starts, lens = pack_tracks([blk])
            d = torch.from_numpy(pcm).to(fpr.tdev)
            end = pos == len(x)
            with pytest.raises(N.CapacityError, match="hash output capacity"):
                sf.push_device(d, starts, lens, end=end, cap_hashes=0)
            r = sf.push_device(d, starts, lens, end=end)
            hs.append(r.hash.cpu().numpy()); ts.append(r.t1.cpu().numpy())
        assert np.array_equal(np.concatenate(hs), want[0]) and np.array_equal(np.concatenate(ts), want[1])
    finally:
        sf.close()
    # a block whose rows do not fit the workspace, then the same audio in smaller blocks
    y = O.synth_track(14, 90 * 44100)
    want = fpr.fingerprint_tracks([y]).track(0)
    sf = _stream_fp(fp_small, 1)
    try:
        r0 = sf.push([y[:50000]])
        with pytest.raises(N.CapacityError, match="rows"):
            sf.push([y[50000:50000 + 1500 * 2048]])
        (got,), _ = run_streams(sf, [y[50000:]], [_cuts(len(y) - 50000, 200000)])
        assert np.array_equal(np.concatenate([r0.hash, got[0]]), want[0])
        assert np.array_equal(np.concatenate([r0.t1, got[1]]), want[1])
    finally:
        sf.close()


def test_push_split_over_chunks_equals_one_chunk(fpr, fp_small):
    tracks = [O.synth_track(400 + i, 20 * 44100 + 977 * i) for i in range(40)]
    cuts = [_cuts(len(t), 2 * 44100) for t in tracks]
    results = []
    for fp in (fp_small, fpr):          # 1024 rows: ~106 rows per stream and push, 9 streams per chunk; 16384: one chunk
        sf = _stream_fp(fp, 40)
        try:
            results.append(run_streams(sf, tracks, cuts))
        finally:
            sf.close()
    (a, ca), (b, cb) = results
    assert ca == cb
    for (h1, t1), (h2, t2) in zip(a, b):
        assert np.array_equal(h1, h2) and np.array_equal(t1, t2)


def test_reset_and_reuse(fpr):
    x = O.synth_track(13, 10 * 44100 + 123)
    sf = _stream_fp(fpr, 2, fan_value=15)
    try:
        cuts = [_cuts(len(x), 5000), _cuts(len(x), 30000)]
        first, c1 = run_streams(sf, [x, x], cuts)
        second, c2 = run_streams(sf, [x, x], cuts)
    finally:
        sf.close()
    assert c1 == c2
    for (h1, t1), (h2, t2) in zip(first, second):
        assert np.array_equal(h1, h2) and np.array_equal(t1, t2) and len(t1) > 0


def test_recognizer_flow_two_channels(fpr):
    """recognizer.py:357-369 with one stream per channel: 26 reads of 8192 samples, hashes unioned and queried."""
    import torch
    from shazam_b200.database import FingerprintIndex
    songs = [O.synth_track(500 + i, 30 * 44100) for i in range(4)]
    ix = FingerprintIndex(0, capacity_rows=1 << 20)
    try:
        ref = fpr.fingerprint_tracks(songs)
        for s in range(len(songs)):
            h, t = ref.track(s)
            ix.insert(s + 1, h, t)
        n = 26 * 8192
        left, right = songs[2][100000:100000 + n], songs[2][100007:100007 + n]
        sf = _stream_fp(fpr, 2)
        try:
            parts = []
            for k in range(26):
                r = sf.push([left[k * 8192:(k + 1) * 8192], right[k * 8192:(k + 1) * 8192]], end=k == 25)
                parts.append(r)
            h = np.concatenate([p.track(c)[0] for c in (0, 1) for p in parts])
            t = np.concatenate([p.track(c)[1] for c in (0, 1) for p in parts])
        finally:
            sf.close()
        batch = fpr.fingerprint_tracks([left, right])
        assert np.array_equal(h, batch.hash) and np.array_equal(t, batch.t1)
        q = [ix.query_batch(torch.from_numpy(np.ascontiguousarray(hh)).to(fpr.tdev), torch.from_numpy(tt).to(fpr.tdev),
                            np.array([0, len(tt)], np.int64), 3) for hh, tt in ((h, t), (batch.hash, batch.t1))]
        for a, b in zip(q[0][:5], q[1][:5]):
            assert torch.equal(a, b)
        assert int(q[0][0][0, 0]) == 3
    finally:
        ix.close()
