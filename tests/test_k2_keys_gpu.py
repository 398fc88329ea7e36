"""Edge cases of the pipeline's K2 kernel (float32, square 21x21, amp_min >= 0), aimed at any filter that compares
quantised values and settles ties on the float32 ones (such as 16-bit order keys spanning 128 dB above the threshold,
DESIGN §8 (5)): neighbours one float ulp or one 128/65535 dB step apart, values at and around the threshold, values at
and above threshold + 128 dB with plateaus wider than the window, ragged multi-track layouts with 1e30 row padding, and
the float32 spectrogram of full-length tracks.  Every case must give exactly the oracle's peaks on the same float32
array."""
import numpy as np
import pytest

from oracle import sia_oracle as O

pytestmark = pytest.mark.gpu

F = 2049
KEY_RANGE = 128.0                     # dB spanned by the 65535 key steps above the threshold
KEY_STEP = KEY_RANGE / 65535


def _lo(amp):
    """amp_min rounded down to float32: the threshold the keys are built against."""
    lo = np.float32(amp)
    if float(lo) > amp:
        lo = np.nextafter(lo, np.float32(-np.inf))
    return lo


def _run(fpr, arrs, amp):
    """K2 on a ragged multi-track float32 layout ([F][T] arrays), row padding 1e30; per-track (t, f) lists of the
    device and of the oracle."""
    import torch
    frames = [a.shape[1] for a in arrs]
    host = np.zeros((sum(frames), 2080), np.float32)
    host[:, F:] = 1e30
    r = 0
    for a in arrs:
        host[r:r + a.shape[1], :F] = a.T
        r += a.shape[1]
    spec = torch.from_numpy(host).to(fpr.tdev)
    pt, pf, tps = fpr.peaks(spec, np.array(frames, np.int64), fpr.params(amp_min=amp))
    tps = tps.cpu().numpy(); pt = pt.cpu().numpy(); pf = pf.cpu().numpy()
    for k, a in enumerate(arrs):
        want = sorted((int(t), int(f)) for f, t in O.get_2D_peaks(a.astype(np.float64), amp))
        got = list(zip(pt[tps[k]:tps[k + 1]].tolist(), pf[tps[k]:tps[k + 1]].tolist()))
        yield k, got, want


def _centres(rng, T, n):
    return rng.integers(0, F, n), rng.integers(0, T, n)


def _key_edge_tracks(rng, lo):
    """Tracks built around the threshold lo (float32) of one run."""
    lo = np.float32(lo)
    up = lambda x: np.nextafter(np.float32(x), np.float32(np.inf))
    down = lambda x: np.nextafter(np.float32(x), np.float32(-np.inf))
    arrs = []
    # 1. ties of one float ulp and of one key step: a value and a neighbour just above / below it, inside the window
    for T, step in [(130, None), (75, KEY_STEP), (64, KEY_STEP / 3), (97, 2 * KEY_STEP)]:
        a = rng.normal(float(lo) + 20, 8, (F, T)).astype(np.float32)
        fs, ts = _centres(rng, T, 600)
        for f, t in zip(fs, ts):
            v = np.float32(float(lo) + rng.uniform(0, 150))
            f2 = min(F - 1, max(0, f + int(rng.integers(-10, 11))))
            t2 = min(T - 1, max(0, t + int(rng.integers(-10, 11))))
            a[f, t] = v
            if step is None:
                a[f2, t2] = up(v) if rng.random() < 0.5 else (down(v) if rng.random() < 0.5 else v)
            else:
                a[f2, t2] = np.float32(float(v) + step * rng.choice([-1.0, -0.5, 0.5, 1.0]))
        arrs.append(a)
    # 2. the threshold: isolated maxima at lo, just above and below it, at 0 and below, over a floor far below
    T = 120
    a = rng.normal(-40, 5, (F, T)).astype(np.float32)
    vals = np.array([lo, up(lo), up(up(lo)), down(lo), 0.0, -0.0, -3.0, -np.inf, np.float32(float(lo) + KEY_STEP / 2),
                     np.float32(float(lo) + 1e-3), np.float32(float(lo) + KEY_STEP)], np.float32)
    fs, ts = _centres(rng, T, 800)
    a[fs, ts] = vals[rng.integers(0, len(vals), len(fs))]
    arrs.append(a)
    # the same values as a dense field: every window mixes them, with ties of every kind
    arrs.append(vals[rng.integers(0, len(vals), (F, 66))])
    # 3. saturation: values at and above lo + 128 dB, plateaus wider than the window, one larger float inside some
    T = 140
    sat = np.float32(float(lo) + KEY_RANGE)
    a = rng.normal(float(lo) + 100, 20, (F, T)).astype(np.float32)
    a[200:260, 10:60] = sat                                            # a plateau of saturated keys
    a[600:640, 30:90] = np.float32(float(lo) + 300)
    a[620, 55] = np.float32(float(lo) + 300.5)                        # the one peak of that plateau, by its float
    a[1000:1040, 70:130] = down(sat)
    a[1500:1530, 0:T] = 1e6
    a[1515, 77] = up(np.float32(1e6))
    fs, ts = _centres(rng, T, 600)
    a[fs, ts] = np.float32(float(lo) + KEY_RANGE) + rng.choice([-KEY_STEP, 0, KEY_STEP, 1.0, 1e3, 3e38], len(fs))
    arrs.append(a)
    # 4. short tracks: tiles that cross track borders at every offset
    for T in (1, 7, 21, 65, 11):
        arrs.append(rng.normal(float(lo) + 5, 10, (F, T)).astype(np.float32))
    return arrs


def test_k2_keys_edges(fpr):
    rng = np.random.default_rng(2024)
    for amp in (0, 10, 10.1, 40):
        arrs = _key_edge_tracks(rng, _lo(amp))
        for k, got, want in _run(fpr, arrs, amp):
            assert got == want, (amp, k, len(got), len(want))


def test_k2_keys_threshold_above_every_value(fpr):
    rng = np.random.default_rng(7)
    arrs = _key_edge_tracks(rng, _lo(10))
    top = max(float(a[np.isfinite(a)].max()) for a in arrs)
    n = 0
    for k, got, want in _run(fpr, arrs, top * 1.5):
        assert got == want == [], (k, len(got))
        n += 1
    assert n == len(arrs)


def test_k2_keys_full_size_tracks(fpr):
    """K1's float32 dB of two full-length bench-recipe tracks (3 min at 44.1 kHz): K2's peaks equal the oracle's
    get_2D_peaks on that same float32 array."""
    import torch
    from shazam_b200.fingerprinter import pack_tracks
    tracks = [O.synth_track(10_000 + i, 7_938_000) for i in range(2)]
    pcm, starts, lens = pack_tracks(tracks)
    d = torch.from_numpy(pcm).to(fpr.tdev)
    p = fpr.params()
    spec = fpr.stft_db(d, starts, lens, p, out_dtype=torch.float32)
    frames = np.array([(n - 4096) // 2048 + 1 for n in lens], np.int64)
    assert int(frames.sum()) == spec.shape[0]
    pt, pf, tps = fpr.peaks(spec, frames, p)
    tps = tps.cpu().numpy(); pt = pt.cpu().numpy(); pf = pf.cpu().numpy()
    host = spec[:, :F].cpu().numpy()
    r = 0
    for k, T in enumerate(frames.tolist()):
        a = host[r:r + T].T.astype(np.float64)
        r += T
        want = sorted((int(t), int(f)) for f, t in O.get_2D_peaks(a, p.amp_min))
        got = list(zip(pt[tps[k]:tps[k + 1]].tolist(), pf[tps[k]:tps[k + 1]].tolist()))
        assert len(want) > 10_000
        assert got == want, (k, len(got), len(want))
