#!/usr/bin/env python
"""Generate the committed golden vectors by EXECUTING THE REFERENCE'S OWN CODE.

Needs a checkout of the reference project, named by ``SIA_REFERENCE_DIR``:
``SIA_REFERENCE_DIR=<checkout> python tests/golden/make_golden.py [out_dir]``

How: the reference scripts cannot be imported (they open PortAudio / MySQL at
import and need matplotlib, pydub, ... which are absent), so the pure functions
``get_2D_peaks``, ``generate_hashes``, ``fingerprint`` (``__init__.py``) and
``return_matches``, ``align_matches`` (``recognizer.py``) plus the UPPER_CASE
module constants are AST-extracted from the reference files and exec'd
unmodified.  Two stand-ins are injected:

* ``mlab`` — ``mlab.specgram`` is the restated third-party call
  (``oracle.sia_oracle.specgram_psd``; matplotlib is not installed);
* ``db``   — an in-memory object answering ``SELECT_MULTIPLE`` /
  ``get_song_by_id`` (MySQL cannot run here).

Outputs (all under ``tests/golden/``):
  wav_fixture.npz   PCM of signal_with_noise.wav + reference peaks/hashes
  synth_cases.npz   seeded short clips (silence gaps, sub-frame input, ...) + reference hashes
  peaks_cases.npz   small float64 spectrograms (plateaus, zeros, negative amp_min) + reference peaks
  match_cases.json  reference return_matches + align_matches on small tables
  apriori_cases.json  reference return_matches of recognizer_apriori.py (early exit, :246-310) on small tables
  csv_cases.json    the five report files of the reference's generate_csv_results (recognizer_test.py:437-513)
  noise_cases.npz   reference get_noise_from_sound (recognizer_test.py:426-435) on seeded signal / noise pairs
"""
import ast
import hashlib
import json
import os
import sys
import warnings
import wave
from itertools import groupby
from operator import itemgetter

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = os.environ.get("SIA_REFERENCE_DIR", "")

from oracle import sia_oracle as O  # noqa: E402


def extract(path, func_names):
    """Compile the named FunctionDefs and every UPPER_CASE constant of `path`."""
    tree = ast.parse(open(path).read())
    keep = []
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and node.name in func_names:
            keep.append(node)
        elif isinstance(node, ast.Assign) and all(
                isinstance(t, ast.Name) and t.id.isupper() for t in node.targets):
            # constants only: literals and f-strings, no calls into pyaudio etc.
            if not any(isinstance(n, (ast.Call, ast.Attribute)) for n in ast.walk(node.value)):
                keep.append(node)
    return compile(ast.Module(body=keep, type_ignores=[]), path, "exec")


class _Mlab:
    window_hanning = staticmethod(lambda x: x)

    @staticmethod
    def specgram(x, NFFT, Fs, window, noverlap):
        return (O.specgram_psd(x, Fs, NFFT, noverlap), None, None)


def ref_namespace():
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from scipy.ndimage import (binary_erosion, generate_binary_structure,
                                   iterate_structure, maximum_filter)
    ns = dict(np=np, hashlib=hashlib, itemgetter=itemgetter, groupby=groupby, mlab=_Mlab,
              binary_erosion=binary_erosion, generate_binary_structure=generate_binary_structure,
              iterate_structure=iterate_structure, maximum_filter=maximum_filter)
    exec(extract(f"{REF}/__init__.py", {"get_2D_peaks", "generate_hashes", "fingerprint"}), ns)
    return ns


class _Cursor:
    def __init__(self, table):
        self.table, self.rows = table, []

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False

    def execute(self, query, params=None):
        assert "SELECT HEX(`hash`), `song_id`, `offset`" in query and "IN (" in query
        assert query.count("UNHEX(%s)") == len(params)
        self.rows = list(self.table.select_multiple(list(params)))

    def __iter__(self):
        return iter(self.rows)


class _Db:
    def __init__(self, table):
        self.table = table

    def cursor(self, **kw):
        return _Cursor(self.table)

    def get_song_by_id(self, sid):
        return self.table.get_song_by_id(sid)


def match_namespace(table):
    ns = dict(np=np, groupby=groupby, db=_Db(table))
    exec(extract(f"{REF}/recognizer.py", {"return_matches", "align_matches"}), ns)
    return ns


def apriori_namespace(table):
    ns = dict(np=np, groupby=groupby, db=_Db(table))
    exec(extract(f"{REF}/recognizer_apriori.py", {"return_matches", "align_matches"}), ns)
    return ns


def hashes_to_arrays(hs):
    if not hs:
        return np.zeros((0, 10), np.uint8), np.zeros((0,), np.int32)
    h = np.frombuffer(bytes.fromhex("".join(x[0] for x in hs)), np.uint8).reshape(-1, 10).copy()
    return h, np.array([int(x[1]) for x in hs], np.int32)


def synth_clip(kind, seed):
    rng = np.random.default_rng(seed)
    if kind == "tones":          # 3 s of the Config-2 generator
        return O.synth_track(seed, 3 * 44100)
    if kind == "gaps":           # music / digital silence / music: exact-zero frames (the 0 dB quirk)
        a = O.synth_track(seed, 44100 + 300)
        return np.concatenate([a, np.zeros(5 * 4096 + 123, np.int16), O.synth_track(seed + 1, 50000)])
    if kind == "noise":          # loud white noise: many peaks, full-scale clipping
        return np.clip(rng.normal(0, 12000, 60000), -32768, 32767).astype(np.int16)
    if kind == "short":          # shorter than one window -> zero padded to 4096
        return O.synth_track(seed, 3000)
    if kind == "oneframe":       # exactly 4096 samples
        return O.synth_track(seed, 4096)
    if kind == "ragged":         # 2 frames + a dropped partial tail
        return O.synth_track(seed, 4096 + 2048 + 2047)
    if kind == "silence":
        return np.zeros(30000, np.int16)
    if kind == "periodic":       # period divides the hop: identical frames -> plateaus along time
        base = (8000 * np.sin(2 * np.pi * np.arange(2048) * 37 / 2048) +
                3000 * np.sin(2 * np.pi * np.arange(2048) * 300 / 2048)).round().astype(np.int16)
        return np.tile(base, 40)
    if kind == "longgap":        # two bursts > 200 frames apart -> dt > MAX_HASH_TIME_DELTA rejected
        a = O.synth_track(seed, 20000)
        return np.concatenate([a, np.zeros(215 * 2048, np.int16), O.synth_track(seed + 7, 20000)])
    raise KeyError(kind)


def main(out_dir=HERE):
    """Writes the four fixture files into ``out_dir`` (default: this directory, i.e. the committed fixtures)."""
    ns = ref_namespace()
    out = {}

    # ---- wav fixture (BASELINE.json configs[0]) ---------------------------------
    w = wave.open(f"{REF}/signal_with_noise.wav")
    assert (w.getnchannels(), w.getsampwidth(), w.getframerate()) == (1, 2, 22050)
    pcm = np.frombuffer(w.readframes(w.getnframes()), np.int16).copy()
    out["pcm"] = pcm
    out["fs"] = np.int64(22050)
    for conn in (2, 1):
        ns["CONNECTIVITY_MASK"] = conn
        arr = O.spectrogram_db(pcm, 22050)
        pk = ns["get_2D_peaks"](arr, amp_min=10)
        out[f"peaks_c{conn}"] = np.array(pk, np.int32).reshape(-1, 2)      # (f, t) freq-major
        for fan in (5, 15):
            for fs in (22050, 44100):
                h, t = hashes_to_arrays(ns["fingerprint"](pcm, Fs=fs, fan_value=fan, amp_min=10))
                out[f"hash_c{conn}_fan{fan}_fs{fs}"] = h
                out[f"t1_c{conn}_fan{fan}_fs{fs}"] = t
    ns["CONNECTIVITY_MASK"] = 2
    # list-of-python-ints input, as the recorder passes it (recognizer.py:361-368)
    h, t = hashes_to_arrays(ns["fingerprint"]([int(v) for v in pcm[:50000]], Fs=44100))
    out["hash_list50k"], out["t1_list50k"] = h, t
    np.savez_compressed(f"{out_dir}/wav_fixture.npz", **out)
    print("wav: peaks", len(out["peaks_c2"]), "hashes fan5", len(out["hash_c2_fan5_fs22050"]),
          "fan15", len(out["hash_c2_fan15_fs22050"]), "diamond peaks", len(out["peaks_c1"]))

    # ---- synthetic clips -----------------------------------------------------------
    out = {}
    kinds = ["tones", "gaps", "noise", "short", "oneframe", "ragged", "silence", "periodic", "longgap"]
    out["kinds"] = np.array(kinds)
    for i, kind in enumerate(kinds):
        x = synth_clip(kind, 100 + i)
        out[f"{kind}_pcm"] = x
        for fan, amp in ((5, 10), (15, 10), (15, 0), (15, -5)):
            h, t = hashes_to_arrays(ns["fingerprint"](x, Fs=44100, fan_value=fan, amp_min=amp))
            out[f"{kind}_hash_fan{fan}_amp{amp}"] = h
            out[f"{kind}_t1_fan{fan}_amp{amp}"] = t
        print(kind, len(x), "samples ->", len(out[f"{kind}_hash_fan15_amp10"]), "hashes @fan15")
    np.savez_compressed(f"{out_dir}/synth_cases.npz", **out)

    # ---- raw peak cases: small float64 spectrograms ----------------------------------
    out = {}
    rng = np.random.default_rng(7)
    cases = {
        "rand": rng.normal(5, 12, (90, 70)),
        "quant": np.round(rng.normal(8, 8, (64, 120))),                     # many exact ties
        "zeros": np.where(rng.random((80, 80)) < 0.7, 0.0, rng.normal(0, 15, (80, 80))),
        "allzero": np.zeros((40, 50)),
        "const": np.full((30, 45), 12.5),
        "neg": rng.normal(-30, 5, (50, 50)),
        "tiny": rng.normal(15, 5, (5, 3)),
        "onecol": rng.normal(15, 5, (2049, 1)),
        "fullF": rng.normal(0, 14, (2049, 24)),
    }
    block = np.zeros((70, 70))
    block[:, 35:] = rng.normal(0, 15, (70, 35))                              # zero background next to signal
    cases["halfzero"] = block
    out["names"] = np.array(list(cases))
    for name, arr in cases.items():
        out[f"{name}_arr"] = arr
        for conn in (2, 1):
            ns["CONNECTIVITY_MASK"] = conn
            for amp in (10, 0, -5, -100):
                pk = ns["get_2D_peaks"](arr, amp_min=amp)
                out[f"{name}_c{conn}_amp{amp}"] = np.array(pk, np.int32).reshape(-1, 2)
    ns["CONNECTIVITY_MASK"] = 2
    np.savez_compressed(f"{out_dir}/peaks_cases.npz", **out)

    # ---- match cases ---------------------------------------------------------------
    mcases = []
    rng = np.random.default_rng(11)

    def hx(i):
        return hashlib.sha1(str(i).encode()).hexdigest()[:20]

    for case_id, (nsongs, per_song, universe, nquery) in enumerate(
            [(3, 40, 25, 30), (8, 300, 120, 200), (5, 60, 10, 40), (4, 50, 30, 0)]):
        table = O.FingerprintTable()
        rows = []
        for s in range(nsongs):
            sid = table.insert_song(f"song{s}", hashlib.sha1(f"file{s}".encode()).hexdigest().upper(), per_song)
            hs = [(hx(int(rng.integers(0, universe))), int(rng.integers(0, 60))) for _ in range(per_song)]
            hs += hs[:5]                                    # duplicates -> INSERT IGNORE
            table.insert_hashes(sid, hs)
            table.set_song_fingerprinted(sid)
            rows += [[sid, h, o] for h, o in hs]
        # query = a time-shifted excerpt of song 2 + random hashes (some absent from the table)
        target = [r for r in rows if r[0] == min(2, nsongs)]
        q = [(h, max(0, o - 7)) for _, h, o in target[: nquery // 2]]
        q += [(hx(int(rng.integers(0, universe * 2))), int(rng.integers(0, 20))) for _ in range(nquery - len(q))]
        q = list(set(q))
        q.sort()
        mns = match_namespace(table)
        matches, dedup = mns["return_matches"](q)
        by_topn = {}
        for topn in (1, 2, 3, 50):
            res = mns["align_matches"](matches, dedup, len(q), topn) if q else []
            by_topn[str(topn)] = [{k: (v.decode() if isinstance(v, bytes) else v) for k, v in r.items()}
                                  for r in res]
        mcases.append({
            "case": case_id, "rows": rows, "query": q,
            "songs": {str(k): v for k, v in table.songs.items()},
            "n_matches": len(matches),
            "matches_sorted_sha": hashlib.sha256(repr(sorted(matches)).encode()).hexdigest(),
            "dedup": {str(k): v for k, v in dedup.items()},
            "results_by_topn": by_topn,
        })
    # the KAT of SURVEY.md §8c
    table = O.FingerprintTable()
    for s in range(9):
        table.insert_song(f"s{s + 1}", "AB" * 20, 100)
    mns = match_namespace(table)
    kat = mns["align_matches"]([(7, 3), (7, 3), (7, 5), (2, 10), (2, 10), (2, -4), (2, -4), (9, 1)],
                               {7: 3, 2: 4, 9: 1}, 10, 3)
    mcases.append({"case": "kat", "results": [{k: (v.decode() if isinstance(v, bytes) else v)
                                               for k, v in r.items()} for r in kat]})
    json.dump(mcases, open(f"{out_dir}/match_cases.json", "w"), indent=0)
    print("match cases:", len(mcases))

    # ---- a-priori early exit (SURVEY §8f-4): recognizer_apriori.py's return_matches, executed from its source --------
    import contextlib
    import io
    acases = []
    rng = np.random.default_rng(23)
    for case_id, (nsongs, per_song, universe, nquery, batch, twin) in enumerate(
            [(6, 300, 3000, 200, 20, False), (5, 200, 150, 120, 16, True), (4, 120, 90, 60, 1000, False),
             (8, 250, 1200, 160, 10, False), (8, 250, 600, 160, 5, False)]):
        table = O.FingerprintTable()
        rows = []
        for s in range(nsongs):
            sid = table.insert_song(f"song{s}", hashlib.sha1(f"afile{s}".encode()).hexdigest().upper(), per_song)
            if twin and s == 2:
                hs = [(h, o) for _, h, o in rows if _ == 2]         # song 3 = a copy of song 2: the exit never triggers
            else:
                hs = [(hx(int(rng.integers(0, universe))), int(rng.integers(0, 80))) for _ in range(per_song)]
            table.insert_hashes(sid, hs)
            table.set_song_fingerprinted(sid)
            rows += [[sid, h, o] for h, o in hs]
        target = [r for r in rows if r[0] == 2]
        q = [(h, max(0, o - 5)) for _, h, o in target[: (3 * nquery) // 4]]
        q += [(hx(int(rng.integers(0, universe))), int(rng.integers(0, 30))) for _ in range(nquery - len(q))]
        q = sorted(set(q))                                          # the batches follow this order
        ans = apriori_namespace(table)
        with contextlib.redirect_stdout(io.StringIO()):
            matches, dedup, songs_arr = ans["return_matches"](q, batch)
        acases.append({
            "case": case_id, "rows": rows, "query": q, "batch_size": batch,
            "songs": {str(k): v for k, v in table.songs.items()},
            "n_matches": len(matches),
            "matches_sorted_sha": hashlib.sha256(repr(sorted(matches)).encode()).hexdigest(),
            "dedup": {str(k): v for k, v in dedup.items()},
            "songs_arr": [{k: (v.decode() if isinstance(v, bytes) else v) for k, v in r.items()} for r in songs_arr],
        })
        full, _ = match_namespace(table)["return_matches"](q)
        print(f"apriori case {case_id}: {len(matches)} of {len(full)} matches read, exit={'yes' if songs_arr else 'no'}")
    json.dump(acases, open(f"{out_dir}/apriori_cases.json", "w"), indent=0)

    # ---- the experiment script's report (SURVEY §8f-3): generate_csv_results executed from its source ----------------
    # Stand-ins: `datetime` (a fixed stamp), `times` (the script's module global), and `pd.crosstab` returning an
    # object-dtype frame — the script writes str(0) / str(1) into the crosstab (:497-498), which the pandas of its era
    # (python 3.7) upcast silently and pandas 3 refuses; nothing else is touched.
    import csv as _csv
    import re as _re
    import tempfile
    import pandas as pd
    from sklearn.metrics import accuracy_score, classification_report, confusion_matrix

    class _DT:
        class datetime:
            @staticmethod
            def now():
                class _Now:
                    def strftime(self, fmt):
                        return "01-01-2021_00-00-00"
                return _Now()

    class _PD:
        Series, DataFrame = pd.Series, pd.DataFrame
        crosstab = staticmethod(lambda a, b: pd.crosstab(a, b).astype(object))

    ccases = []
    crng = np.random.default_rng(77)
    pool = [f"{100000 + 37 * i}" for i in range(15)]                # numeric track names like the reference's mp3 files
    big_played = [pool[int(i)] for i in crng.integers(0, 15, 60)]
    big_pred = [t if crng.random() < 0.75 else (pool[int(crng.integers(0, 15))] if crng.random() < 0.7 else f"other{int(crng.integers(0, 4))}")
                for t in big_played]
    for case_id, (played, pred, add_noise, snr, secs, it) in enumerate([
            (["a", "b", "c", "d", "e", "f", "g", "h"], ["a", "b", "x", "d", "a", "f", "g", "b"], True, 10, 5, 3),
            (["t1", "t2", "t3", "t2"], ["t1", "t2", "t3", "t2"], False, 0, 15, 0),
            (["k", "a", "k", "m", "q", "b", "q"], ["zz", "a", "k", "m", "c", "a", "q"], True, 0, 5, 678),
            (big_played, big_pred, False, 0, 15, 2713)]):
        songs = [f"songs/{i % 3:03d}/{n}.mp3" for i, n in enumerate(played)]
        tms = [{"song_start_time": 7 * i, "fingerprint_times": 0.25 + 0.01 * i, "query_time": 0.05 * (i + 1),
                "align_time": 0.01, "total_time": 0.31 + 0.06 * i} for i in range(len(played))]
        finals = [str([{"song_id": i + 1, "song_name": p}]) for i, p in enumerate(pred)]
        cns = dict(re=_re, csv=_csv, datetime=_DT, pd=_PD, confusion_matrix=confusion_matrix,
                   classification_report=classification_report, accuracy_score=accuracy_score, times=tms,
                   print=lambda *a, **k: None)
        exec(extract(f"{REF}/recognizer_test.py", {"generate_csv_results"}), cns)
        cns.update(ADD_NOISE=add_noise, SNR=snr, RECORD_SECONDS=secs)     # the script's run-time switches (:38-40)
        cwd = os.getcwd()
        with tempfile.TemporaryDirectory() as td:
            os.chdir(td)
            try:
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    cns["generate_csv_results"](songs, pred, it, finals)
                files = {f: open(f, newline="").read() for f in sorted(os.listdir("."))}
            finally:
                os.chdir(cwd)
        assert len(files) == 5
        ccases.append({"case": case_id, "songs_to_recognize": songs, "recognized_song_names": pred, "times": tms,
                       "final_results_arr": finals, "add_noise": add_noise, "snr": snr, "record_seconds": secs,
                       "iteration": it, "stamp": "01-01-2021_00-00-00", "files": files})
    json.dump(ccases, open(f"{out_dir}/csv_cases.json", "w"), indent=0)
    print("csv cases:", len(ccases))

    # ---- SNR mixer of the experiment script (SURVEY §8f-3) ----------------------------------------------
    import math
    nns = dict(np=np, math=math)
    exec(extract(f"{REF}/recognizer_test.py", {"get_noise_from_sound"}), nns)
    out = {"snrs": np.array([0.0, 10.0, -5.0, 3.5])}
    rng = np.random.default_rng(2024)
    for k, n in enumerate((2048, 8192)):
        # the script rescales both to [-1, 1] before the call (recognizer_test.py:547-551); keep that range
        t = np.arange(n) / 22050.0
        signal = 0.6 * np.sin(2 * np.pi * 440 * t) + 0.2 * rng.standard_normal(n)
        signal = np.interp(signal, (signal.min(), signal.max()), (-1, 1))
        noise = np.cumsum(rng.standard_normal(n))                  # coloured, non-zero mean
        noise = np.interp(noise, (noise.min(), noise.max()), (-1, 1))
        out[f"signal_{k}"], out[f"noise_{k}"] = signal, noise
        for j, snr in enumerate(out["snrs"]):
            out[f"scaled_{k}_{j}"] = nns["get_noise_from_sound"](signal, noise, float(snr))
    np.savez_compressed(f"{out_dir}/noise_cases.npz", **out)
    print("noise cases: 2 x", len(out["snrs"]))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else HERE)
