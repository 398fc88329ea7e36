"""Match side of the reference interface (``recognizer.py:222-338``) on the GPU index.

``return_matches`` / ``find_matches`` / ``align_matches`` keep the reference's signatures and
result shapes and work on the module global ``db`` exactly like the scripts do (set it with
``set_database``).  ``recognize_batch`` is the array fast path that never materialises the
``(song_id, offset_difference)`` tuple list: lookup, vote and top-n stay on the device.
"""
from __future__ import annotations

from time import time
from typing import Optional, Sequence

import numpy as np
import torch

from . import _native as N
from .database import GPUDatabase, vote_tuples
from .fingerprinter import hex_to_digests

# result-dict keys and constants, recognizer.py:30-68
DEFAULT_FS = 44100
DEFAULT_WINDOW_SIZE = 4096
DEFAULT_OVERLAP_RATIO = 0.5
SONG_ID = "song_id"
SONG_NAME = "song_name"
FIELD_TOTAL_HASHES = "total_hashes"
INPUT_HASHES = "input_total_hashes"
INPUT_CONFIDENCE = "input_confidence"
FINGERPRINTED_HASHES = "fingerprinted_hashes_in_db"
HASHES_MATCHED = "hashes_matched_in_input"
FINGERPRINTED_CONFIDENCE = "fingerprinted_confidence"
OFFSET = "offset"
OFFSET_SECS = "offset_seconds"
FIELD_FILE_SHA1 = "file_sha1"
TOPN = 2

db: Optional[GPUDatabase] = None


def set_database(database: GPUDatabase) -> None:
    global db
    db = database


def return_matches(hashes, batch_size: int = 1000, apriori: bool = False):
    """``recognizer.py:222-271``: ``(results, dedup_hashes)`` with ``results`` a list of
    ``(song_id, db_offset - query_offset)`` and ``dedup_hashes[song_id]`` the number of DB rows
    matched (each row once, however many query offsets share its hash).

    ``apriori=True`` is the early exit of ``recognizer_apriori.py:297-308`` (SURVEY §8f-4): after every batch of
    ``batch_size`` distinct hashes the matches so far are aligned, and the lookup stops as soon as the best song has
    more than twice the matched hashes of the runner-up.  It changes ``hashes_matched`` (fewer batches are read), so
    it is off by default and outside the parity tests; the return value then has the reference's third element,
    the aligned results at the point of exit (``[]`` if the exit never triggered).  This is the tuple-returning
    drop-in; ``recognize_batch(..., apriori_batch=batch_size)`` runs the same rule on the device for many queries."""
    mapper = {}
    for hsh, offset in hashes:
        mapper.setdefault(hsh.upper(), []).append(offset)
    values = list(mapper.keys())
    dedup_hashes = {}
    results = []
    songs_arr = []
    with db.cursor() as cur:
        for index in range(0, len(values), batch_size):
            batch = values[index: index + batch_size]
            cur.execute(db.SELECT_MULTIPLE % ", ".join([db.IN_MATCH] * len(batch)), batch)
            for hsh, sid, offset in cur:
                dedup_hashes[sid] = dedup_hashes.get(sid, 0) + 1
                for song_sampled_offset in mapper[hsh]:
                    results.append((sid, offset - song_sampled_offset))
            if apriori:
                songs_arr = align_matches(results, dedup_hashes, len(hashes))
                if len(songs_arr) > 1 and songs_arr[0][HASHES_MATCHED] / 2 > songs_arr[1][HASHES_MATCHED]:
                    break
                songs_arr = []
    if apriori:
        return results, dedup_hashes, songs_arr
    return results, dedup_hashes


def find_matches(hashes):
    """``recognizer.py:273-286``."""
    t = time()
    matches, dedup_hashes = return_matches(hashes)
    return matches, dedup_hashes, time() - t


def _result_dict(song_id: int, offset: int, hashes_matched: int, queried_hashes: int) -> dict:
    song = db.get_song_by_id(song_id)
    song_hashes = song.get(FIELD_TOTAL_HASHES, None)
    nseconds = round(float(offset) / DEFAULT_FS * DEFAULT_WINDOW_SIZE * DEFAULT_OVERLAP_RATIO, 5)
    return {
        SONG_ID: song_id,
        SONG_NAME: song.get(SONG_NAME, None).encode("utf8"),
        INPUT_HASHES: queried_hashes,
        FINGERPRINTED_HASHES: song_hashes,
        HASHES_MATCHED: hashes_matched,
        INPUT_CONFIDENCE: round(hashes_matched / queried_hashes, 2),
        FINGERPRINTED_CONFIDENCE: round(hashes_matched / song_hashes, 2),
        OFFSET: offset,
        OFFSET_SECS: nseconds,
        FIELD_FILE_SHA1: song.get(FIELD_FILE_SHA1, None).encode("utf8"),
    }


def align_matches(matches, dedup_hashes, queried_hashes, topn: int = TOPN):
    """``recognizer.py:289-338``.  The vote (sort, run-length count, per-song first maximum,
    stable descending sort) runs on the GPU: the tuples are uploaded as vote keys (``sia_vote_tuples``)."""
    if len(matches) == 0:
        return []
    m = np.asarray(matches, dtype=np.int64).reshape(-1, 2)
    sid, diff = m[:, 0], m[:, 1]
    if sid.min() < 0 or sid.max() >= 1 << 24 or np.abs(diff).max() >= 1 << 24:
        raise N.SiaError(N.E_INVALID, "song ids / offset differences outside the 24-bit range")
    # vote keys of query 0 without the head flag (dedup_hashes comes from the caller's dict), sia_b200.h
    key = torch.from_numpy((sid << 25) | (diff + (1 << 24))).to(db.index.tdev)
    song, dif, cnt, rows, nres = vote_tuples(db.index.device, key, 1, int(topn), int(sid.max()))
    k = int(nres[0].item())
    song = song[0, :k].cpu().tolist()
    dif = dif[0, :k].cpu().tolist()
    return [_result_dict(s, d, dedup_hashes[s], queried_hashes) for s, d in zip(song, dif)]


def recognize_batch(queries: Sequence, topn: int = TOPN, want_stats: bool = False, apriori_batch: Optional[int] = None):
    """Array fast path for many queries at once.  ``queries[i]`` is ``(digests uint8[n,10],
    offsets int32[n])`` (host arrays or CUDA tensors).  Returns, per query, the list of result
    dicts ``align_matches`` would return for ``len(set(pairs))`` queried hashes.

    ``apriori_batch=B`` applies the early exit of ``recognizer_apriori.py:246-310`` on the device
    (``FingerprintIndex.query_batch_apriori``): the distinct hashes are read in batches of B in ascending digest
    order, and a query's results are those at the batch where its best song first had more than twice the matched
    rows of the runner-up (``hashes_matched_in_input`` = rows read up to then), else those of the whole query."""
    index = db.index
    dig, off, starts, nq_hashes = [], [], [0], []
    for d, o in queries:
        d = torch.as_tensor(d).to(index.tdev).reshape(-1, N.HASH_BYTES)
        o = torch.as_tensor(o).to(index.tdev, dtype=torch.int32)
        dig.append(d); off.append(o)
        starts.append(starts[-1] + o.numel())
    if not dig:
        return []
    D = torch.cat(dig) if dig else torch.empty((0, N.HASH_BYTES), dtype=torch.uint8, device=index.tdev)
    O = torch.cat(off)
    if apriori_batch is None:
        out = index.query_batch(D, O, np.array(starts, np.int64), topn, want_stats=want_stats)
    else:
        out = index.query_batch_apriori(D, O, np.array(starts, np.int64), topn, apriori_batch, want_stats=want_stats)
    song, dif, cnt, rows, nres = [t.cpu().numpy() for t in out[:5]]
    results = []
    for q in range(len(queries)):
        # queried_hashes = len(set of (hash, offset) pairs), as the callers pass len(hashes) of a set
        s, e = starts[q], starts[q + 1]
        if e > s:
            pairs = torch.cat([D[s:e].to(torch.int32), O[s:e, None]], 1)
            nq = int(torch.unique(pairs, dim=0).shape[0])
        else:
            nq = 0
        results.append([_result_dict(int(song[q, r]), int(dif[q, r]), int(rows[q, r]), nq) for r in range(int(nres[q]))])
    if want_stats:
        return results, out[-1]
    return results


def hashes_to_arrays(hashes):
    """``[(hex20, offset), ...]`` -> (uint8[n,10], int32[n])."""
    hashes = list(hashes)
    return hex_to_digests([h for h, _ in hashes]), np.array([int(t) for _, t in hashes], np.int32)
