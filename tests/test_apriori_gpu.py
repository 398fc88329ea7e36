"""The a-priori early exit on the device (sia_index_query_apriori, recognizer_apriori.py:246-310) against the
reference's own outputs (apriori_cases.json) and against the pinned full vote (query_batch) run on prefix queries:
batches 0..k of a query as a query of their own, the exit rule applied on the host."""
import hashlib
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _strip(results):
    return [{k: (v.decode() if isinstance(v, bytes) else v) for k, v in r.items()} for r in results]


@pytest.fixture()
def torch_dev(native_lib):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


@pytest.fixture()
def gpudb(torch_dev):
    from shazam_b200.database import GPUDatabase
    from shazam_b200 import recognize
    made = []

    def make(**kw):
        d = GPUDatabase(device=0, capacity_rows=kw.pop("capacity_rows", 1 << 20), **kw)
        recognize.set_database(d)
        made.append(d)
        return d
    yield make
    for d in made:
        d.index.close()


def _load_case(db, case):
    for sid, s in sorted(case["songs"].items(), key=lambda kv: int(kv[0])):
        assert db.insert_song(s["song_name"], s["file_sha1"], s["total_hashes"]) == int(sid)
    by_song = {}
    for sid, h, o in case["rows"]:
        by_song.setdefault(sid, []).append((h, o))
    for sid, hs in by_song.items():
        db.insert_hashes(sid, hs)
        db.set_song_fingerprinted(sid)


def test_apriori_golden(gpudb):
    """The reference's a-priori return_matches, executed from its source: the same results where it exits, the
    whole-query results where it never does, and the same tuples and rows read."""
    import torch
    from shazam_b200 import recognize
    cases = json.load(open(os.path.join(GOLDEN, "apriori_cases.json")))
    exits = 0
    for case in cases:
        db = gpudb()
        _load_case(db, case)
        q = [tuple(x) for x in case["query"]]
        B = case["batch_size"]
        got = recognize.recognize_batch([recognize.hashes_to_arrays(q)], topn=2, apriori_batch=B)[0]
        d, o = recognize.hashes_to_arrays(q)
        out = db.index.query_batch_apriori(torch.from_numpy(d).to(db.index.tdev), torch.from_numpy(o).to(db.index.tdev),
                                           np.array([0, len(q)]), 2, B, want_stats=True)
        ex, stats = int(out[6][0].item()), out[7]
        if case["songs_arr"]:
            assert _strip(got) == case["songs_arr"], case["case"]
            assert ex == 1
            exits += 1
        else:
            matches, dedup, _ = recognize.find_matches(q)
            assert _strip(got) == _strip(recognize.align_matches(matches, dedup, len(q))), case["case"]
            assert ex == 0
            assert int(out[5][0].item()) == -(-len({h for h, _ in q}) // B)
        assert stats[2] == case["n_matches"], case["case"]
        assert stats[1] == sum(case["dedup"].values()), case["case"]
    assert exits == 3


# ---- the independent check: prefix queries through the pinned full vote ----------------------------------------------
def _prefix_reference(ix, qd_h, qo_h, qs, B, topn_max):
    """Per query: the full vote of every prefix (batches 0..k, distinct hashes in ascending digest order), and the
    expected a-priori outputs for each topn <= topn_max."""
    import torch
    nq = len(qs) - 1
    pd, po, starts, owner, nb = [], [], [0], [], []
    for q in range(nq):
        d, o = qd_h[qs[q]:qs[q + 1]], qo_h[qs[q]:qs[q + 1]]
        keys = [bytes(r) for r in d]
        uniq = sorted(set(keys))
        k_q = -(-len(uniq) // B)
        nb.append(k_q)
        for k in range(k_q):
            allowed = set(uniq[:(k + 1) * B])
            sel = np.array([x in allowed for x in keys])
            pd.append(d[sel]); po.append(o[sel]); starts.append(starts[-1] + int(sel.sum())); owner.append((q, k))
    dev = ix.tdev
    L = max(topn_max, 2)
    if owner:
        res = [t.cpu().numpy() for t in ix.query_batch(torch.from_numpy(np.concatenate(pd)).to(dev),
                                                       torch.from_numpy(np.concatenate(po)).to(dev),
                                                       np.array(starts, np.int64), L)]
    pick = {}                                   # query -> (prefix index, batches read, fired)
    for p, (q, k) in enumerate(owner):
        if q in pick and pick[q][2]:
            continue
        song, diff, cnt, rows, nres = (r[p] for r in res)
        fired = nres >= 2 and rows[0] > 2 * rows[1]
        pick[q] = (p, k + 1, fired)
    chosen = [pick[q][0] for q in range(nq) if q in pick]
    sel_starts = np.concatenate([[0], np.cumsum([starts[p + 1] - starts[p] for p in chosen])]).astype(np.int64)
    stats = [0, 0, 0, 0]
    if chosen:
        stats = ix.query_batch(torch.from_numpy(np.concatenate([pd[p] for p in chosen])).to(dev),
                               torch.from_numpy(np.concatenate([po[p] for p in chosen])).to(dev), sel_starts, L,
                               want_stats=True)[5]

    def expected(topn):
        out = [np.zeros((nq, topn), np.int32) for _ in range(4)] + [np.zeros(nq, np.int32) for _ in range(3)]
        for q in range(nq):
            out[5][q] = nb[q]
            if q not in pick:
                continue
            p, b, fired = pick[q]
            for i in range(4):
                out[i][q] = res[i][p][:topn]
            out[4][q] = min(int(res[4][p]), topn)
            out[5][q], out[6][q] = b, int(fired)
        return out
    return expected, (int(stats[1]), int(stats[2]), int(sum(nb[q] if q not in pick else pick[q][1] for q in range(nq))))


NAMES = ("song", "diff", "count", "rows", "nres", "batches", "exit")


def _check(ix, qd_h, qo_h, qs, topn, B, want, want_stats, label):
    import torch
    dev = ix.tdev
    out = ix.query_batch_apriori(torch.from_numpy(qd_h).to(dev), torch.from_numpy(qo_h).to(dev), qs, topn, B, want_stats=True)
    got = [t.cpu().numpy() for t in out[:7]]
    for a, b, name in zip(got, want, NAMES):
        assert np.array_equal(a, b), (label, name, topn, B, np.argwhere(a != b)[:5])
    assert out[7][0] == qs[-1] and tuple(out[7][1:]) == want_stats, (label, out[7], want_stats)
    return got


def _random_index(rng, torch_dev, id_stride):
    """12 songs from a universe of 400 hashes, a hash in every song, a twin of song 3 and a song of its own hashes."""
    import torch
    from shazam_b200.database import FingerprintIndex
    universe = rng.integers(0, 256, (400, 10), dtype=np.uint8)
    common = rng.integers(0, 256, 10, dtype=np.uint8)
    songs, digs, offs = [], [], []
    for s in range(1, 13):
        k = rng.integers(0, 400, 150)
        d = np.concatenate([universe[k], common[None]])
        o = np.concatenate([rng.integers(0, 300, 150), [rng.integers(0, 300)]]).astype(np.int32)
        songs.append(np.full(len(d), s * id_stride, np.int32)); digs.append(d); offs.append(o)
    songs.append(np.full(len(digs[2]), 13 * id_stride, np.int32)); digs.append(digs[2]); offs.append(offs[2])   # twin of 3
    solo = rng.integers(0, 256, (80, 10), dtype=np.uint8)
    solo[:, 0] = 0xff                                         # hashes of song 14 alone
    songs.append(np.full(80, 14 * id_stride, np.int32)); digs.append(solo); offs.append(rng.integers(0, 300, 80).astype(np.int32))
    song, dig, off = np.concatenate(songs), np.concatenate(digs), np.concatenate(offs)
    ix = FingerprintIndex(0, len(song) + 1024)
    ix.insert_rows(torch.from_numpy(song).to(torch_dev), torch.from_numpy(dig).to(torch_dev), torch.from_numpy(off).to(torch_dev))
    ix.finalize()
    queries = [(np.zeros((0, 10), np.uint8), np.zeros(0, np.int32))]                          # empty
    nm = rng.integers(0, 256, (30, 10), dtype=np.uint8); nm[:, 0] = 0xfe
    queries.append((nm, rng.integers(0, 50, 30).astype(np.int32)))                             # no match
    queries.append((solo[:60], np.maximum(0, offs[-1][:60] - 4).astype(np.int32)))            # one song only
    queries.append((digs[2][:120], np.maximum(0, offs[2][:120] - 7).astype(np.int32)))        # twins tie
    queries.append((np.concatenate([common[None], digs[5][:40]]), np.array([3] + list(np.maximum(0, offs[5][:40] - 2)), np.int32)))
    for _ in range(30):
        s = int(rng.integers(0, 12))
        n = int(rng.integers(1, 220))
        k = rng.integers(0, len(digs[s]), n)
        d = np.concatenate([digs[s][k], universe[rng.integers(0, 400, n // 3)]])
        o = np.concatenate([np.maximum(0, offs[s][k] - 5), rng.integers(0, 40, n // 3)]).astype(np.int32)
        queries.append((d, o))
    qs = np.concatenate([[0], np.cumsum([len(o) for _, o in queries])]).astype(np.int64)
    qd = np.ascontiguousarray(np.concatenate([d for d, _ in queries]), np.uint8)
    qo = np.ascontiguousarray(np.concatenate([o for _, o in queries]), np.int32)
    return ix, qd, qo, qs


@pytest.mark.parametrize("id_stride", [1, 40_000])            # dense song tables / open addressing
def test_apriori_prefix_exact(torch_dev, id_stride):
    import torch
    rng = np.random.default_rng(7 + id_stride)
    ix, qd, qo, qs = _random_index(rng, torch_dev, id_stride)
    try:
        exits = 0
        for B in (1, 3, 64, 1000, 10 ** 6):
            expected, want_stats = _prefix_reference(ix, qd, qo, qs, B, 5)
            for topn in (1, 2, 3, 5):
                want = expected(topn)
                got = _check(ix, qd, qo, qs, topn, B, want, want_stats, "random")
                exits += int(got[6].sum())
                assert got[5][0] == 0 and got[4][0] == 0            # the empty query
                assert got[6][1] == 0 and got[4][1] == 0            # no match
                assert got[6][2] == 0 and got[4][2] == 1            # one song only: never exits
                assert got[6][3] == 0                               # tied twins: never exits
            # input order: shuffled and duplicated pairs give the same outputs
            perm_d, perm_o = [], []
            starts = [0]
            for q in range(len(qs) - 1):
                idx = np.arange(qs[q], qs[q + 1])
                idx = rng.permutation(np.concatenate([idx, idx[: len(idx) // 3]]))
                perm_d.append(qd[idx]); perm_o.append(qo[idx]); starts.append(starts[-1] + len(idx))
            pd_, po_ = np.ascontiguousarray(np.concatenate(perm_d)), np.ascontiguousarray(np.concatenate(perm_o))
            st = np.array(starts, np.int64)
            for topn in (2, 3):
                want = expected(topn)
                out = ix.query_batch_apriori(torch.from_numpy(pd_).to(torch_dev), torch.from_numpy(po_).to(torch_dev), st, topn, B,
                                             want_stats=True)
                for a, b, name in zip([t.cpu().numpy() for t in out[:7]], want, NAMES):
                    assert np.array_equal(a, b), ("shuffled", name, topn, B)
                assert tuple(out[7][1:]) == want_stats
        assert exits > 0
    finally:
        ix.close()


def test_apriori_several_groups(torch_dev, monkeypatch):
    """A hash with 300 000 postings in every query: > 1M tuples, so a small SIA_VOTE_GROUP_TUPLES splits the call."""
    import torch
    from shazam_b200.database import FingerprintIndex
    rng = np.random.default_rng(11)
    heavy = rng.integers(0, 256, 10, dtype=np.uint8)
    universe = rng.integers(0, 256, (2000, 10), dtype=np.uint8)
    song = np.concatenate([np.repeat(np.arange(1, 3001, dtype=np.int32), 100), np.repeat(np.arange(1, 41, dtype=np.int32), 200)])
    dig = np.concatenate([np.repeat(heavy[None], 300_000, 0), universe[rng.integers(0, 2000, 8000)]])
    off = np.concatenate([np.tile(np.arange(100, dtype=np.int32) * 7, 3000), rng.integers(0, 400, 8000).astype(np.int32)])
    ix = FingerprintIndex(0, len(song) + 1024)
    try:
        ix.insert_rows(torch.from_numpy(song).to(torch_dev), torch.from_numpy(dig).to(torch_dev), torch.from_numpy(off).to(torch_dev))
        ix.finalize()
        queries = []
        for q in range(12):
            s = int(rng.integers(0, 40))
            rows = np.flatnonzero(song[300_000:] == s + 1)[:150] + 300_000
            d = np.concatenate([dig[rows], heavy[None]])
            o = np.concatenate([np.maximum(0, off[rows] - 3), [q]]).astype(np.int32)
            queries.append((d, o))
        qs = np.concatenate([[0], np.cumsum([len(o) for _, o in queries])]).astype(np.int64)
        qd = np.ascontiguousarray(np.concatenate([d for d, _ in queries]))
        qo = np.ascontiguousarray(np.concatenate([o for _, o in queries]))
        for B in (16, 64):
            expected, want_stats = _prefix_reference(ix, qd, qo, qs, B, 3)
            for budget in (None, "1"):
                if budget is None:
                    monkeypatch.delenv("SIA_VOTE_GROUP_TUPLES", raising=False)
                else:
                    monkeypatch.setenv("SIA_VOTE_GROUP_TUPLES", budget)
                for topn in (1, 3):
                    _check(ix, qd, qo, qs, topn, B, expected(topn), want_stats, f"groups {budget}")
        monkeypatch.delenv("SIA_VOTE_GROUP_TUPLES", raising=False)
    finally:
        ix.close()


def test_apriori_matches_host_return_matches(gpudb):
    """Where the exit fires, return_matches(sorted(set(q)), B, apriori=True) gives the same songs_arr."""
    from shazam_b200 import recognize
    rng = np.random.default_rng(3)
    fired = 0
    for case in range(6):
        db = gpudb()
        nsongs, universe = 6, 300 + 200 * case
        hx = lambda i: hashlib.sha1(str(i).encode()).hexdigest()[:20]
        rows = {}
        for s in range(nsongs):
            sid = db.insert_song(f"s{s}", hashlib.sha1(f"f{s}".encode()).hexdigest().upper(), 200)
            rows[sid] = [(hx(int(rng.integers(0, universe))), int(rng.integers(0, 80))) for _ in range(200)]
            db.insert_hashes(sid, rows[sid])
            db.set_song_fingerprinted(sid)
        target = rows[1 + case % nsongs]
        q = [(h, max(0, o - 4)) for h, o in target[:120]] + [(hx(int(rng.integers(0, universe))), int(rng.integers(0, 30)))
                                                             for _ in range(40)]
        q = sorted(set(q))
        for B in (5, 17, 60):
            _, _, songs_arr = recognize.return_matches(q, B, apriori=True)
            got = recognize.recognize_batch([recognize.hashes_to_arrays(q)], topn=2, apriori_batch=B)[0]
            if songs_arr:
                fired += 1
                assert _strip(got) == _strip(songs_arr), (case, B)
    assert fired > 0
