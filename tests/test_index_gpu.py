"""Parity of the GPU index / lookup / vote (through the C ABI) with the reference's
return_matches + align_matches semantics (oracle + golden vectors)."""
import hashlib

import os

import numpy as np
import pytest

from oracle import sia_oracle as O

pytestmark = pytest.mark.gpu


def _hx(i):
    return hashlib.sha1(str(i).encode()).hexdigest()[:20]


def _strip(results):
    return [{k: (v.decode() if isinstance(v, bytes) else v) for k, v in r.items()} for r in results]


@pytest.fixture()
def gpudb(native_lib):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
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


def test_golden_match_cases(gpudb, match_cases):
    from shazam_b200 import recognize
    for case in match_cases:
        db = gpudb()
        if case["case"] == "kat":
            for s in range(9):
                db.insert_song(f"s{s + 1}", "AB" * 20, 100)
            got = recognize.align_matches([(7, 3), (7, 3), (7, 5), (2, 10), (2, 10), (2, -4), (2, -4), (9, 1)],
                                          {7: 3, 2: 4, 9: 1}, 10, 3)
            assert _strip(got) == case["results"]
            continue
        for sid, s in sorted(case["songs"].items(), key=lambda kv: int(kv[0])):
            assert db.insert_song(s["song_name"], s["file_sha1"], s["total_hashes"]) == int(sid)
        by_song = {}
        for sid, h, o in case["rows"]:
            by_song.setdefault(sid, []).append((h, o))
        for sid, hs in by_song.items():
            db.insert_hashes(sid, hs)                      # contains duplicates -> INSERT IGNORE
            db.set_song_fingerprinted(sid)
        assert db.get_num_fingerprints() == len({(r[0], r[1], r[2]) for r in case["rows"]})
        q = [tuple(x) for x in case["query"]]
        matches, dedup, qt = recognize.find_matches(q)
        assert len(matches) == case["n_matches"]
        assert hashlib.sha256(repr(sorted(matches)).encode()).hexdigest() == case["matches_sorted_sha"]
        assert {str(k): v for k, v in dedup.items()} == case["dedup"]
        for topn, want in case["results_by_topn"].items():
            got = recognize.align_matches(matches, dedup, len(q), int(topn)) if q else []
            assert _strip(got) == want, (case["case"], topn)
            if q:   # the fused device path gives the same dicts
                fused = recognize.recognize_batch([recognize.hashes_to_arrays(q)], int(topn))[0]
                assert _strip(fused) == want, ("fused", case["case"], topn)


def test_apriori_early_exit_golden(gpudb):
    """SURVEY §8f-4: ``return_matches(..., apriori=True)`` against the outputs of recognizer_apriori.py's own
    return_matches (:246-310, executed from the reference's source by tests/golden/make_golden.py): the tuples read up
    to the exit, dedup_hashes at that point and the aligned results that triggered it — lookup and vote on the GPU."""
    import json
    from shazam_b200 import recognize
    cases = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "apriori_cases.json")))
    exits = 0
    for case in cases:
        db = gpudb()
        for sid, s in sorted(case["songs"].items(), key=lambda kv: int(kv[0])):
            assert db.insert_song(s["song_name"], s["file_sha1"], s["total_hashes"]) == int(sid)
        by_song = {}
        for sid, h, o in case["rows"]:
            by_song.setdefault(sid, []).append((h, o))
        for sid, hs in by_song.items():
            db.insert_hashes(sid, hs)
            db.set_song_fingerprinted(sid)
        q = [tuple(x) for x in case["query"]]
        matches, dedup, songs_arr = recognize.return_matches(q, case["batch_size"], apriori=True)
        assert len(matches) == case["n_matches"], case["case"]
        assert hashlib.sha256(repr(sorted(matches)).encode()).hexdigest() == case["matches_sorted_sha"]
        assert {str(k): v for k, v in dedup.items()} == case["dedup"]
        assert _strip(songs_arr) == case["songs_arr"], case["case"]
        exits += bool(songs_arr)
    assert exits >= 2


def _random_table(rng, nsongs, per_song, universe, max_off=500):
    table = O.FingerprintTable()
    rows = []
    for s in range(nsongs):
        sid = table.insert_song(f"song{s}", hashlib.sha1(f"f{s}".encode()).hexdigest().upper(), per_song)
        hs = [(_hx(int(rng.integers(0, universe))), int(rng.integers(0, max_off))) for _ in range(per_song)]
        table.insert_hashes(sid, hs)
        table.set_song_fingerprinted(sid)
        rows.append((sid, hs))
    return table, rows


def _load(db, rows, table):
    for sid, hs in rows:
        s = table.songs[sid]
        assert db.insert_song(s["song_name"], s["file_sha1"], s["total_hashes"]) == sid
        db.insert_hashes(sid, hs)
        db.set_song_fingerprinted(sid)


def test_batch_queries_vs_oracle(gpudb):
    """Many queries at once: empty query, no-match query, duplicate pairs, one hash at several offsets,
    heavy keys (one hash in every song)."""
    from shazam_b200 import recognize
    rng = np.random.default_rng(5)
    table, rows = _random_table(rng, 40, 400, 3000)
    heavy = _hx("heavy")
    for sid, hs in rows:                                   # a key present in every song, several times
        extra = [(heavy, int(o)) for o in rng.integers(0, 500, 5)]
        table.insert_hashes(sid, extra)
        hs.extend(extra)
    db = gpudb()
    _load(db, rows, table)
    assert db.get_num_fingerprints() == table.num_rows()
    queries = []
    for qi in range(25):
        sid, hs = rows[int(rng.integers(0, len(rows)))]
        shift = int(rng.integers(0, 50))
        q = [(h, o - shift) for h, o in hs[:150] if o - shift >= 0]
        q += [(_hx(int(rng.integers(0, 6000))), int(rng.integers(0, 100))) for _ in range(60)]
        if qi % 3 == 0:
            q += [(heavy, 3), (heavy, 9)]                   # same hash at two query offsets
        queries.append(q)
    queries[4] = []                                        # empty query
    queries[7] = [(_hx("absent%d" % i), i) for i in range(30)]   # nothing matches
    queries[9] = queries[9] + queries[9][:20]              # duplicate (hash, offset) pairs
    for topn in (1, 3, 10):
        got = recognize.recognize_batch([recognize.hashes_to_arrays(q) for q in queries], topn)
        for q, g in zip(queries, got):
            qs = set(q)
            matches, dedup = O.return_matches(table, qs)
            want = O.align_matches(table, matches, dedup, len(qs), topn) if qs else []
            assert _strip(g) == _strip(want)
    # the tuple-typed compat path on one query
    matches, dedup, _ = recognize.find_matches(set(queries[0]))
    om, od = O.return_matches(table, set(queries[0]))
    assert sorted(matches) == sorted(om) and dedup == od


def test_sort_dedup_and_select_large(gpudb):
    """1.5M rows with duplicates and a 20k-row heavy key: the sorted, de-duplicated index equals numpy's."""
    import torch
    rng = np.random.default_rng(9)
    n = 1_500_000
    dig = rng.integers(0, 256, (n, 10), dtype=np.uint8)
    dig[:20000] = dig[0]                                   # heavy key
    dig[20000:40000, :9] = dig[20000, :9]                  # differ only in the last digest byte
    song = rng.integers(1, 5000, n).astype(np.int32)
    off = rng.integers(0, 1 << 20, n).astype(np.int32)
    dup = rng.integers(0, n, 100_000)
    dig = np.concatenate([dig, dig[dup]]); song = np.concatenate([song, song[dup]]); off = np.concatenate([off, off[dup]])
    db = gpudb(capacity_rows=2_000_000)
    ix = db.index
    dev = ix.tdev
    ix.insert_rows(torch.from_numpy(song).to(dev), torch.from_numpy(dig).to(dev), torch.from_numpy(off).to(dev))
    stored = ix.finalize()
    rec = np.zeros(len(off), dtype=[("h", "S10"), ("s", "<i4"), ("o", "<i4")])
    rec["h"] = [bytes(r) for r in dig] if False else np.frombuffer(dig.tobytes(), dtype="S10")
    rec["s"] = song; rec["o"] = off
    uniq = np.unique(rec)
    assert stored == len(uniq)
    # select: the heavy key, the near-identical keys, random present keys, absent keys
    probe = np.concatenate([dig[:1], dig[20000:20003], dig[rng.integers(40000, n, 200)],
                            rng.integers(0, 256, (50, 10), dtype=np.uint8)])
    probe = np.unique(np.frombuffer(probe.tobytes(), dtype="S10"))
    pd = np.frombuffer(probe.tobytes(), np.uint8).reshape(-1, 10)
    idx, sid, o = ix.select(pd)
    got = sorted(zip([probe[i] for i in idx.tolist()], sid.tolist(), o.tolist()))
    want = sorted((r["h"], int(r["s"]), int(r["o"])) for r in uniq[np.isin(uniq["h"], probe)])
    assert got == want and len(got) > 20000
    # a second insert + finalize merges into the sorted index; re-inserting existing rows is ignored
    ix.insert_rows(torch.from_numpy(song[:1000]).to(dev), torch.from_numpy(dig[:1000]).to(dev), torch.from_numpy(off[:1000]).to(dev))
    assert ix.finalize() == len(uniq)


def test_delete_unfingerprinted_cascade(gpudb):
    db = gpudb()
    a = db.insert_song("a", "AA" * 20, 2)
    db.insert_hashes(a, [(_hx(1), 1), (_hx(2), 2)])
    db.set_song_fingerprinted(a)
    b = db.insert_song("b", "BB" * 20, 2)                 # crashed before set_song_fingerprinted
    db.insert_hashes(b, [(_hx(1), 5), (_hx(3), 6)])
    assert db.get_num_fingerprints() == 4
    with db.cursor() as cur:                               # the ingest driver's start-up sweep, __init__.py:421-424
        cur.execute(db.CREATE_SONGS_TABLE)
        cur.execute(db.CREATE_FINGERPRINTS_TABLE)
        cur.execute(db.DELETE_UNFINGERPRINTED)
    assert db.get_num_fingerprints() == 2
    assert [r[:4] for r in db.get_songs()] == [(a, "a", "AA" * 20, 2)]
    assert db.select_multiple([_hx(1).upper()]) == [(_hx(1).upper(), a, 1)]
    assert [d["_source"] for d in db.find_matches([_hx(2)])] == [{"hash": _hx(2), "song_id": a, "offset": 2}]
    c = db.insert_song("c", "CC" * 20, 1)
    assert c == 3                                          # AUTO_INCREMENT does not reuse ids
    with pytest.raises(Exception):
        db.insert_hashes(c, [(_hx(4), 1 << 24)])
    with pytest.raises(Exception):
        with db.cursor() as cur:
            cur.execute("DROP TABLE songs")


def test_hash_prefix_slots_equal_single_index(gpudb):
    """Hash-prefix sharding on one GPU: the device steps of a distributed query pass (route entries -> per-shard lookup +
    expansion into key slots -> vote over the keys of all shards, csrc/index_dist.cu) give the results of one index and of
    the oracle; slot overflow is reported, never silent."""
    import torch
    from shazam_b200.database import FingerprintIndex, route_entries, vote_finish, vote_key_slots, vote_tuples
    from shazam_b200.fingerprinter import hex_to_digests
    rng = np.random.default_rng(21)
    table, rows = _random_table(rng, 30, 300, 800)
    db = gpudb()
    _load(db, rows, table)
    G, QP = 3, 8                                        # shards; queries per "rank" and pass
    shards = [FingerprintIndex(0, 1 << 18) for _ in range(G)]
    try:
        for sid, hs in rows:
            d = hex_to_digests([h for h, _ in hs]); o = np.array([t for _, t in hs], np.int32)
            own = (((d[:, 0].astype(np.int64) << 8) | d[:, 1]) * G) >> 16
            for g in range(G):
                shards[g].insert(sid, d[own == g], o[own == g])
        queries = []
        for qi in range(2 * QP - 3):                    # two "ranks" own the queries: 8 + 5
            sid, hs = rows[int(rng.integers(0, len(rows)))]
            q = list({(h, max(0, o - 11)) for h, o in hs[:120]} | {(_hx(int(rng.integers(0, 1600))), 3) for _ in range(40)})
            queries.append(q + q[:7])                   # duplicate (hash, offset) pairs are ignored
        queries[2] = []
        dev = db.index.tdev
        D = torch.from_numpy(np.concatenate([hex_to_digests([h for h, _ in q]) for q in queries if q])).to(dev)
        Oq = torch.from_numpy(np.concatenate([np.array([t for _, t in q], np.int32) for q in queries if q])).to(dev)
        starts = np.cumsum([0] + [len(q) for q in queries])
        ref = db.index.query_batch(D, Oq, starts, 3)
        max_song = db.index.max_song
        owners = [(0, QP), (QP, len(queries))]          # query ranges of the two query-owning ranks
        ecap, kcap = 800, 12000
        for attempt in range(2):
            sent = []
            for r, (a, b) in enumerate(owners):
                st = torch.zeros(1, dtype=torch.int32, device=dev)
                qs = torch.as_tensor(starts[a:b + 1] - starts[a], dtype=torch.int64, device=dev)
                sent.append(route_entries(0, D[starts[a]:starts[b]], Oq[starts[a]:starts[b]], qs, r * QP, G, ecap, st))
                assert int(st.item()) == 0
            # "all-to-all #1": shard g receives slot g of every owner (an owner that is not a rank sends empty slots)
            infos, keys = [], []
            for g in range(G):
                recv = torch.zeros((G, ecap, 2), dtype=torch.int64, device=dev)
                for r in range(len(owners)):
                    recv[r] = sent[r][g]
                info = torch.zeros(4, dtype=torch.int64, device=dev)
                keys.append(shards[g].expand_slots(recv, G, QP, kcap, info))
                infos.append(info.cpu().numpy())
            flags = max(int(i[0]) for i in infos)
            if attempt == 0:
                assert flags == 0
            # "all-to-all #2": owner r receives slot r of every shard
            for r, (a, b) in enumerate(owners):
                recv = torch.stack([keys[g][r] for g in range(G)])
                got = vote_key_slots(0, recv, b - a, 3, max_song, defer=attempt == 1)
                if attempt == 1:
                    vote_finish(0)                          # the deferred form: enqueue, then complete
                for x, y in zip(ref, got):
                    assert torch.equal(x[a:b], y), (attempt, r)
            if attempt == 0:
                # the same pass with the second exchange fused into the scatter kernel (csrc/index_pvote.cu): every shard
                # looks its entries up, the per-query tuple counts are summed (the all-reduce), every shard scatters its
                # tuples straight into the owners' regions (here: G buffers on one GPU stand in for the peers' memory),
                # every owner counts its regions
                from shazam_b200.database import PeerBuffers, vote_count_regions
                for cap in (None, "64"):                # "64": tiny regions -> every query is flagged for the key exchange
                    if cap:
                        os.environ["SIA_PVOTE_CAP"] = cap
                    bufs = [PeerBuffers(0, r, G, QP, 1 << 16, 4096) for r in range(G)]
                    try:
                        for pb in bufs:
                            pb.connect([x.local for x in bufs])
                            pb.counters.zero_()
                        recvs, infos2, t_total = [], [], torch.zeros(G * QP, dtype=torch.int64, device=dev)
                        for g in range(G):
                            recv = torch.zeros((G, ecap, 2), dtype=torch.int64, device=dev)
                            for r in range(len(owners)):
                                recv[r] = sent[r][g]
                            recvs.append(recv)
                        for g in range(G):              # every shard keeps the lookup of its pass inside its handle
                            info = torch.zeros(4, dtype=torch.int64, device=dev)
                            t_total += shards[g].lookup_slots(recvs[g], G, QP, info)
                            infos2.append(info)
                        for g in range(G):
                            shards[g].scatter_peers(G, QP, t_total, bufs[g], infos2[g])
                        assert all(int(i[0].item()) == 0 for i in infos2)
                        for r, (a, b) in enumerate(owners):
                            info = torch.zeros(4, dtype=torch.int64, device=dev)
                            got = vote_count_regions(0, t_total[r * QP:(r + 1) * QP], QP, 3, bufs[r], info)
                            flagged = int(info[1].item()) & 0xffffffff
                            if cap:
                                assert flagged > 0      # nothing wrong is reported for a flagged query: it stays empty
                            else:
                                assert flagged == 0
                                for x, y in zip(ref, got):
                                    assert torch.equal(x[a:b], y[:b - a]), ("peer regions", r)
                        # regions that do not fit the owner's buffer: flag 4 and the size needed, nothing scattered
                        info = torch.zeros(4, dtype=torch.int64, device=dev)
                        tiny = PeerBuffers(0, 0, G, QP, 64, 4096)
                        tiny.connect([tiny.local] * G)
                        shards[0].lookup_slots(recvs[0], G, QP, info)
                        shards[0].scatter_peers(G, QP, t_total, tiny, info)
                        assert int(info[0].item()) & 4 and int(info[3].item()) > 64
                        tiny.close()
                    finally:
                        os.environ.pop("SIA_PVOTE_CAP", None)
                        for pb in bufs:
                            pb.close()
                # the same keys, unslotted, through the plain key vote
                allk = torch.cat([keys[g][0][1:1 + int(keys[g][0][0])] for g in range(G)])
                got = vote_tuples(0, allk[torch.randperm(allk.numel(), device=dev)], QP, 3, max_song)
                for x, y in zip(ref, got):
                    assert torch.equal(x[0:QP], y)
                # too-small slots: flagged, with the sizes they needed
                st = torch.zeros(1, dtype=torch.int32, device=dev)
                qs = torch.as_tensor(starts[0:QP + 1], dtype=torch.int64, device=dev)
                small = route_entries(0, D[:starts[QP]], Oq[:starts[QP]], qs, 0, G, 16, st)
                info = torch.zeros(4, dtype=torch.int64, device=dev)
                recv = torch.zeros((G, 16, 2), dtype=torch.int64, device=dev)
                recv[0] = small[0]
                shards[0].expand_slots(recv, G, QP, 64, info)
                flags, need_k, need_e = (int(v) for v in info[:3].cpu())
                assert flags == 3 and need_e > 16 and need_k > 64
        # and the single index equals the oracle
        song, dif, cnt, rws, nres = [t.cpu().numpy() for t in ref]
        for i, q in enumerate(queries):
            m, dd = O.return_matches(table, set(q))
            best = O.best_offsets(m, 3)
            assert [(int(song[i, r]), int(dif[i, r]), int(cnt[i, r])) for r in range(nres[i])] == [tuple(b) for b in best]
            assert [int(rws[i, r]) for r in range(nres[i])] == [dd[b[0]] for b in best]
    finally:
        for s_ in shards:
            s_.close()


def test_incremental_finalize_and_cursor_statement(gpudb):
    """The reference commits per song (__init__.py:381-386): rows inserted and finalized in many small batches, in any
    order, with re-inserted duplicates, give the same table as one bulk load; and the cursor answers exactly the
    statement return_matches builds (recognizer.py:252-259): rows (HEXUPPER str, song_id int, offset int), here in
    IN-list order then (song_id, offset)."""
    import torch
    rng = np.random.default_rng(3)
    table, rows = _random_table(rng, 25, 500, 900, max_off=4000)
    db = gpudb(capacity_rows=1 << 16)
    order = rng.permutation(len(rows))
    for k, idx in enumerate(order):
        sid, hs = rows[idx]
        s = table.songs[sid]
        db.songs[sid] = {"song_name": s["song_name"], "file_sha1": s["file_sha1"], "total_hashes": s["total_hashes"],
                         "fingerprinted": 1, "date_created": None}
        half = len(hs) // 2
        db.insert_hashes(sid, hs[:half])
        if k % 3 == 0:
            assert db.get_num_fingerprints() > 0        # finalize between the two halves of a song
        db.insert_hashes(sid, hs[half:] + hs[:10])      # some rows twice: INSERT IGNORE
        if k % 2 == 0:
            db.index.finalize()
    assert db.get_num_fingerprints() == table.num_rows()
    assert db.index.keys == len(table.rows)
    d, s, o = db.index.export()
    got = list(zip((bytes(x).hex().upper() for x in d.cpu().numpy()), s.cpu().tolist(), o.cpu().tolist()))
    want = sorted((h, sid, off) for h, v in table.rows.items() for sid, off in v)
    assert got == want                                  # (hash, song_id, offset) order, nothing lost or doubled
    # the literal statement of recognizer.py:252-259
    values = [h for h in list(table.rows)[:40]] + ["AB" * 10]
    with db.cursor() as cur:
        n = cur.execute(db.SELECT_MULTIPLE % ", ".join([db.IN_MATCH] * len(values)), values)
        got_rows = [(hsh, sid, offset) for hsh, sid, offset in cur]
    assert n == len(got_rows)
    assert all(isinstance(h, str) and h == h.upper() and isinstance(a, int) and isinstance(b, int) for h, a, b in got_rows)
    assert got_rows == [(h, sid, off) for h in values for sid, off in sorted(table.rows.get(h, ()))]
    # delete a third of the songs (ON DELETE CASCADE), then insert again: still equal to the model
    dead = [rows[i][0] for i in order[::3]]
    assert db.index.delete_songs(dead) == sum(1 for h, v in table.rows.items() for sid, _ in v if sid not in dead)
    d, s, o = db.index.export()
    got = list(zip((bytes(x).hex().upper() for x in d.cpu().numpy()), s.cpu().tolist(), o.cpu().tolist()))
    assert got == [w for w in want if w[1] not in dead]
    assert db.index.keys == len({w[0] for w in want if w[1] not in dead})
    for i in order[::3]:
        db.insert_hashes(rows[i][0], rows[i][1])
    d, s, o = db.index.export()
    assert list(zip((bytes(x).hex().upper() for x in d.cpu().numpy()), s.cpu().tolist(), o.cpu().tolist())) == want


def test_recognition_end_to_end_noisy_clips(gpudb, fpr):
    """Config-3 in miniature: index synthetic tracks fingerprinted ON THE GPU, recognise 5 s clips
    mixed with coloured noise at SNR 10 and 0 dB; GPU results must equal the oracle path run on
    the same audio (same song ids, offsets, counts), and the hash sets must agree (Jaccard >= 0.99)."""
    from shazam_b200 import recognize
    rng = np.random.default_rng(77)
    fs = 44100
    tracks = [O.synth_track(300 + i, 20 * fs) for i in range(8)]
    db = gpudb()
    table = O.FingerprintTable()
    batch = fpr.fingerprint_tracks(tracks, fan_value=15)
    jac = []
    for i, t in enumerate(tracks):
        h, t1 = batch.track(i)
        oh, ot = O.fingerprint_arrays(t, fs, 15)
        sa = set(zip(map(bytes, h), t1.tolist())); sb = set(zip(map(bytes, oh), ot.tolist()))
        jac.append(len(sa & sb) / max(1, len(sa | sb)))
        sid = db.insert_song(f"t{i}", "AB" * 20, len(sa))
        db.insert_hashes_array(sid, h, t1)
        db.set_song_fingerprinted(sid)
        osid = table.insert_song(f"t{i}", "AB" * 20, len(sb))
        table.insert_hashes(osid, [(bytes(a).hex(), int(b)) for a, b in zip(oh, ot)])
    assert min(jac) >= 0.99, jac
    clips, truth = [], []
    for snr in (10.0, 0.0):
        for i in range(8):
            start = int(rng.integers(0, 14)) * fs
            sig = tracks[i][start:start + 5 * fs].astype(np.float64)
            noise = np.convolve(rng.normal(0, 1, len(sig) + 63), np.hanning(64), "valid")    # band-limited noise
            mixed = O.mix_noise(sig, noise, snr)                                            # recognizer_test.py:426-435
            clips.append(np.clip(np.rint(mixed), -32768, 32767).astype(np.int16))
            truth.append(i + 1)
    qb = fpr.fingerprint_tracks(clips, fan_value=15)
    got = recognize.recognize_batch([qb.track(i) for i in range(len(clips))], topn=3)
    correct = 0
    for i, clip in enumerate(clips):
        oh, ot = O.fingerprint_arrays(clip, fs, 15)
        q = set(zip([bytes(a).hex() for a in oh], ot.tolist()))
        m, dd = O.return_matches(table, q)
        want = O.align_matches(table, m, dd, len(q), 3)
        assert _strip(got[i]) == _strip(want), i
        correct += bool(got[i]) and got[i][0]["song_id"] == truth[i]
    assert correct >= 14, correct          # 16 clips; the 0 dB ones may miss, identically in both paths


def test_ingest_directory_flow(tmp_path, fpr):
    """The ingest main flow (__init__.py:417-432) against the 'gpu' backend: registry, start-up sweep,
    stereo set-union, resume by file SHA-1; then a clip is recognised through the compat functions."""
    import wave
    from shazam_b200 import compat, ingest, recognize
    from shazam_b200.database import get_database
    compat.set_fingerprinter(fpr)
    fs = 44100
    mono = O.synth_track(900, 6 * fs)
    left, right = O.synth_track(901, 5 * fs), O.synth_track(902, 5 * fs)
    same = O.synth_track(903, 4 * fs)
    files = {"mono.wav": [mono], "stereo.wav": [left, right], "dual.wav": [same, same]}
    for name, chans in files.items():
        with wave.open(str(tmp_path / name), "wb") as w:
            w.setnchannels(len(chans)); w.setsampwidth(2); w.setframerate(fs)
            w.writeframes(np.stack(chans, 1).astype("<i2").tobytes())
    (tmp_path / "broken.wav").write_bytes(b"not a wav")
    with pytest.raises(TypeError):
        get_database("oracle")
    db = get_database("gpu")(host="127.0.0.1", user="root", password="x", database="music_recognition",
                             capacity_rows=1 << 20)
    try:
        ingest.set_database(db); recognize.set_database(db)
        with db.cursor() as cur:
            cur.execute(db.CREATE_SONGS_TABLE); cur.execute(db.CREATE_FINGERPRINTS_TABLE); cur.execute(db.DELETE_UNFINGERPRINTED)
        known = ingest.load_fingerprinted_audio_hashes(set())
        assert ingest.fingerprint_directory(str(tmp_path), [".wav"], 4, known) == 3
        songs = {r[1]: r for r in db.get_songs()}
        assert set(songs) == {"mono", "stereo", "dual"}
        for name, chans in files.items():
            want = set()
            for c in chans:
                want |= set(O.fingerprint(c, Fs=fs))
            row = songs[name[:-4]]
            assert row[3] == len(want)                                   # total_hashes = len(set), __init__.py:381
            assert row[2] == ingest.unique_hash(str(tmp_path / name))
            fset, fh = ingest.get_file_fingerprints(str(tmp_path / name))
            assert fset == want and fh == row[2]
            # the same with the channel split and the set union on the device (SURVEY 8f-1)
            d, o, fh2 = ingest.get_file_fingerprints_device(str(tmp_path / name))
            got = set(zip((bytes(r).hex() for r in d.cpu().numpy()), o.cpu().tolist()))
            assert got == want and fh2 == row[2] and d.shape[0] == len(want)
        assert db.get_num_fingerprints() == sum(r[3] for r in songs.values())
        assert ingest.fingerprint_directory(str(tmp_path), ["wav"], None, ingest.load_fingerprinted_audio_hashes(set())) == 0
        # recognise 3 s of the stereo file's left channel (recognizer.py:379-397 flow)
        clip = left[fs:4 * fs]
        hashes = set(compat.generate_fingerprints(clip, Fs=fs)[0])
        matches, dedup, _ = recognize.find_matches(hashes)
        res = recognize.align_matches(matches, dedup, len(hashes))
        assert res[0]["song_name"] == b"stereo" and res[0]["offset"] == round(fs / 2048)
        assert res[0]["offset_seconds"] == round(float(res[0]["offset"]) / 44100 * 4096 * 0.5, 5)
    finally:
        compat.set_fingerprinter(None)
        db.index.close()


def test_dump_load_and_sql_rows(tmp_path, gpudb):
    """Index persistence in the schema's vocabulary (SURVEY §8f-2): dump -> load gives the same table and answers."""
    import torch
    from shazam_b200 import recognize
    from shazam_b200.database import GPUDatabase
    rng = np.random.default_rng(31)
    table, rows = _random_table(rng, 12, 200, 500)
    db = gpudb()
    _load(db, rows, table)
    n = db.dump(str(tmp_path / "dump"))
    assert n == table.num_rows()
    sql = sorted(db.iter_sql_rows(chunk_rows=700))                       # (song_id, HEXUPPER, offset) for INSERT_FINGERPRINT
    assert sql == sorted((sid, h.upper(), o) for h, v in ((k, v) for k, v in table.rows.items()) for sid, o in v)
    d, s, o = db.index.export()
    key = [bytes(x) for x in d.cpu().numpy()]
    assert key == sorted(key) and len(key) == n                          # (hash, song, offset) order
    db2 = GPUDatabase.load(str(tmp_path / "dump"), device=0)
    try:
        assert db2.get_num_fingerprints() == n and db2.get_songs() == db.get_songs()
        assert db2.insert_song("new", "CD" * 20, 0) == len(rows) + 1     # AUTO_INCREMENT state survives
        q = [(h, max(0, off - 5)) for h, off in rows[3][1][:80]]
        recognize.set_database(db)
        want = recognize.recognize_batch([recognize.hashes_to_arrays(q)], 3)
        recognize.set_database(db2)
        got = recognize.recognize_batch([recognize.hashes_to_arrays(q)], 3)
        assert _strip(got[0]) == _strip(want[0]) and got[0][0]["song_id"] == rows[3][0]
    finally:
        db2.index.close()


def test_union_channels_device(fpr):
    """Stereo set-union on the device (SURVEY §8f-1) equals the host union / Python set."""
    import torch
    from shazam_b200 import ingest
    a = O.synth_track(70, 4 * 44100)
    b = a.copy(); b[44100:] = O.synth_track(71, 3 * 44100)               # second channel shares its first second
    batch = fpr.fingerprint_tracks([a, b], fan_value=15)
    hd, td = ingest.union_channels_device(torch.from_numpy(batch.hash).to(fpr.tdev), torch.from_numpy(batch.t1).to(fpr.tdev))
    hh, th = ingest.union_channels(batch, 0, 2)
    dev_set = set(zip(map(bytes, hd.cpu().numpy()), td.cpu().tolist()))
    host_set = set(zip(map(bytes, hh), th.tolist()))
    want = set(O.fingerprint(a, fan_value=15)) | set(O.fingerprint(b, fan_value=15))
    assert dev_set == host_set == {(bytes.fromhex(h), int(t)) for h, t in want}
    assert len(dev_set) == hd.shape[0] < len(batch.t1)                   # duplicates existed and were dropped


def _np_vote(qid, song, diff, head, nq, topn):
    """Vectorised restatement of best_offsets (recognizer.py:303-310) over (query, song, diff) tuples: per
    (query, song) the largest bin, smallest diff on ties; per query (count desc, song asc); rows = head tuples."""
    key = (qid.astype(np.int64) << 49) | (song.astype(np.int64) << 25) | (diff.astype(np.int64) + (1 << 24))
    bins, cnt = np.unique(key, return_counts=True)
    bq, bs, bd = bins >> 49, (bins >> 25) & 0xffffff, (bins & 0x1ffffff) - (1 << 24)
    order = np.lexsort((bd, -cnt, bs, bq))                       # per (q, song): count desc, diff asc
    first = np.ones(len(order), bool)
    first[1:] = (bq[order][1:] != bq[order][:-1]) | (bs[order][1:] != bs[order][:-1])
    sel = order[first]
    sq, ss, sd, sc = bq[sel], bs[sel], bd[sel], cnt[sel]
    rk, rc = np.unique((qid[head].astype(np.int64) << 24) | song[head], return_counts=True)
    out = [np.zeros((nq, topn), np.int32) for _ in range(4)]
    nres = np.zeros(nq, np.int32)
    o2 = np.lexsort((ss, -sc, sq))
    sq, ss, sd, sc = sq[o2], ss[o2], sd[o2], sc[o2]
    starts = np.searchsorted(sq, np.arange(nq + 1))
    for q in range(nq):
        a, b = starts[q], min(starts[q + 1], starts[q] + topn)
        nres[q] = b - a
        out[0][q, :b - a], out[1][q, :b - a], out[2][q, :b - a] = ss[a:b], sd[a:b], sc[a:b]
        pos = np.searchsorted(rk, (q << 24) | ss[a:b])
        out[3][q, :b - a] = rc[pos]
    return out + [nres]


@pytest.mark.parametrize("id_stride,off_range", [(1, 64), (50000, 64), (1, 1 << 16)])
def test_vote_large_table_vs_oracle(gpudb, monkeypatch, id_stride, off_range):
    """The production vote on a 1.2 M-row table (~200 postings per key) against a vectorised restatement of
    recognizer.py:303-310 for EVERY query and against the oracle's own Python functions (return_matches + best_offsets
    over an array-backed table) for a subsample — counts, smallest-diff and ascending-song tie-breaks, dedup rows,
    stats — for any grouping of the queries.  id_stride 1: dense song tables; 50000: song ids up to 1.5e7 ->
    open-addressing song tables.  off_range 64: tie-heavy bins (most tuples are candidates); 65536: mostly distinct
    bins (the singles pass decides).  One query has 40 000 entries and a bin of 33 000 matches."""
    import torch
    from shazam_b200.database import vote_tuples
    rng = np.random.default_rng(77)
    nsongs, per_song, universe = 300, 4000, 6000       # ~200 postings per key; offsets in a small range -> many ties
    n = nsongs * per_song
    keys = rng.integers(0, universe, n)
    pool = np.frombuffer(b"".join(hashlib.sha1(str(i).encode()).digest()[:10] for i in range(universe)),
                         np.uint8).reshape(universe, 10)
    dig = pool[keys]
    song = np.repeat(np.arange(1, nsongs + 1, dtype=np.int32) * id_stride, per_song)
    off = rng.integers(0, off_range, n).astype(np.int32)
    # one more song whose 33000 rows all align with query 70 at the same difference
    n_big = 33000
    big = np.frombuffer(b"".join(hashlib.sha1(b"big%d" % i).digest()[:10] for i in range(n_big)), np.uint8).reshape(n_big, 10)
    dig = np.concatenate([dig, big]); song = np.concatenate([song, np.full(n_big, (nsongs + 1) * id_stride, np.int32)])
    off = np.concatenate([off, (np.arange(n_big) % 3000 + 16).astype(np.int32)])
    n += n_big
    db = gpudb(capacity_rows=n + 16)
    ix = db.index
    dev = ix.tdev
    half = n // 2                                       # two finalizes: the second merges into the first
    for a, b in ((0, half), (half, n)):
        ix.insert_rows(torch.from_numpy(song[a:b]).to(dev), torch.from_numpy(dig[a:b]).to(dev), torch.from_numpy(off[a:b]).to(dev))
        ix.finalize()
    otable = O.ArrayFingerprintTable(dig, song, off)
    assert ix.rows == otable.num_rows()
    sizes = rng.integers(0, 400, 120)
    sizes[3] = 0; sizes[50] = 3000; sizes[70] = 40000   # an empty query, a big one, one beyond 32767 entries
    qs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    qk = rng.integers(0, universe + 500, qs[-1])        # some absent keys
    pool2 = np.concatenate([pool, rng.integers(0, 256, (500, 10), dtype=np.uint8)])
    qd_h = pool2[qk]
    qo_h = rng.integers(0, 16, qs[-1]).astype(np.int32)
    qd_h[qs[70]:qs[70] + n_big] = big
    qo_h[qs[70]:qs[70] + n_big] = np.arange(n_big) % 3000
    qd = torch.from_numpy(qd_h).to(dev)
    qo = torch.from_numpy(qo_h).to(dev)
    nq = len(sizes)
    # every tuple on the host: distinct (query, hash, offset) entries joined with the table
    ent = np.unique(np.rec.fromarrays([np.repeat(np.arange(nq), sizes), np.frombuffer(qd_h.tobytes(), "S10"), qo_h],
                                      names="q,h,o"))
    th = np.frombuffer(dig.tobytes(), "S10")
    trow = np.unique(np.rec.fromarrays([th, song, off], names="h,s,o"))
    lo = np.searchsorted(trow.h, ent.h, "left"); hi = np.searchsorted(trow.h, ent.h, "right")
    reps = hi - lo
    idx = np.repeat(lo, reps) + (np.arange(reps.sum()) - np.repeat(np.cumsum(reps) - reps, reps))
    t_q, t_qo = np.repeat(ent.q, reps), np.repeat(ent.o, reps)
    head = np.repeat(np.r_[True, (ent.q[1:] != ent.q[:-1]) | (ent.h[1:] != ent.h[:-1])], reps)
    t_song, t_diff = trow.s[idx].astype(np.int64), trow.o[idx].astype(np.int64) - t_qo
    assert len(t_q) > 1_000_000

    def run(topn):
        out = ix.query_batch(qd, qo, qs, topn, want_stats=True)
        return [t.cpu().numpy() for t in out[:5]], out[5]

    for topn in (1, 3, 9, 40):                          # 40 > kPvMaxTopn: the table vote for every query
        want = _np_vote(t_q, t_song, t_diff, head, nq, topn)
        assert want[4].max() == topn
        assert want[2][70, 0] == n_big and want[0][70, 0] == (nsongs + 1) * id_stride and want[1][70, 0] == 16
        for q in (0, 7, 50) if topn == 3 else (11,):     # the oracle's own Python functions on a subsample
            pairs = {(bytes(h).hex(), int(o)) for h, o in zip(qd_h[qs[q]:qs[q + 1]], qo_h[qs[q]:qs[q + 1]])}
            m, dd = O.return_matches(otable, pairs)
            best = O.best_offsets(m, topn)
            assert [tuple(b) for b in best] == [(int(want[0][q, r]), int(want[1][q, r]), int(want[2][q, r])) for r in range(want[4][q])]
            assert [dd[b[0]] for b in best] == [int(want[3][q, r]) for r in range(want[4][q])]
        # default = the partitioned vote (shared-memory tables; query 70's bin of 33000 matches does not fit a region and
        # goes to the table vote); SIA_PVOTE_CAP: small regions, so that most queries are split or handed over; regions
        # of 2 tuples overflow for almost every query, which then goes to the table vote
        names = ("SIA_VOTE_GROUP_TUPLES", "SIA_PVOTE_CAP")
        for setting in ((None, None), ("1000", None), ("200000", None), (str(1 << 40), None),
                        (None, "64"), ("200000", "1024"), (None, "2"), ("200000", "2")):
            for name, val in zip(names, setting):
                if val is None:
                    monkeypatch.delenv(name, raising=False)
                else:
                    monkeypatch.setenv(name, val)
            got, stats = run(topn)
            assert stats[0] == qs[-1] and stats[1] == int(head.sum()) and stats[2] == len(t_q), (stats, topn, setting)
            assert stats[3] == len(np.unique((t_q << 49) | (t_song << 25) | (t_diff + (1 << 24)))), (topn, setting)
            for a, b, name in zip(got, want, ("song", "diff", "count", "rows", "nres")):
                assert np.array_equal(a, b), (name, topn, setting, np.argwhere(a != b)[:5])
        for name in names:
            monkeypatch.delenv(name, raising=False)
        # the same tuples as vote keys in random order (the exchanged-keys vote of hash-prefix sharding); query ids < 2^14
        key = (head.astype(np.int64) << 63) | (t_q << 49) | (t_song << 25) | (t_diff + (1 << 24))
        perm = key[rng.permutation(len(key))]
        by_query = perm[np.argsort((perm >> 49) & 0x3fff, kind="stable")]      # grouped by query: the partitioned vote
        for label, arr, cap in (("any order", perm, None), ("by query", by_query, None), ("by query, small regions", by_query, "512")):
            if cap is None:
                monkeypatch.delenv("SIA_PVOTE_CAP", raising=False)
            else:
                monkeypatch.setenv("SIA_PVOTE_CAP", cap)
            got = [t.cpu().numpy() for t in vote_tuples(0, torch.from_numpy(arr).to(dev), nq, topn, int(song.max()))]
            for a, b, name in zip(got, want, ("song", "diff", "count", "rows", "nres")):
                assert np.array_equal(a, b), ("vote_tuples", label, name, topn, np.argwhere(a != b)[:5])
        monkeypatch.delenv("SIA_PVOTE_CAP", raising=False)
