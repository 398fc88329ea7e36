"""``GPUDatabase`` — the reference's database-backend interface on an HBM-resident index.

Registered as ``DATABASES['gpu'] = ("shazam_b200.database", "GPUDatabase")`` it slots into
``get_database`` (``__init__.py:24-27,54-67``).  The method set, argument meaning and
return shapes follow ``MySQLDatabase`` (``mysql_database.py:28-255``); ``find_matches``
follows ``ElasticDatabase`` (``elastic_database.py:195-226``).  The songs table lives on
the host (it is a few rows per track); the fingerprints table is ``sia_index`` on the GPU.

``cursor()`` understands exactly the statements the reference drivers issue through it:
the two CREATEs and DELETE_UNFINGERPRINTED (``__init__.py:421-424``) and SELECT_MULTIPLE
with ``UNHEX(%s)`` parameters (``recognizer.py:251-259``).
"""
from __future__ import annotations

import ctypes as C
import datetime
from typing import Iterable, Optional, Sequence

import os
import sys
import time

import numpy as np
import torch

from . import _native as N
from .fingerprinter import digests_to_hex, hex_to_digests

FIELD_SONG_ID = "song_id"
FIELD_SONGNAME = "song_name"
FIELD_FINGERPRINTED = "fingerprinted"
FIELD_FILE_SHA1 = "file_sha1"
FIELD_TOTAL_HASHES = "total_hashes"
FIELD_HASH = "hash"
FIELD_OFFSET = "offset"
SONGS_TABLENAME = "songs"
FINGERPRINTS_TABLENAME = "fingerprints"


# the reference's backend registry (__init__.py:24-27) with this backend added
DATABASES = {
    "mysql": ("mysql_database", "MySQLDatabase"),
    "postgres": ("dejavu.database_handler.postgres_database", "PostgreSQLDatabase"),
    "gpu": ("shazam_b200.database", "GPUDatabase"),
}


def get_database(database_type: str = "gpu"):
    """``__init__.py:54-67``: resolve a backend CLASS by name; unknown names raise TypeError."""
    import importlib
    try:
        path, db_class_name = DATABASES[database_type]
        return getattr(importlib.import_module(path), db_class_name)
    except (ImportError, KeyError):
        raise TypeError("Unsupported database type supplied.")


class FingerprintIndex:
    """Thin owner of one ``sia_index`` (one shard of the fingerprints table on one GPU)."""

    def __init__(self, device: int = 0, capacity_rows: int = 1 << 24):
        if not torch.cuda.is_available():
            raise RuntimeError("sia_b200 needs a CUDA device (B200); there is no CPU fallback")
        self.lib = N.lib()
        self.device = int(device)
        self.tdev = torch.device("cuda", self.device)
        self.capacity = int(capacity_rows)
        h = C.c_void_p()
        N.check(self.lib.sia_index_create(self.device, self.capacity, C.byref(h)))
        self._h = h
        self._dirty = False

    def close(self):
        if getattr(self, "_h", None):
            self.lib.sia_index_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.tdev).cuda_stream)

    @property
    def rows(self) -> int:
        self.finalize()
        return int(self.lib.sia_index_rows(self._h))

    # ---- build -------------------------------------------------------------------------
    def insert(self, song_id: int, digests, offsets) -> None:
        """Append rows (pending until ``finalize``).  Host arrays or CUDA tensors."""
        n = len(offsets)
        if n == 0:
            return
        if isinstance(digests, torch.Tensor) and digests.is_cuda:
            d = digests.contiguous()
            o = offsets.to(torch.int32).contiguous()
            assert d.dtype == torch.uint8 and d.shape == (n, N.HASH_BYTES)
            N.check(self.lib.sia_index_insert(self._h, int(song_id), C.c_void_p(d.data_ptr()),
                                              C.c_void_p(o.data_ptr()), n, self._stream()))
        else:
            d = np.ascontiguousarray(digests, np.uint8).reshape(n, N.HASH_BYTES)
            o = np.ascontiguousarray(offsets, np.int32)
            N.check(self.lib.sia_index_insert_host(self._h, int(song_id), C.c_void_p(d.ctypes.data),
                                                   C.c_void_p(o.ctypes.data), n))
        self._dirty = True

    def insert_rows(self, songs: torch.Tensor, digests: torch.Tensor, offsets: torch.Tensor) -> None:
        """Rows of many songs at once (CUDA tensors; ``songs[i]`` is row i's song id)."""
        n = offsets.numel()
        if n == 0:
            return
        s = songs.to(torch.int32).contiguous()
        d = digests.contiguous()
        o = offsets.to(torch.int32).contiguous()
        N.check(self.lib.sia_index_insert_rows(self._h, C.c_void_p(s.data_ptr()), C.c_void_p(d.data_ptr()),
                                               C.c_void_p(o.data_ptr()), n, self._stream()))
        self._dirty = True

    def finalize(self) -> int:
        if self._dirty:
            r = C.c_int64()
            N.check(self.lib.sia_index_finalize(self._h, C.byref(r)))
            self._dirty = False
        return int(self.lib.sia_index_rows(self._h))

    def delete_songs(self, song_ids: Sequence[int]) -> int:
        self.finalize()
        ids = np.ascontiguousarray(list(song_ids), np.int32)
        r = C.c_int64()
        N.check(self.lib.sia_index_delete_songs(self._h, ids.ctypes.data_as(C.POINTER(C.c_int32)), len(ids), C.byref(r)))
        return int(r.value)

    def export(self, first_row: int = 0, n: Optional[int] = None):
        """Rows ``[first_row, first_row + n)`` of the sorted table as CUDA tensors
        (digest uint8[n,10], song_id int32[n], offset int32[n]), in (hash, song_id, offset) order."""
        total = self.finalize()
        n = total - first_row if n is None else int(n)
        d = torch.empty((n, N.HASH_BYTES), dtype=torch.uint8, device=self.tdev)
        s = torch.empty(n, dtype=torch.int32, device=self.tdev)
        o = torch.empty(n, dtype=torch.int32, device=self.tdev)
        N.check(self.lib.sia_index_export(self._h, int(first_row), n, C.c_void_p(d.data_ptr()), C.c_void_p(s.data_ptr()),
                                          C.c_void_p(o.data_ptr()), self._stream()))
        torch.cuda.current_stream(self.tdev).synchronize()
        return d, s, o

    # ---- lookup ------------------------------------------------------------------------
    def select(self, digests: np.ndarray):
        """SELECT_MULTIPLE: every stored row whose hash is in ``digests`` (distinct).
        Returns (hash_index, song_id, offset) int32 arrays."""
        self.finalize()
        d = np.ascontiguousarray(digests, np.uint8).reshape(-1, N.HASH_BYTES)
        n = len(d)
        cap = max(1024, 8 * n)
        while True:
            idx = np.empty(cap, np.int32); sid = np.empty(cap, np.int32); off = np.empty(cap, np.int32)
            nr = C.c_int64()
            N.check(self.lib.sia_index_select_host(self._h, C.c_void_p(d.ctypes.data), n, C.c_void_p(idx.ctypes.data),
                                                   C.c_void_p(sid.ctypes.data), C.c_void_p(off.ctypes.data), cap,
                                                   C.byref(nr)))
            if nr.value <= cap:
                m = nr.value
                order = np.argsort(idx[:m], kind="stable")      # the device answers in hash order: back to IN-list order
                return idx[:m][order], sid[:m][order], off[:m][order]
            cap = int(nr.value)

    def query_batch(self, digests: torch.Tensor, qoffsets: torch.Tensor, query_starts: np.ndarray, topn: int,
                    want_stats: bool = False):
        """return_matches + the align_matches vote for Q queries.  Returns CUDA int32 tensors
        (song[Q,topn], diff[Q,topn], count[Q,topn], rows[Q,topn], nres[Q]) (+ stats)."""
        t0 = time.perf_counter()
        self.finalize()
        qs = np.ascontiguousarray(query_starts, np.int64)
        Q = len(qs) - 1
        d = digests.contiguous()
        o = qoffsets.to(torch.int32).contiguous()
        assert d.is_cuda and o.is_cuda and d.dtype == torch.uint8
        outs = [torch.zeros((Q, topn), dtype=torch.int32, device=self.tdev) for _ in range(4)]
        nres = torch.zeros(Q, dtype=torch.int32, device=self.tdev)
        stats = (C.c_int64 * 4)()
        N.check(self.lib.sia_index_query_batch(self._h, C.c_void_p(d.data_ptr()), C.c_void_p(o.data_ptr()),
                                               qs.ctypes.data_as(C.POINTER(C.c_int64)), Q, int(topn),
                                               C.c_void_p(outs[0].data_ptr()), C.c_void_p(outs[1].data_ptr()),
                                               C.c_void_p(outs[2].data_ptr()), C.c_void_p(outs[3].data_ptr()),
                                               C.c_void_p(nres.data_ptr()), stats, self._stream()))
        if os.environ.get("SIA_QUERY_TIMING"):
            print("[sia] query_batch python wall %.2f ms" % ((time.perf_counter() - t0) * 1e3), file=sys.stderr)
        if want_stats:
            return (*outs, nres, list(stats))
        return (*outs, nres)

    def query_batch_apriori(self, digests: torch.Tensor, qoffsets: torch.Tensor, query_starts: np.ndarray, topn: int,
                            batch_hashes: int = 1000, want_stats: bool = False):
        """The a-priori early exit of ``recognizer_apriori.py:246-310`` for Q queries: each query's distinct hashes are
        read in batches of ``batch_hashes`` in ascending digest order, and the query stops once its best song has more
        than twice the matched DB rows of the runner-up.  Returns the five tensors of ``query_batch`` at that point,
        plus ``batches[Q]`` (batches read) and ``exit[Q]`` (1 if the rule fired) (+ stats: query pairs, DB rows read,
        vote tuples read, batches read)."""
        self.finalize()
        qs = np.ascontiguousarray(query_starts, np.int64)
        Q = len(qs) - 1
        d = digests.contiguous()
        o = qoffsets.to(torch.int32).contiguous()
        assert d.is_cuda and o.is_cuda and d.dtype == torch.uint8
        outs = [torch.zeros((Q, topn), dtype=torch.int32, device=self.tdev) for _ in range(4)]
        per_q = [torch.zeros(Q, dtype=torch.int32, device=self.tdev) for _ in range(3)]      # nres, batches, exit
        stats = (C.c_int64 * 4)()
        N.check(self.lib.sia_index_query_apriori(self._h, C.c_void_p(d.data_ptr()), C.c_void_p(o.data_ptr()),
                                                 qs.ctypes.data_as(C.POINTER(C.c_int64)), Q, int(topn), int(batch_hashes),
                                                 *[C.c_void_p(t.data_ptr()) for t in outs + per_q], stats, self._stream()))
        if want_stats:
            return (*outs, *per_q, list(stats))
        return (*outs, *per_q)

    def trim(self) -> None:
        """Release build / lookup / vote scratch (re-allocated on demand); the table stays."""
        self.finalize()
        N.check(self.lib.sia_index_trim(self._h))

    def query_timing(self):
        """(lookup ms, vote ms): device time of the last ``query_batch`` call (CUDA events on its stream)."""
        ms = (C.c_double * 2)()
        N.check(self.lib.sia_index_query_timing(self._h, ms))
        return float(ms[0]), float(ms[1])

    @property
    def keys(self) -> int:
        """Distinct hashes stored (one 16-byte key entry each; postings are 8 bytes per row)."""
        self.finalize()
        return int(self.lib.sia_index_keys(self._h))

    @property
    def max_song(self) -> int:
        """Largest song id ever inserted (sizes the dense per-query song tables of the vote)."""
        self.finalize()
        return int(self.lib.sia_index_max_song(self._h))

    # ---- hash-prefix sharding: the device steps around the two all-to-alls (distributed.ShardedIndex) ------------
    def expand_slots(self, entry_slots: torch.Tensor, world: int, queries_per_rank: int, key_cap: int,
                     info: torch.Tensor) -> torch.Tensor:
        """Received entry slots (int64[world, entry_cap, 2]) -> vote-key slots int64[world, key_cap] for the
        ranks that own the queries; ``info`` (int64[4], zeroed per pass) accumulates overflow flags and sizes."""
        self.finalize()
        assert entry_slots.is_cuda and entry_slots.dtype == torch.int64 and entry_slots.is_contiguous()
        entry_cap = entry_slots.shape[1]
        out = torch.empty((world, int(key_cap)), dtype=torch.int64, device=self.tdev)
        N.check(self.lib.sia_index_expand_slots(self._h, C.c_void_p(entry_slots.data_ptr()), int(world), int(entry_cap),
                                                int(queries_per_rank), C.c_void_p(out.data_ptr()), int(key_cap),
                                                C.c_void_p(info.data_ptr()), self._stream()))
        return out

    def lookup_slots(self, entry_slots: torch.Tensor, world: int, queries_per_rank: int, info: torch.Tensor) -> torch.Tensor:
        """Peer-memory pass, step 1 on the shard: sort + look up the received entries (kept inside the handle) and
        return the vote tuples this shard holds for every global query, int64[world * queries_per_rank]."""
        self.finalize()
        assert entry_slots.is_cuda and entry_slots.dtype == torch.int64 and entry_slots.is_contiguous()
        t = torch.zeros(world * queries_per_rank, dtype=torch.int64, device=self.tdev)
        N.check(self.lib.sia_index_lookup_slots(self._h, C.c_void_p(entry_slots.data_ptr()), int(world), int(entry_slots.shape[1]),
                                                int(queries_per_rank), C.c_void_p(t.data_ptr()), C.c_void_p(info.data_ptr()),
                                                self._stream()))
        return t

    def scatter_peers(self, world: int, queries_per_rank: int, tuples_total: torch.Tensor, peers: "PeerBuffers",
                      info: torch.Tensor) -> None:
        """Step 2 on the shard: posting runs -> vote tuples -> the owners' regions, through NVLink."""
        t = tuples_total.contiguous()
        N.check(self.lib.sia_index_scatter_peers(self._h, int(world), int(peers.rank), int(queries_per_rank), C.c_void_p(t.data_ptr()),
                                                 peers.p_regions, peers.p_fill, peers.p_qover, peers.region_cap, peers.fill_cap,
                                                 C.c_void_p(info.data_ptr()), self._stream()))


class _RawCuda:
    """A device pointer as an object torch can alias (``__cuda_array_interface__``)."""

    def __init__(self, ptr: int, n: int, typestr: str):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (int(ptr), False), "version": 2}


class PeerBuffers:
    """The regions of the partitioned vote of one rank, mapped by every rank of the group (CUDA IPC over NVLink):
    ``[query flags: qp x u32][fill counters: fill_cap x u32][regions: region_cap x u64]``.  ``PeerBuffers.create`` is the
    collective constructor: every rank allocates, the 64-byte handles are all-gathered, every rank opens the others'.
    (``__init__`` + ``connect`` are the two halves; a test that plays all ranks on one GPU connects local pointers.)"""

    def __init__(self, device: int, rank: int, world: int, qp: int, region_cap: int, fill_cap: int):
        self.lib = N.lib()
        self.device, self.rank, self.world = device, rank, world
        self.qp, self.region_cap, self.fill_cap = int(qp), int(region_cap), int(fill_cap)
        up = lambda x: (x + 255) // 256 * 256
        self.off_fill = up(4 * self.qp)
        self.off_regions = up(self.off_fill + 4 * self.fill_cap)
        self.nbytes = self.off_regions + 8 * self.region_cap
        ptr = C.c_void_p()
        handle = (C.c_uint8 * 64)()
        N.check(self.lib.sia_peer_alloc(device, self.nbytes, C.byref(ptr), C.cast(handle, C.c_void_p)))
        self.local = int(ptr.value)
        self.handle = bytes(handle)
        self.base, self._opened = None, []
        # local counters (query flags + fill) as one int32 tensor, for the stream-ordered zeroing before every pass
        self.counters = torch.as_tensor(_RawCuda(self.local, self.off_regions // 4, "<i4"), device=torch.device("cuda", device))

    def connect(self, bases) -> None:
        """``bases[r]``: rank r's buffer as a pointer valid in THIS process."""
        self.base = [int(b) for b in bases]
        arr = lambda off: (C.c_void_p * self.world)(*[b + off for b in self.base])
        self.p_qover, self.p_fill, self.p_regions = arr(0), arr(self.off_fill), arr(self.off_regions)

    @classmethod
    def create(cls, device: int, rank: int, world: int, qp: int, region_cap: int, fill_cap: int, group=None) -> "PeerBuffers":
        import torch.distributed as dist
        self = cls(device, rank, world, qp, region_cap, fill_cap)
        handles = [None] * world
        dist.all_gather_object(handles, self.handle, group=group)
        bases = []
        for r in range(world):
            if r == rank:
                bases.append(self.local)
                continue
            q = C.c_void_p()
            buf = (C.c_uint8 * 64).from_buffer_copy(handles[r])
            N.check(self.lib.sia_peer_open(device, C.cast(buf, C.c_void_p), C.byref(q)))
            bases.append(int(q.value))
            self._opened.append(int(q.value))
        self.connect(bases)
        return self

    def close(self, group=None):
        if self.local is None:
            return
        torch.cuda.synchronize(self.device)
        for b in self._opened:
            N.check(self.lib.sia_peer_close(self.device, C.c_void_p(b)))
        if self._opened:
            import torch.distributed as dist
            dist.barrier(group=group)             # nobody maps this rank's buffer any more
        self._opened = []
        del self.counters
        N.check(self.lib.sia_peer_free(self.device, C.c_void_p(self.local)))
        self.local = None


def vote_count_regions(device: int, tuples_total: torch.Tensor, n_queries: int, topn: int, peers: "PeerBuffers", info: torch.Tensor):
    """The owner's half of the peer-memory pass: count the regions the shards filled (``sia_vote_count_regions``)."""
    lib = N.lib()
    tdev = torch.device("cuda", device)
    outs, nres = _vote_outputs(tdev, n_queries, topn)
    t = tuples_total.contiguous()
    N.check(lib.sia_vote_count_regions(device, C.c_void_p(t.data_ptr()), int(n_queries), int(topn),
                                       C.c_void_p(peers.local + peers.off_regions), C.c_void_p(peers.local + peers.off_fill),
                                       C.c_void_p(peers.local), peers.region_cap, peers.fill_cap,
                                       C.c_void_p(outs[0].data_ptr()), C.c_void_p(outs[1].data_ptr()), C.c_void_p(outs[2].data_ptr()),
                                       C.c_void_p(outs[3].data_ptr()), C.c_void_p(nres.data_ptr()), C.c_void_p(info.data_ptr()),
                                       C.c_void_p(torch.cuda.current_stream(tdev).cuda_stream)))
    return (*outs, nres)


def route_entries(device: int, digests: torch.Tensor, qoffsets: torch.Tensor, query_starts: torch.Tensor, qid_base: int,
                  world: int, slot_cap: int, status: torch.Tensor) -> torch.Tensor:
    """(hash, offset) pairs of this rank's queries -> one slot of packed entries per destination shard
    (int64[world, slot_cap, 2]; element 0 of a slot is its count).  ``query_starts``: int64[Q+1] on the device."""
    lib = N.lib()
    tdev = torch.device("cuda", device)
    d = digests.contiguous(); o = qoffsets.to(torch.int32).contiguous()
    n = o.numel()
    nq = query_starts.numel() - 1
    slots = torch.empty((world, int(slot_cap), 2), dtype=torch.int64, device=tdev)
    N.check(lib.sia_route_entries(device, C.c_void_p(d.data_ptr()), C.c_void_p(o.data_ptr()),
                                  C.c_void_p(query_starts.data_ptr()), nq, n, int(qid_base), int(world), int(slot_cap),
                                  C.c_void_p(slots.data_ptr()), C.c_void_p(status.data_ptr()),
                                  C.c_void_p(torch.cuda.current_stream(tdev).cuda_stream)))
    return slots


def _vote_outputs(tdev, n_queries, topn):
    outs = [torch.zeros((n_queries, topn), dtype=torch.int32, device=tdev) for _ in range(4)]
    return outs, torch.zeros(n_queries, dtype=torch.int32, device=tdev)


def vote_key_slots(device: int, key_slots: torch.Tensor, n_queries: int, topn: int, max_song: int, defer: bool = False):
    """Vote the key slots received from every shard (int64[world, key_cap], element 0 of a slot = its count).
    ``defer=True`` returns once the work is enqueued on the current stream; ``vote_finish(device)`` completes it (keep
    ``key_slots`` and the returned tensors alive until then)."""
    lib = N.lib()
    tdev = torch.device("cuda", device)
    outs, nres = _vote_outputs(tdev, n_queries, topn)
    ks = key_slots.contiguous()
    N.check(lib.sia_vote_key_slots(device, C.c_void_p(ks.data_ptr()), ks.shape[0], ks.shape[1], n_queries, int(topn),
                                   int(max_song), C.c_void_p(outs[0].data_ptr()), C.c_void_p(outs[1].data_ptr()),
                                   C.c_void_p(outs[2].data_ptr()), C.c_void_p(outs[3].data_ptr()),
                                   C.c_void_p(nres.data_ptr()), 1 if defer else 0,
                                   C.c_void_p(torch.cuda.current_stream(tdev).cuda_stream)))
    return (*outs, nres)


def vote_finish(device: int) -> None:
    N.check(N.lib().sia_vote_finish(device))


def vote_tuples(device: int, keys: torch.Tensor, n_queries: int, topn: int, max_song: int):
    """The align_matches vote over vote keys in any order (head | query | song | diff + 2^24, ``sia_b200.h``).
    CUDA tensors in and out."""
    lib = N.lib()
    tdev = torch.device("cuda", device)
    outs, nres = _vote_outputs(tdev, n_queries, topn)
    k = keys.contiguous()
    N.check(lib.sia_vote_tuples(device, C.c_void_p(k.data_ptr()), k.numel(), n_queries, int(topn), int(max_song),
                                C.c_void_p(outs[0].data_ptr()), C.c_void_p(outs[1].data_ptr()),
                                C.c_void_p(outs[2].data_ptr()), C.c_void_p(outs[3].data_ptr()),
                                C.c_void_p(nres.data_ptr()), C.c_void_p(torch.cuda.current_stream(tdev).cuda_stream)))
    return (*outs, nres)


class _Cursor:
    """What ``db.cursor()`` yields: ``execute(sql, params)`` + row iteration for the statements
    the reference issues through a raw cursor."""

    def __init__(self, db: "GPUDatabase", dictionary: bool = False):
        self.db = db
        self.rows = []
        self.lastrowid = None

    def __enter__(self):
        return self

    def __exit__(self, extype, exvalue, tb):
        return False

    def execute(self, query: str, params=None):
        q = " ".join(query.split())
        db = self.db
        if q.startswith("CREATE TABLE"):
            self.rows = []
        elif q.startswith("DELETE FROM") and FIELD_FINGERPRINTED in q:
            db.delete_unfingerprinted()
            self.rows = []
        elif q.startswith("SELECT HEX(") and " IN (" in q:
            values = list(params or [])
            if q.count("UNHEX(%s)") != len(values):
                raise ValueError("SELECT_MULTIPLE: parameter count does not match the IN list")
            self.rows = db.select_multiple(values)
        else:
            raise N.SiaError(N.E_UNSUPPORTED, f"GPUDatabase cursor does not implement: {q[:80]}")
        return len(self.rows)

    def __iter__(self):
        return iter(self.rows)

    def fetchone(self):
        return self.rows[0] if self.rows else None

    def fetchall(self):
        return list(self.rows)

    def close(self):
        pass


class GPUDatabase:
    type = "gpu"

    # statements the drivers pass to cursor.execute (same attribute names as MySQLDatabase)
    CREATE_SONGS_TABLE = f"CREATE TABLE IF NOT EXISTS `{SONGS_TABLENAME}` (host-side table)"
    CREATE_FINGERPRINTS_TABLE = f"CREATE TABLE IF NOT EXISTS `{FINGERPRINTS_TABLENAME}` (sia_index in HBM)"
    DELETE_UNFINGERPRINTED = f"DELETE FROM `{SONGS_TABLENAME}` WHERE `{FIELD_FINGERPRINTED}` = 0;"
    SELECT_MULTIPLE = (f"SELECT HEX(`{FIELD_HASH}`), `{FIELD_SONG_ID}`, `{FIELD_OFFSET}` "
                       f"FROM `{FINGERPRINTS_TABLENAME}` WHERE `{FIELD_HASH}` IN (%s);")
    IN_MATCH = "UNHEX(%s)"

    def __init__(self, device: Optional[int] = None, capacity_rows: int = 1 << 24, metadata: Optional[dict] = None,
                 **options):
        # host/user/password/database of config["database"] (__init__.py:29-37) are accepted and ignored
        self._options = dict(options, device=device, capacity_rows=capacity_rows, metadata=metadata)
        dev = torch.cuda.current_device() if device is None and torch.cuda.is_available() else (device or 0)
        self.index = FingerprintIndex(dev, capacity_rows)
        self.songs = {}           # song_id -> dict(song_name, file_sha1, total_hashes, fingerprinted, date_created)
        self._next_id = 1         # MEDIUMINT UNSIGNED AUTO_INCREMENT
        self._metadata = metadata or {}

    # ---- MySQLDatabase surface ------------------------------------------------------------
    def setup(self) -> None:
        with self.cursor() as cur:
            cur.execute(self.CREATE_SONGS_TABLE)
            cur.execute(self.CREATE_FINGERPRINTS_TABLE)
            cur.execute(self.DELETE_UNFINGERPRINTED)

    def cursor(self, **options):
        return _Cursor(self, **options)

    def after_fork(self) -> None:
        pass

    def insert_song(self, song_name: str, file_hash: str, total_hashes: int) -> int:
        sid = self._next_id
        if sid >= 1 << 24:
            raise N.SiaError(N.E_CAPACITY, "song_id exceeds MEDIUMINT UNSIGNED")
        self._next_id += 1
        self.songs[sid] = {FIELD_SONGNAME: song_name, FIELD_FILE_SHA1: str(file_hash).upper(),
                           FIELD_TOTAL_HASHES: int(total_hashes), FIELD_FINGERPRINTED: 0,
                           "date_created": datetime.datetime.now()}
        return sid

    def insert_hashes(self, song_id: int, hashes, batch_size: int = 1000) -> None:
        """``hashes``: iterable of ``(hex20, offset)`` (a set in the ingest flow, ``__init__.py:265,383``)."""
        hashes = list(hashes)
        if not hashes:
            return
        d = hex_to_digests([h for h, _ in hashes])
        o = np.array([int(t) for _, t in hashes], np.int64)
        if o.min() < 0 or o.max() >= 1 << 24:
            raise N.SiaError(N.E_INVALID, "offset outside 0..2^24-1")
        self.index.insert(song_id, d, o.astype(np.int32))

    def insert_hashes_array(self, song_id: int, digests, offsets) -> None:
        """Array fast path: uint8[N,10] digests + int32 offsets (host arrays or CUDA tensors)."""
        self.index.insert(song_id, digests, offsets)

    def set_song_fingerprinted(self, song_id: int) -> None:
        self.songs[song_id][FIELD_FINGERPRINTED] = 1

    def delete_unfingerprinted(self) -> None:
        dead = [sid for sid, s in self.songs.items() if not s[FIELD_FINGERPRINTED]]
        if dead:
            self.index.delete_songs(dead)      # ON DELETE CASCADE
            for sid in dead:
                del self.songs[sid]

    def get_songs(self):
        """Rows ``(song_id, song_name, file_sha1, total_hashes, date_created)`` of fingerprinted songs
        — ``row[2]`` is the upper-hex file SHA-1 (``FIELD_FILE_SHA1 = 2``, ``__init__.py:40,413``)."""
        return [(sid, s[FIELD_SONGNAME], s[FIELD_FILE_SHA1], s[FIELD_TOTAL_HASHES], s["date_created"])
                for sid, s in sorted(self.songs.items()) if s[FIELD_FINGERPRINTED]]

    def get_song_by_id(self, song_id: int):
        s = self.songs[int(song_id)]
        return {"song_name": s[FIELD_SONGNAME], "total_hashes": s[FIELD_TOTAL_HASHES], "file_sha1": s[FIELD_FILE_SHA1]}

    def get_metadata(self, song_id: int):
        return self._metadata.get(int(song_id))

    def get_num_fingerprints(self) -> int:
        return self.index.rows

    # ---- lookups ----------------------------------------------------------------------------
    def select_multiple(self, hex_values: Sequence[str]):
        """Rows ``(HEXUPPER, song_id, offset)`` for ``WHERE hash IN (...)``."""
        if not hex_values:
            return []
        uniq = list(dict.fromkeys(v.upper() for v in hex_values))      # SQL IN is a set
        idx, sid, off = self.index.select(hex_to_digests(uniq))
        return [(uniq[i], int(s), int(o)) for i, s, o in zip(idx.tolist(), sid.tolist(), off.tolist())]

    def find_matches(self, hashes: Iterable[str]):
        """ES-style lookup (``elastic_database.py:195-226``): docs ``{'_source': {...}}``."""
        hx = list(dict.fromkeys(hashes))
        if not hx:
            return
        idx, sid, off = self.index.select(hex_to_digests(hx))
        for i, s, o in zip(idx.tolist(), sid.tolist(), off.tolist()):
            yield {"_source": {FIELD_HASH: hx[i], FIELD_SONG_ID: int(s), FIELD_OFFSET: int(o)}}

    # ---- persistence in the reference's on-disk vocabulary -----------------------------------------
    ROW_DTYPE = np.dtype([("hash", "V10"), ("song_id", "<u4"), ("offset", "<u4")])    # BINARY(10), MEDIUMINT, INT

    def iter_sql_rows(self, chunk_rows: int = 1 << 20):
        """``(song_id, HEXUPPER, offset)`` tuples — the parameter rows of ``INSERT_FINGERPRINT``
        (``mysql_database.py:62-68``), so ``cur.executemany(MySQLDatabase.INSERT_FINGERPRINT, rows)`` seeds a
        MySQL `fingerprints` table from this index."""
        total = self.index.finalize()
        for first in range(0, total, chunk_rows):
            d, s, o = self.index.export(first, min(chunk_rows, total - first))
            hx = digests_to_hex(d)
            for h, sid, off in zip(hx, s.cpu().tolist(), o.cpu().tolist()):
                yield sid, h.upper(), off

    def dump(self, path: str, chunk_rows: int = 1 << 24) -> int:
        """Write ``<path>/songs.json`` (the `songs` table) and ``<path>/fingerprints.bin`` (the `fingerprints`
        table as packed ``ROW_DTYPE`` records).  Returns the number of fingerprint rows."""
        import json
        import os
        os.makedirs(path, exist_ok=True)
        total = self.index.finalize()
        with open(os.path.join(path, "fingerprints.bin"), "wb") as f:
            for first in range(0, total, chunk_rows):
                n = min(chunk_rows, total - first)
                d, s, o = self.index.export(first, n)
                rec = np.empty(n, self.ROW_DTYPE)
                rec["hash"] = np.frombuffer(d.cpu().numpy().tobytes(), dtype="V10")
                rec["song_id"] = s.cpu().numpy()
                rec["offset"] = o.cpu().numpy()
                rec.tofile(f)
        songs = {str(sid): {k: (v.isoformat() if hasattr(v, "isoformat") else v) for k, v in row.items()}
                 for sid, row in self.songs.items()}
        with open(os.path.join(path, "songs.json"), "w") as f:
            json.dump({"next_id": self._next_id, "songs": songs, "rows": total}, f)
        return total

    @classmethod
    def load(cls, path: str, device: Optional[int] = None, capacity_rows: Optional[int] = None,
             chunk_rows: int = 1 << 24, **options) -> "GPUDatabase":
        """Rebuild a database from ``dump``'s files (or from rows exported out of MySQL in ``ROW_DTYPE``)."""
        import json
        import os
        meta = json.load(open(os.path.join(path, "songs.json")))
        rec = np.memmap(os.path.join(path, "fingerprints.bin"), dtype=cls.ROW_DTYPE, mode="r")
        db = cls(device=device, capacity_rows=capacity_rows or max(len(rec) + (len(rec) >> 3), 1 << 16), **options)
        for sid, row in meta["songs"].items():
            row = dict(row)
            row["date_created"] = datetime.datetime.fromisoformat(row["date_created"])
            db.songs[int(sid)] = row
        db._next_id = int(meta["next_id"])
        for first in range(0, len(rec), chunk_rows):
            part = np.ascontiguousarray(rec[first:first + chunk_rows])
            d = torch.from_numpy(np.frombuffer(part["hash"].tobytes(), np.uint8).reshape(-1, N.HASH_BYTES).copy())
            db.index.insert_rows(torch.from_numpy(part["song_id"].astype(np.int32)).to(db.index.tdev), d.to(db.index.tdev),
                                 torch.from_numpy(part["offset"].astype(np.int32)).to(db.index.tdev))
        db.index.finalize()
        return db

    def __getstate__(self):
        """``mysql_database.py:202-204``: only the constructor options travel — the index lives in this process's GPU
        memory; the other side gets an EMPTY database with the same options (use ``dump``/``load`` to move rows)."""
        return (self._options,)

    def __setstate__(self, state):
        """``mysql_database.py:206-207``."""
        (options,) = state
        self.__init__(**options)
