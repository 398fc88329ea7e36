// K4 — shared declarations of the fingerprint index (index_store.cu: build side, index_query.cu: lookup + vote,
// index_dist.cu: the hash-prefix-sharded exchange steps).
//
// Storage ("hash once, postings packed"; replaces the MySQL `fingerprints` table, mysql_database.py:46-59):
//   keys : one 16-byte entry per DISTINCT hash, sorted by hash:
//            .y = digest bytes 0..7 (big-endian, so integer order = byte order)
//            .x = digest bytes 8..9 (16 bits) << 48 | first posting of the hash's run (48 bits)
//          keys[n_keys] is a sentinel (all-ones hash, start = n_rows), so a run's length is
//          keys[k+1].start - keys[k].start.
//   dir  : bucket directory on the top `dir_bits` bits of the digest -> first key of the bucket
//          (SHA-1 output is uniform: ~8 keys per bucket).
//   post : one 8-byte posting per fingerprint row, song_id (24 bits) << 24 | offset (24 bits), runs in key order,
//          sorted by (song_id, offset) inside a run — UNIQUE(song_id, offset, hash) / INSERT IGNORE is "no equal
//          neighbours".
// Rows waiting for sia_index_finalize ("pending") are 16-byte records (digest, song, offset) like a key entry with
// the posting in the low 48 bits; finalize sorts only the pending run and MERGES it into the table in place.
#pragma once
#include "sia_common.cuh"
#include "sort.cuh"

#include <algorithm>
#include <cstdlib>
#include <functional>
#include <string>
#include <utility>
#include <vector>

namespace sia {

constexpr uint64_t kM24 = 0xffffffull;
constexpr uint64_t kM48 = 0xffffffffffffull;

struct Arena {
  char *base = nullptr;
  size_t cap = 0, used = 0;
  int reserve(size_t bytes) {
    if (bytes <= cap) { used = 0; return SIA_OK; }
    if (base) cudaFree(base);
    base = nullptr; cap = 0; used = 0;
    size_t want = bytes + (bytes >> 3) + (1 << 20);
    SIA_CUDA(cudaMalloc(&base, want));
    cap = want;
    return SIA_OK;
  }
  template <typename T> T *take(size_t n) {
    used = (used + 255) & ~(size_t)255;
    T *p = reinterpret_cast<T *>(base + used);
    used += n * sizeof(T);
    return used <= cap ? p : nullptr;
  }
  void release() { if (base) cudaFree(base); base = nullptr; cap = used = 0; }
};

// Sorted, de-duplicated query entries of one pass with their posting runs.
struct Lookup {
  ulonglong2 *ent = nullptr;      // packed (qid, digest, qoff) entries, sorted
  int64_t *first = nullptr;       // first posting of the entry's run
  uint32_t *cnt_head = nullptr;   // run length if the entry is the first of its (query, hash), else 0
  int64_t *off_all = nullptr, *off_head = nullptr;   // exclusive scans of the run lengths / head run lengths
  int64_t n = 0, tuples = 0, head_rows = 0;
};

inline unsigned grid_for(int64_t n, int threads = 256) {
  int64_t b = ceil_div(n > 0 ? n : 1, threads);
  return (unsigned)std::min<int64_t>(b, kNumSMs * 32);
}

// ---- device helpers shared by the three translation units --------------------------------------------------
__device__ __forceinline__ void load_digest(const uint8_t *__restrict__ h, uint64_t &hi, uint32_t &lo16) {
  const uint16_t *p = reinterpret_cast<const uint16_t *>(h);   // 10*i is 2-byte aligned
  uint32_t w[5];
#pragma unroll
  for (int k = 0; k < 5; ++k) { const uint32_t v = p[k]; w[k] = ((v & 0xff) << 8) | (v >> 8); }   // big-endian pairs
  hi = ((uint64_t)w[0] << 48) | ((uint64_t)w[1] << 32) | ((uint64_t)w[2] << 16) | (uint64_t)w[3];
  lo16 = w[4];
}

__device__ __forceinline__ void store_digest(uint8_t *__restrict__ out, uint64_t hi, uint32_t lo16) {
  uint16_t *h = reinterpret_cast<uint16_t *>(out);
  const uint32_t w[5] = {(uint32_t)(hi >> 48) & 0xffffu, (uint32_t)(hi >> 32) & 0xffffu, (uint32_t)(hi >> 16) & 0xffffu,
                         (uint32_t)hi & 0xffffu, lo16 & 0xffffu};
#pragma unroll
  for (int k = 0; k < 5; ++k) h[k] = (uint16_t)(((w[k] & 0xff) << 8) | (w[k] >> 8));
}

__device__ __forceinline__ bool rec_eq(const ulonglong2 &a, const ulonglong2 &b) { return a.x == b.x && a.y == b.y; }
__device__ __forceinline__ bool rec_less(const ulonglong2 &a, const ulonglong2 &b) {
  return a.y < b.y || (a.y == b.y && a.x < b.x);
}
__device__ __forceinline__ bool same_hash(const ulonglong2 &a, const ulonglong2 &b) {
  return a.y == b.y && (a.x >> 48) == (b.x >> 48);
}

// first index in [lo, hi) of a hash-sorted array of 16-byte records (keys or pending rows: .y = digest high 64 bits,
// .x >> 48 = digest low 16 bits) whose digest >= (khi, klo16)
__device__ __forceinline__ int64_t hash_lower_bound(const ulonglong2 *__restrict__ r, int64_t lo, int64_t hi, uint64_t khi,
                                                    uint32_t klo16) {
  while (lo < hi) {
    const int64_t mid = lo + ((hi - lo) >> 1);
    const ulonglong2 v = r[mid];
    const bool less = v.y < khi || (v.y == khi && (uint32_t)(v.x >> 48) < klo16);
    if (less) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// the same through a bucket directory on the top `bits` bits of the digest (dir[b] = first record of bucket b,
// dir[2^bits] = n)
__device__ __forceinline__ int64_t hash_lower_bound_dir(const ulonglong2 *__restrict__ r, const uint32_t *__restrict__ dir,
                                                        int bits, uint64_t khi, uint32_t klo16) {
  const uint64_t b = khi >> (64 - bits);
  return hash_lower_bound(r, dir[b], dir[b + 1], khi, klo16);
}

// first index in [lo, hi) with a[i] >= v
__device__ __forceinline__ int64_t lower_bound_u64(const uint64_t *__restrict__ a, int64_t lo, int64_t hi, uint64_t v) {
  while (lo < hi) { const int64_t mid = lo + ((hi - lo) >> 1); if (a[mid] < v) lo = mid + 1; else hi = mid; }
  return lo;
}

// query entry record, sorted by all 16 bytes = (qid, digest, qoff):
//   .y = qid (24) | digest bits 79..40 (40)      .x = digest bits 39..16 (24) | digest lo16 (16) | qoff (24)
__device__ __forceinline__ ulonglong2 make_entry(uint32_t qid, uint64_t hi, uint32_t lo16, uint32_t qoff) {
  return make_ulonglong2(((hi & kM24) << 40) | ((uint64_t)lo16 << 24) | ((uint64_t)qoff & kM24),
                         ((uint64_t)qid << 40) | (hi >> 24));
}
__device__ __forceinline__ void entry_key(const ulonglong2 &e, uint64_t &khi, uint32_t &klo16, uint32_t &qid, uint32_t &qoff) {
  qid = (uint32_t)(e.y >> 40);
  khi = (e.y << 24) | (e.x >> 40);
  klo16 = (uint32_t)(e.x >> 24) & 0xffffu;
  qoff = (uint32_t)(e.x & kM24);
}

// ---- entry points shared between the translation units -----------------------------------------------------
// entries [0, n) packed by the caller into `a` (alt buffer `b`): sort by (query, hash, offset), look the hashes up.
// query_starts (device, may be NULL): the entries arrive grouped by query -> per-query shared-memory sort when every
// query has <= max_query_entries entries; else a global radix sort.  Synchronises the stream once (totals).
int lookup_sorted(::sia_index *ix, Arena &ar, ulonglong2 *a, ulonglong2 *b, int64_t n, const int64_t *d_query_starts,
                  int64_t i0, int n_queries, int64_t max_query_entries, Lookup &L, cudaStream_t s);
size_t lookup_bytes(int64_t n);

// vote of u64 keys (SIA vote-key layout, see sia_b200.h) stored in n_slots slots of `cap` keys, slot i holding
// d_counts[i] valid keys (a header-less layout; d_counts on the device)
int vote_key_slots(int device, const uint64_t *d_keys, int n_slots, int64_t cap, const int64_t *d_counts, int32_t n_queries,
                   int32_t topn, int32_t max_song, int32_t *d_out_song, int32_t *d_out_diff, int32_t *d_out_count,
                   int32_t *d_out_rows, int32_t *d_out_nres, cudaStream_t s, int defer);
int vote_key_slots_finish(int device);

// frees the per-device scratch of vote_key_slots
void vote_scratch_release(int device);

// keys of slot `sl` of a slotted key array: counts != NULL -> slot s holds counts[s] keys from its first element;
// counts == NULL -> element 0 of every slot is its count and the keys follow (the exchanged layout, index_dist.cu)
__device__ __forceinline__ const uint64_t *slot_keys(const uint64_t *__restrict__ keys, int64_t cap,
                                                     const int64_t *__restrict__ counts, int sl, int64_t &n) {
  const uint64_t *base = keys + (int64_t)sl * cap;
  if (counts) { n = min(counts[sl], cap); return base; }
  n = min((int64_t)base[0], cap - 1);
  return base + 1;
}

// ---- the table vote's per-query HBM tables (index_query.cu), shared with the a-priori rounds (index_apriori.cu) ----------
namespace tvote {

constexpr int kQidBits = SIA_KEY_QID_BITS, kSongBits = SIA_KEY_SONG_BITS, kDiffBits = SIA_KEY_DIFF_BITS;
constexpr int64_t kMaxQueriesPerPass = 1ll << kQidBits;
constexpr uint64_t kDiffMask = (1ull << kDiffBits) - 1;
constexpr int kTopK = 4;                  // results extracted per scan of a query's song table

struct QMeta {
  int64_t bin_base, song_base, filt_base;   // first slot / word of the query's sub-tables inside the group's tables
  int64_t cand_base;                        // first entry of the query's candidate list
  uint32_t bin_cap, song_cap, filt_words, cand;   // cand: tuples in twice-hit buckets (pass 1), sizes the bin table
  uint32_t cursor, pad_;                    // candidates collected so far (pass 2)
};

struct Tables {
  unsigned long long *bins;       // [nb] key words ((song << 25 | biased diff) + 1; 0 = empty)
  uint32_t *bin_cnt;              // [nb]
  unsigned long long *song_best;  // [ns]
  uint32_t *song_key;             // [ns] open addressing only (song + 1)
  uint32_t *filter;               // [nf]
  unsigned long long *cand;       // [nb / 2] candidate vote keys (query | song | biased diff), per-query lists
};

// queries [qa, qb) of a pass as one group: sub-table layout of its queries in h_meta (filter words = tuples + 1, song
// slots dense = span or open addressing = 2 * head rows + 32) from the scanned tuple / head-row offsets at the queries'
// first entries
struct Group { int qa, qb; bool dense; int64_t nf, ns; };
Group make_group(int qa, int qb, const int64_t *h_off_all, const int64_t *h_off_head, int64_t span, QMeta *h_meta);

// the groups [qa, qb) of consecutive queries q of a pass with keep[q] != 0 (keep NULL: every query), each within
// `budget` vote tuples or a single query; groups without tuples are left out
std::vector<std::pair<int, int>> split_groups(const int64_t *h_off_all, int nq, int64_t budget, const uint32_t *keep);

__device__ __forceinline__ uint32_t mix32(uint32_t k) {
  k ^= k >> 16; k *= 0x85ebca6bu; k ^= k >> 13; k *= 0xc2b2ae35u; k ^= k >> 16;
  return k;
}
__device__ __forceinline__ uint32_t slot_of(uint32_t h, uint32_t cap) { return (uint32_t)(((uint64_t)h * cap) >> 32); }

// song slot of `song` in query m's song table (dense: the id itself; else find-or-insert by open addressing)
template <bool DENSE>
__device__ __forceinline__ int64_t song_slot(const QMeta &m, uint32_t song, uint32_t *__restrict__ song_key) {
  if (DENSE) return song < m.song_cap ? m.song_base + song : -1;
  uint32_t t = slot_of(mix32(song), m.song_cap);
  for (uint32_t probes = 0; probes < m.song_cap; ++probes) {     // bounded: a full table (inconsistent inputs) cannot hang
    const uint32_t old = atomicCAS(&song_key[m.song_base + t], 0u, song + 1u);
    if (old == 0u || old == song + 1u) return m.song_base + t;
    if (++t == m.song_cap) t = 0;
  }
  return -1;
}

// count one vote tuple (song, biased diff) in query m's bin table; returns the bin's count including this tuple
// (0 and flag 8 if the table is full, which the sizing rules out)
__device__ __forceinline__ unsigned long long bin_count(const QMeta &m, uint32_t song, uint32_t dbits, const Tables &T,
                                                        uint32_t &fresh, int32_t *__restrict__ flags) {
  const unsigned long long key = (((unsigned long long)song << kDiffBits) | dbits) + 1ull;     // never 0
  uint32_t s = slot_of(mix32(song * 0x9e3779b1u + dbits), m.bin_cap);
  for (uint32_t probes = 0; probes < m.bin_cap; ++probes) {
    const int64_t at = m.bin_base + s;
    const unsigned long long old = atomicCAS(T.bins + at, 0ull, key);
    if (old == 0ull) ++fresh;
    if (old == 0ull || old == key) return (unsigned long long)atomicAdd(T.bin_cnt + at, 1u) + 1ull;
    if (++s == m.bin_cap) s = 0;
  }
  atomicOr(flags, 8);
  return 0;
}

// song best key: count (high) | inverted biased diff, so the largest key is the largest count with the smallest
// difference (Python's max() keeps the first maximum, recognizer.py:308)
__device__ __forceinline__ unsigned long long best_key(unsigned long long count, uint32_t dbits) {
  return (count << kDiffBits) | (kDiffMask - dbits);
}

// raise a song's best to at least `val`; true if this call raised it.  Best only grows, so a (possibly stale) read
// that already covers the value makes the atomic unnecessary.
__device__ __forceinline__ bool best_raise(unsigned long long *best, unsigned long long val) {
  return __ldcg(best) < val && atomicMax(best, val) < val;
}

// keep the song's best (count, smallest diff) current
template <bool DENSE>
__device__ __forceinline__ void song_update(const QMeta &m, uint32_t song, uint32_t dbits, unsigned long long count,
                                            const Tables &T, int32_t *__restrict__ flags) {
  const int64_t ss = song_slot<DENSE>(m, song, T.song_key);
  if (ss < 0) { atomicOr(flags, 8); return; }
  best_raise(&T.song_best[ss], best_key(count, dbits));
}

}  // namespace tvote

// SIA_QUERY_TIMING: events between the stages of a vote, created on first use (on the current device).  mark() does
// nothing unless `on`; ms(a, b) waits for mark b.
struct StageEvents {
  bool on = false;
  cudaEvent_t ev[9] = {};
  void mark(int k, cudaStream_t s) {
    if (!on) return;
    if (!ev[k]) cudaEventCreate(&ev[k]);
    cudaEventRecord(ev[k], s);
  }
  float ms(int a, int b) {
    float t = 0;
    cudaEventSynchronize(ev[b]);
    cudaEventElapsedTime(&t, ev[a], ev[b]);
    return t;
  }
  void release() { for (auto &e : ev) if (e) { cudaEventDestroy(e); e = nullptr; } }
};

// ---- the passes of a query call (index_query.cu) -----------------------------------------------------------------
// outputs of a query call: [n_queries][topn] song / diff / count / rows, [n_queries] result counts and, a-priori only,
// batches read and exit flags
struct PvOut { int32_t *song, *diff, *count, *rows, *nres; };
struct QueryOut : PvOut { int32_t *batches, *exit; };

// one pass of up to kMaxQueriesPerPass queries [q0, q0 + nq), looked up: what its vote step gets
struct QueryPass {
  Lookup L;                                  // entries [i0, i0 + n) of the pass's pairs, sorted, with their runs
  int64_t q0 = 0, i0 = 0, n = 0;
  int nq = 0;
  const int64_t *h_qs = nullptr, *d_qs = nullptr;   // entry offsets of the pass's queries (absolute) [nq + 1]
  // scanned tuple / head-row offsets at the queries' first entries [nq + 1]; d_goff: both on the device, one after the other
  const int64_t *h_off_all = nullptr, *h_off_head = nullptr, *d_goff = nullptr;
  int64_t budget = 0;                        // vote tuples per group of queries
  cudaStream_t s = nullptr;
  size_t groups = 0;                         // set by the vote step: table-vote groups, for the SIA_QUERY_TIMING line
};

// The frame of sia_index_query_batch and sia_index_query_apriori: argument checks, zeroed outputs, then per pass the
// lookup (scratch in ix->arena, extra_bytes(nq, n) more of it left for the vote step), the tuple offsets, vote(pass)
// and the lookup / vote times (ix->last_lookup_ms, last_vote_ms; with `timing` one line per pass on stderr).  Fills
// h_stats[0] (query pairs); the vote step fills h_stats[1..3].
int query_passes(::sia_index *ix, const uint8_t *d_hash, const int32_t *d_qoff, const int64_t *h_query_starts,
                 int32_t n_queries, int32_t topn, const QueryOut &out, int64_t *h_stats, cudaStream_t s, bool timing,
                 size_t (*extra_bytes)(int nq, int64_t n), const std::function<int(QueryPass &)> &vote);

// ---- partitioned vote (index_pvote.cu) ------------------------------------------------------------------------
// The vote tuples of every query are split by a hash of the SONG into partitions small enough for an exact hash table
// in shared memory: one scatter pass (posting runs / received vote keys -> per-(query, partition) regions, staged and
// sorted by partition in shared memory so that the global writes are contiguous runs), one count pass (one CTA per
// region: bins counted in shared memory, the region's top-n songs), one merge (top-n over a query's regions: a song
// lives in exactly one partition, so the merge of per-partition top-n lists is exact).  Queries whose partitions do
// not fit (a song with > 16384 tuples, > 512 * 16384 tuples, thousands of tied bins in one partition) are flagged in d_qover and left to the table vote.
constexpr int kPvMaxTopn = 32;
constexpr int kPvMaxPeers = 16;
// scratch bytes for `tuples` vote tuples of nq queries arriving from n_src sources (worst case)
size_t pvote_bytes(int64_t tuples, int64_t nq, int n_src, int topn);
// per entry of a lookup what the scatter walk reads (once per pass): d_info[L.n] (16 B each), d_qh[L.n]
int pvote_entry_info(const Lookup &L, longlong2 *d_info, uint32_t *d_qh, cudaStream_t s);
// entries of the queries [qa, qb) of a lookup.  d_qs: entry offsets of the pass's queries (absolute, i0 = first);
// d_goff / h_goff: tuple offsets (off_all) at the queries' first entries, [nq_pass + 1].  Rows are NOT counted here.
int pvote_entries(Arena &ar, const Lookup &L, const longlong2 *d_info, const uint32_t *d_qh, const uint64_t *post, const int64_t *d_qs,
                  int64_t i0, const int64_t *d_goff, const int64_t *h_goff, int qa, int qb, int qid_base, int topn, const PvOut &out,
                  uint32_t *d_qover, uint32_t *d_qbins /* [nq_pass], zeroed: distinct bins per query */,
                  unsigned long long *d_nbins /* NULL, or += the bins of the settled queries */, cudaStream_t s,
                  StageEvents &tm /* marks 0..3 around layout, scatter, count + merge */);
// slotted vote keys, each slot sorted by query id (else d_flags2[0] is set and the outputs are garbage); rows counted from the regions.
// d_over_count: incremented once per flagged query.
// hash-prefix sharding over peer memory (index_dist.cu: sia_index_scatter_peers / sia_vote_count_regions)
int pvote_scatter_peers(Arena &ar, const Lookup &L, const longlong2 *d_einfo, const uint32_t *d_qh, const uint64_t *post,
                        const int64_t *d_q_ent, const int64_t *d_goff, int world, int rank, int qp, const int64_t *d_t_total,
                        void *const *peer_regions, void *const *peer_fill, void *const *peer_qover, int64_t region_cap,
                        int64_t fill_cap, int64_t *d_info, cudaStream_t s);
int pvote_count_regions(Arena &ar, const int64_t *d_t_total, int nq, int topn, uint64_t *d_regions, uint32_t *d_fill,
                        uint32_t *d_qover, int64_t region_cap, int64_t fill_cap, const PvOut &out, int64_t *d_info,
                        uint32_t *d_over_count, cudaStream_t s);
Arena &vote_arena(int device);
int vote_scratch_finish_and_reserve(int device, size_t bytes);
int pvote_key_slots(Arena &ar, const uint64_t *d_keys, int n_slots, int64_t cap, const int64_t *d_counts, int nq, int topn,
                    const PvOut &out, uint32_t *d_qover, uint32_t *d_flags2 /* [0] unsorted, [1] flagged queries */,
                    cudaStream_t s);

}  // namespace sia

struct sia_index {
  int device = 0;
  int64_t capacity = 0;             // postings the table can hold
  uint64_t *post = nullptr;         // [capacity]
  ulonglong2 *keys[2] = {nullptr, nullptr};   // key tables (double-buffered: a merge writes the other one)
  int64_t keys_cap[2] = {0, 0};     // entries each buffer can hold (incl. the sentinel)
  int cur = 0;
  int64_t n_rows = 0, n_keys = 0;
  uint32_t *dir = nullptr;          // [2^dir_bits + 1]
  int dir_bits = 0;
  int64_t dir_cap = 0;              // entries allocated
  ulonglong2 *pend[2] = {nullptr, nullptr};   // pending rows + the sort's alternate buffer
  int64_t pend_cap = 0, n_pending = 0;
  int32_t *status = nullptr;        // [0] device flags: 1 = song/offset out of range on insert, 2 = query offset / id out of
                                    //     range; [1] largest song id ever inserted
  int32_t max_song = 0;             // host copy of status[1], refreshed by finalize
  cudaEvent_t insert_done = nullptr;   // recorded after every insert's pack kernel (inserts may run on any stream)
  sia::Arena arena;                 // build / lookup scratch
  sia::Arena arena3;                // vote tables
  cudaEvent_t ev_q[3] = {nullptr, nullptr, nullptr};   // start / after lookup / end of a query pass
  sia::StageEvents ev_stage;        // SIA_QUERY_TIMING: between the stages of the vote
  double last_lookup_ms = 0, last_vote_ms = 0;          // device time of the last sia_index_query_batch call
  // hash-prefix sharding over peer memory: the lookup of the pass in flight (lives in `arena` until the next reserve)
  sia::Lookup dist_L;
  longlong2 *dist_einfo = nullptr;
  uint32_t *dist_qh = nullptr;
  int64_t *dist_q_ent = nullptr, *dist_goff = nullptr;
  int dist_nq = 0;
  uint64_t *stage = nullptr;        // staging chunk of the in-place posting moves
  int64_t stage_cap = 0;

  const ulonglong2 *key_table() const { return keys[cur]; }
};
