// K4, query side — the SELECT ... WHERE hash IN (...) lookup (recognizer.py:60-64, 252-259) and the vote inside
// align_matches (recognizer.py:303-310) for a batch of queries.  The default vote is the partitioned vote of
// index_pvote.cu (called from here per group of queries); this file holds the lookup, the grouping, and the TABLE vote
// described below — the path of queries the partitioned vote flags (a bin above a region's size) and of every query
// when topn is above what the partitioned vote ranks (kPvMaxTopn).
//
// query_passes is the frame of both device query calls (sia_index_query_batch here, sia_index_query_apriori in
// index_apriori.cu): argument checks, passes of up to kMaxQueriesPerPass queries, per pass the lookup and the tuple
// offsets, then the caller's vote step.  split_groups cuts a pass into groups under the tuple budget, and table_vote
// runs one attempt of the table vote over one group, for the entries of a lookup and for vote keys alike.
//
// Lookup: the (hash, offset) pairs of the queries are packed into 16-byte entries, sorted by (query, hash, offset)
// — duplicates drop out, equal hashes of one query become adjacent — and each is looked up: directory -> binary
// search in the key table -> the run [start, next start) of 8-byte postings.
//
// Vote (per group of queries, every query owning zero-initialised sub-tables):
//   pass 1  every vote tuple (query, song, db_offset - query_offset) marks a 2-bit bucket (seen / seen twice) of the
//           query's duplicate filter with one atomicOr, and the tuples that landed in a twice-hit bucket are counted
//           per query (exactly: the later arrivals + one for the bucket's first arrival);
//   layout  the bin tables are sized from those counts on the device (2 slots per candidate tuple);
//   pass 2  the tuples of twice-hit buckets — every bin of count >= 2 is among them — are counted in the bin table
//           (open addressing, one 64-bit key word + a 32-bit count per slot) and keep the song's best
//           (count << 25 | inverted diff: largest count, smallest difference on ties — Python's max() keeps the first
//           maximum, recognizer.py:308) current with atomicMax; all other tuples are bins of count 1 and touch nothing;
//   top-n   one block per query scans its song table: (count desc, song asc) — the stable sort of recognizer.py:307-310;
//   singles a query whose n-th result has a count below 2 (or that has fewer than n results) needs the count-1 bins
//           too: its tuples are voted again as (1, diff) and its top-n is redone (rare on a large index, the normal
//           case on a tiny one);
//   rows    dedup_hashes[song] (recognizer.py:259-264: DB rows matched, once per row) is counted for the winners only,
//           in a last pass over the head postings.
// The same passes run over vote keys that arrived from other shards (vote_key_slots, hash-prefix sharding).
#include "index.cuh"

#include <chrono>
#include <type_traits>

using namespace sia;
using namespace sia::tvote;

namespace {

constexpr int kVoteTuples = 4096;         // vote tuples per block of the entry-walking kernels (512 per warp): the tuples
                                          // in flight on the whole GPU then belong to 2-3 queries, whose filters stay in L2

// ---- lookup ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
pack_queries_kernel(const uint8_t *__restrict__ hash, const int32_t *__restrict__ qoff, const int32_t *__restrict__ qid_arr,
                    const int64_t *__restrict__ query_starts, int n_queries, int64_t i0, int64_t n,
                    ulonglong2 *__restrict__ out, int32_t *__restrict__ status) {
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = i0 + k;
    uint64_t hi; uint32_t lo16;
    load_digest(hash + i * SIA_HASH_BYTES, hi, lo16);
    const int32_t q = qid_arr ? qid_arr[i] : find_segment(query_starts, n_queries, i);
    const int32_t o = qoff[i];
    if (o < 0 || o > (int32_t)kM24 || q < 0 || q >= (1 << 24)) atomicOr(status, 2);
    out[k] = make_entry((uint32_t)q, hi, lo16, (uint32_t)o);
  }
}

// Per-query sort of the packed entries in shared memory (the entries of a pass arrive grouped by query, and all entries
// of a query share the query id in the top bits, so sorting each query's slice by the whole 128 bits gives the
// (query, hash, offset) order of a global sort).  One CTA per query, bitonic network on 16-byte keys, slices of up to
// kSmemSortMax entries (64 KB); a pass with a longer query takes the global LSD radix sort.
constexpr int kSmemSortMax = 4096;
constexpr int kSmemSortThreads = 512;

__global__ void __launch_bounds__(kSmemSortThreads)
sort_queries_kernel(ulonglong2 *__restrict__ ent, const int64_t *__restrict__ query_starts, int64_t i0) {
  extern __shared__ __align__(16) unsigned char sort_smem[];
  ulonglong2 *key = reinterpret_cast<ulonglong2 *>(sort_smem);
  const int64_t s0 = query_starts[blockIdx.x] - i0;
  const int n = (int)(query_starts[blockIdx.x + 1] - i0 - s0);
  if (n < 2) return;
  int P = 2;
  while (P < n) P <<= 1;
  for (int i = threadIdx.x; i < P; i += kSmemSortThreads) key[i] = i < n ? ent[s0 + i] : make_ulonglong2(~0ull, ~0ull);
  __syncthreads();
  for (int k = 2; k <= P; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < (P >> 1); t += kSmemSortThreads) {
        const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));      // the lower index of the t-th pair at distance j
        const int l = i | j;
        const ulonglong2 a = key[i], b = key[l];
        const bool up = (i & k) == 0;
        if (rec_less(b, a) == up) { key[i] = b; key[l] = a; }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < n; i += kSmemSortThreads) ent[s0 + i] = key[i];
}

// entry -> posting run.  An all-ones entry is padding (sorts last, matches nothing).
__global__ void __launch_bounds__(256)
lookup_kernel(const ulonglong2 *__restrict__ ent, int64_t n, const ulonglong2 *__restrict__ keys, int64_t n_keys,
              const uint32_t *__restrict__ dir, int bits, int64_t *__restrict__ first, uint32_t *__restrict__ cnt_all,
              uint32_t *__restrict__ cnt_head, int32_t *__restrict__ status) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const ulonglong2 e = ent[i];
    bool dup = (e.x & e.y) == ~0ull, head = true;
    if (i > 0) {
      const ulonglong2 p = ent[i - 1];
      dup = dup || rec_eq(e, p);
      head = !(p.y == e.y && (p.x >> 24) == (e.x >> 24));   // same (qid, digest) as the previous entry?
    }
    int64_t f = 0;
    uint32_t c = 0;
    if (!dup && n_keys > 0) {
      uint64_t khi; uint32_t klo16, qid, qoff;
      entry_key(e, khi, klo16, qid, qoff);
      const int64_t ki = hash_lower_bound_dir(keys, dir, bits, khi, klo16);
      const ulonglong2 k = keys[ki];
      if (ki < n_keys && k.y == khi && (uint32_t)(k.x >> 48) == klo16) {
        f = (int64_t)(k.x & kM48);
        const int64_t len = (int64_t)(keys[ki + 1].x & kM48) - f;
        if (len > 0xffffffffll) atomicOr(status, 4);          // a run of 2^32 postings: not representable
        c = (uint32_t)len;
      }
    }
    first[i] = f;
    cnt_all[i] = c;
    cnt_head[i] = head ? c : 0u;
  }
}

__global__ void __launch_bounds__(256)
select_rows_kernel(const ulonglong2 *__restrict__ ent, int64_t n, const int64_t *__restrict__ first,
                   const int64_t *__restrict__ off, const uint64_t *__restrict__ post, int32_t *__restrict__ o_idx,
                   int32_t *__restrict__ o_song, int32_t *__restrict__ o_off, int64_t cap) {
  // entries here are packed with qoff = position of the hash in the caller's list
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = off[i], c = off[i + 1] - b;
    for (int64_t k = 0; k < c; ++k) {
      if (b + k >= cap) break;
      const uint64_t r = post[first[i] + k];
      o_idx[b + k] = (int32_t)(ent[i].x & kM24);
      o_song[b + k] = (int32_t)((r >> 24) & kM24);
      o_off[b + k] = (int32_t)(r & kM24);
    }
  }
}

__global__ void gather_offsets_kernel(const int64_t *__restrict__ off_all, const int64_t *__restrict__ off_head,
                                      const int64_t *__restrict__ query_starts, int64_t i0, int nq,
                                      int64_t *__restrict__ out) {
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q <= nq; q += gridDim.x * blockDim.x) {
    const int64_t e = query_starts[q] - i0;
    out[q] = off_all[e];
    out[nq + 1 + q] = off_head[e];
  }
}

// duplicate filter: 2 bits per bucket (seen, seen twice), 16 buckets per 32-bit word, ~16 buckets per tuple
__device__ __forceinline__ uint32_t *filter_word(const QMeta &m, uint32_t song, uint32_t dbits, uint32_t *__restrict__ filter,
                                                 uint32_t &seen_bit) {
  const uint32_t h = mix32(song * 0x85ebca6bu ^ (dbits * 0xc2b2ae35u + 0x27d4eb2fu));
  seen_bit = 1u << (2 * (h & 15u));
  return filter + m.filt_base + slot_of(h, m.filt_words);
}

// pass 1 of one tuple, second half: `old` is what the atomicOr of the bucket's seen bit returned; returns how many
// candidate tuples this arrival accounts for
__device__ __forceinline__ uint32_t mark_finish(uint32_t *__restrict__ w, uint32_t seen, uint32_t old) {
  if (!(old & seen)) return 0;                      // first arrival in its bucket
  if (old & (seen << 1)) return 1;                  // a later arrival of a bucket already known to be hit twice
  return (atomicOr(w, seen << 1) & (seen << 1)) ? 1u : 2u;   // the arrival that marks "twice" also accounts for the first one
}

enum { PASS_MARK = 1, PASS_VOTE = 2, PASS_SINGLES = 3, PASS_ROWS = 4 };

constexpr int kCandBuf = 320;             // candidate keys a warp buffers in shared memory before it flushes them

// write a warp's buffered candidate keys (all of query q) to q's candidate list: one atomic per flush
__device__ __forceinline__ void cand_flush(unsigned long long *__restrict__ buf, int &n, uint32_t q, QMeta *__restrict__ meta,
                                           unsigned long long *__restrict__ cand, int lane, int32_t *__restrict__ flags) {
  if (n == 0) return;                                // warp-uniform
  __syncwarp();
  unsigned long long base = 0;
  if (lane == 0) {
    const uint32_t at = atomicAdd(&meta[q].cursor, (uint32_t)n);
    if (at + (uint32_t)n > meta[q].cand) { atomicOr(flags, 8); base = ~0ull; }     // cannot happen: pass 1 counted them
    else base = (unsigned long long)meta[q].cand_base + at;
  }
  base = __shfl_sync(0xffffffffu, base, 0);
  if (base != ~0ull)
    for (int i = lane; i < n; i += 32) cand[base + i] = buf[i];
  __syncwarp();
  n = 0;
}

// append the candidates among (a, b) of every lane to the warp's buffer (lane order)
__device__ __forceinline__ void cand_push(unsigned long long *__restrict__ buf, int &n, bool ca, unsigned long long ka, bool cb,
                                          unsigned long long kb, int lane) {
  const uint32_t ma = __ballot_sync(0xffffffffu, ca), mb = __ballot_sync(0xffffffffu, cb);
  const uint32_t lt = (1u << lane) - 1u;
  if (ca) buf[n + __popc(ma & lt)] = ka;
  if (cb) buf[n + __popc(ma) + __popc(mb & lt)] = kb;
  n += __popc(ma) + __popc(mb);
}

// Two vote tuples per lane and step, so that the two L2 round trips (the atomicOr of pass 1, the filter read of
// pass 2) of a step are in flight together.  PASS_MARK: acc += candidate tuples accounted for.  PASS_VOTE: tuples alone
// in their bucket are bins of count 1 (acc += 1 each, nothing else to do); the others — every bin of count >= 2 is among
// them — are only COLLECTED here (ca / cb), and voted by cand_vote_kernel with all lanes busy.
template <bool DENSE, int PASS>
__device__ __forceinline__ void tuple_pair_pass(const QMeta &m, bool va, uint32_t song_a, uint32_t db_a, bool vb, uint32_t song_b,
                                                uint32_t db_b, const Tables &T, uint32_t &acc, bool &ca, bool &cb,
                                                int32_t *__restrict__ flags) {
  ca = cb = false;
  if (PASS == PASS_SINGLES) {
    if (va) song_update<DENSE>(m, song_a, db_a, 1ull, T, flags);
    if (vb) song_update<DENSE>(m, song_b, db_b, 1ull, T, flags);
    return;
  }
  uint32_t sa, sb;
  uint32_t *wa = filter_word(m, song_a, db_a, T.filter, sa);
  uint32_t *wb = filter_word(m, song_b, db_b, T.filter, sb);
  if (PASS == PASS_MARK) {
    const uint32_t oa = va ? atomicOr(wa, sa) : 0u;
    const uint32_t ob = vb ? atomicOr(wb, sb) : 0u;
    if (va) acc += mark_finish(wa, sa, oa);
    if (vb) acc += mark_finish(wb, sb, ob);
  } else {
    const uint32_t fa = va ? __ldcg(wa) : 0u;
    const uint32_t fb = vb ? __ldcg(wb) : 0u;
    ca = va && (fa & (sa << 1));
    cb = vb && (fb & (sb << 1));
    acc += (uint32_t)(va && !ca) + (uint32_t)(vb && !cb);
  }
}

// a warp's step left query cur_q: PASS_MARK adds the warp's candidate count to cur_q's, PASS_VOTE writes the buffered
// candidates to cur_q's list (the buffer holds one query's candidates)
template <int PASS>
__device__ __forceinline__ void leave_query(uint32_t cur_q, uint32_t &acc, unsigned long long *__restrict__ cbuf, int &ncand,
                                            QMeta *__restrict__ meta, const Tables &T, int lane, int32_t *__restrict__ flags) {
  if (PASS == PASS_MARK) {
#pragma unroll
    for (int d = 16; d; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    if (lane == 0 && acc) atomicAdd(&meta[cur_q].cand, acc);
    acc = 0;
  }
  if (PASS == PASS_VOTE) cand_flush(cbuf, ncand, cur_q, meta, T.cand, lane, flags);
}

__device__ __forceinline__ unsigned long long cand_key(uint32_t q, uint32_t song, uint32_t dbits) {
  return ((unsigned long long)q << (kSongBits + kDiffBits)) | ((unsigned long long)song << kDiffBits) | dbits;
}

// Pass 2b: the collected candidates, densely — bin table (CAS the key word, bump the count) and the song's best; two
// keys per thread so that their L2 round trips overlap.
template <bool DENSE>
__global__ void __launch_bounds__(256)
cand_vote_kernel(const unsigned long long *__restrict__ cand, const QMeta *__restrict__ meta, int q_lo, int q_hi, Tables T,
                 unsigned long long *__restrict__ n_bins, int32_t *__restrict__ flags) {
  if (*flags & 32) return;
  const int64_t lo = meta[q_lo].cand_base, total = meta[q_hi - 1].cand_base + meta[q_hi - 1].cand - lo;
  uint32_t fresh = 0;
  const uint32_t qmask = (1u << kQidBits) - 1u;
  for (int64_t i0 = (int64_t)blockIdx.x * 512; i0 < total; i0 += (int64_t)gridDim.x * 512) {
    __syncwarp();
    const int64_t ia = i0 + threadIdx.x, ib = ia + 256;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const int64_t i = half ? ib : ia;
      if (i >= total) continue;
      const unsigned long long k = cand[lo + i];
      const QMeta m = meta[(uint32_t)(k >> (kSongBits + kDiffBits)) & qmask];
      const uint32_t song = (uint32_t)(k >> kDiffBits) & 0xffffffu, dbits = (uint32_t)(k & kDiffMask);
      const unsigned long long c = bin_count(m, song, dbits, T, fresh, flags);
      if (c) song_update<DENSE>(m, song, dbits, c, T, flags);
    }
  }
  if (n_bins) {
#pragma unroll
    for (int d = 16; d; d >>= 1) fresh += __shfl_xor_sync(0xffffffffu, fresh, d);
    if ((threadIdx.x & 31) == 0 && fresh) atomicAdd(n_bins, (unsigned long long)fresh);
  }
}

// winners' rows: lanes whose posting belongs to winner r add up inside the warp, one atomic per warp and winner
__device__ __forceinline__ void rows_pass(uint32_t active, bool mine, uint32_t song, const int32_t *__restrict__ win, int nwin,
                                          int32_t *__restrict__ out_rows, int lane) {
  for (int r = 0; r < nwin; ++r) {
    const uint32_t hit = __ballot_sync(active, mine && song == (uint32_t)win[r]);
    if (hit && lane == (__ffs(active) - 1)) atomicAdd(out_rows + r, __popc(hit));
  }
}

// One block handles kVoteTuples consecutive vote tuples (postings of the entries [e0, e0+n), numbered by the exclusive
// scan off[]), whatever entries they belong to: a heavy key's run is shared by many blocks.  Each warp takes an eighth
// of the block's tuples and walks the entries they belong to: everything that depends on the entry (query tables,
// query offset, first posting) is warp-uniform and loaded once per entry, the lanes then take the entry's
// postings 64 at a time (two per lane), the next step's postings in flight during this one.
// entry in which every warp's piece of kVoteTuples / 8 tuples starts (relative to e0): computed once per group, read by
// all passes instead of a 24-step binary search at the start of every warp of every pass
__global__ void __launch_bounds__(256)
piece_entries_kernel(const int64_t *__restrict__ off, int64_t e0, int64_t n, int64_t n_pieces, uint32_t *__restrict__ piece_ent) {
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n_pieces; p += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = off[e0] + p * (kVoteTuples >> 3);
    int64_t ei = e0, hi = e0 + n;            // largest entry in [e0, e0+n) with off[ei] <= j
    while (hi - ei > 1) { const int64_t mid = ei + ((hi - ei) >> 1); if (off[mid] <= j) ei = mid; else hi = mid; }
    piece_ent[p] = (uint32_t)(ei - e0);
  }
}

template <bool DENSE, int PASS>
__global__ void __launch_bounds__(256)
entries_pass_kernel(const ulonglong2 *__restrict__ ent, int64_t e0, int64_t n, const int64_t *__restrict__ first,
                    const int64_t *__restrict__ off, const uint32_t *__restrict__ piece_ent,
                    const uint64_t *__restrict__ post, QMeta *__restrict__ meta, Tables T,
                    const uint32_t *__restrict__ qflag, const int32_t *__restrict__ n_flagged,
                    unsigned long long *__restrict__ n_bins, int32_t *__restrict__ flags) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int per_warp = kVoteTuples >> 3;
  if (PASS == PASS_VOTE && (*flags & 32)) return;    // the bin tables did not fit their reservation: the host redoes the group
  if (PASS == PASS_SINGLES && *n_flagged == 0) return;            // every query was settled by its bins of count >= 2
  const int64_t j_lo = off[e0] + (int64_t)blockIdx.x * kVoteTuples + (int64_t)warp * per_warp;
  const int64_t j_hi = min(off[e0 + n], j_lo + per_warp);
  if (j_lo >= j_hi) return;
  uint32_t acc = 0;                        // PASS_MARK: candidate tuples of the current query; PASS_VOTE: bins of count 1
  uint32_t cur_q = 0xffffffffu;
  __shared__ unsigned long long s_cand[PASS == PASS_VOTE ? 8 * kCandBuf : 1];
  unsigned long long *cbuf = s_cand + (PASS == PASS_VOTE ? warp * kCandBuf : 0);
  int ncand = 0;                           // PASS_VOTE: candidate keys of query cur_q waiting in cbuf (warp-uniform)
  int64_t ei = e0 + piece_ent[(int64_t)blockIdx.x * 8 + warp];    // the entry this warp's first tuple belongs to
  for (; ei < e0 + n; ++ei) {
    const int64_t o_this = off[ei], o_next = off[ei + 1];
    if (o_this >= j_hi) break;
    if (o_next == o_this) continue;                              // a hash without postings (or a duplicate pair)
    const ulonglong2 e = ent[ei];
    const uint32_t q = (uint32_t)(e.y >> 40);
    if (PASS == PASS_SINGLES && !qflag[q]) continue;
    if ((PASS == PASS_MARK || PASS == PASS_VOTE) && q != cur_q) {
      leave_query<PASS>(cur_q, acc, cbuf, ncand, meta, T, lane, flags);
      cur_q = q;
    }
    const QMeta m = meta[q];
    const uint32_t qoff = (uint32_t)(e.x & kM24);
    const uint64_t *__restrict__ run = post + first[ei];
    const uint32_t k_hi = (uint32_t)(min(j_hi, o_next) - o_this);
    const uint32_t k_lo = (uint32_t)(max(j_lo, o_this) - o_this);
    uint64_t na = 0, nb = 0;                                     // streaming loads: the postings pass through, the filters
    if (k_lo + lane < k_hi) na = __ldcs(run + k_lo + lane);      // and tables are what should stay in L2
    if (k_lo + 32 + lane < k_hi) nb = __ldcs(run + k_lo + 32 + lane);
    for (uint32_t kw = k_lo; kw < k_hi; kw += 64) {
      __syncwarp();                                              // the probe loops below diverge
      const uint32_t ka = kw + lane, kb = ka + 32;
      const uint64_t ra = na, rb = nb;
      if (ka + 64 < k_hi) na = __ldcs(run + ka + 64);
      if (kb + 64 < k_hi) nb = __ldcs(run + kb + 64);
      // db offset - query offset, biased
      const uint32_t song_a = (uint32_t)(ra >> 24) & 0xffffffu, db_a = (uint32_t)(ra & kM24) - qoff + SIA_DIFF_BIAS;
      const uint32_t song_b = (uint32_t)(rb >> 24) & 0xffffffu, db_b = (uint32_t)(rb & kM24) - qoff + SIA_DIFF_BIAS;
      bool ca, cb;
      tuple_pair_pass<DENSE, PASS>(m, ka < k_hi, song_a, db_a, kb < k_hi, song_b, db_b, T, acc, ca, cb, flags);
      if (PASS == PASS_VOTE) {
        if (ncand > kCandBuf - 64) cand_flush(cbuf, ncand, q, meta, T.cand, lane, flags);
        cand_push(cbuf, ncand, ca, cand_key(q, song_a, db_a), cb, cand_key(q, song_b, db_b), lane);
      }
    }
    __syncwarp();
  }
  leave_query<PASS>(cur_q, acc, cbuf, ncand, meta, T, lane, flags);
  if (PASS == PASS_VOTE && n_bins) {                             // this warp's bins of count 1
#pragma unroll
    for (int d = 16; d; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    if (lane == 0 && acc) atomicAdd(n_bins, (unsigned long long)acc);
  }
}

// dedup_hashes of the winners (recognizer.py:259-264): one warp per head entry.  A run is sorted by (song, offset), so a
// long run is not read at all: two binary searches per winner bracket its rows (lanes 2r, 2r+1); short runs are read.
__global__ void __launch_bounds__(256)
entries_rows_kernel(const ulonglong2 *__restrict__ ent, int64_t e0, int64_t n, const int64_t *__restrict__ first,
                    const uint32_t *__restrict__ cnt_head, const uint64_t *__restrict__ post, int qid_base, int topn,
                    const int32_t *__restrict__ out_song, const int32_t *__restrict__ out_nres, int32_t *__restrict__ out_rows) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n; i += warps) {
    const int64_t ei = e0 + i;
    const uint32_t c = cnt_head[ei];                              // 0: not the first entry of its (query, hash), or no postings
    if (c == 0) continue;
    const uint32_t q = (uint32_t)(ent[ei].y >> 40);
    const int nwin = out_nres[q + qid_base];
    if (nwin == 0) continue;
    const int64_t obase = ((int64_t)q + qid_base) * topn;
    const uint64_t *__restrict__ run = post + first[ei];
    if (c <= 64) {
      for (uint32_t kw = 0; kw < c; kw += 32) {
        const uint32_t k = kw + lane;
        const uint32_t song = k < c ? (uint32_t)(run[k] >> 24) & 0xffffffu : 0xffffffffu;
        rows_pass(0xffffffffu, k < c, song, out_song + obase, nwin, out_rows + obase, lane);
      }
    } else {
      for (int r0 = 0; r0 < nwin; r0 += 16) {
        const int r = r0 + (lane >> 1);
        int64_t pos = 0;
        if (r < nwin) pos = lower_bound_u64(run, 0, (int64_t)c, ((uint64_t)(uint32_t)out_song[obase + r] + (lane & 1)) << 24);
        const int64_t lo = __shfl_sync(0xffffffffu, pos, lane & ~1), hi = __shfl_sync(0xffffffffu, pos, lane | 1);
        if (!(lane & 1) && r < nwin && hi > lo) atomicAdd(out_rows + obase + r, (int32_t)(hi - lo));
      }
    }
  }
}

// The same passes over vote keys stored in slots (keys from other shards, or a caller's tuples): blockIdx.y = slot, every
// warp takes pieces of 512 consecutive keys of the slot, two keys per lane and step.  Keys of one query are adjacent
// (the shards emit them in query order), so a step normally belongs to one query; the few steps that straddle queries
// are handled one query after the other.
template <bool DENSE, int PASS>
__global__ void __launch_bounds__(256)
keys_pass_kernel(const uint64_t *__restrict__ keys, int64_t cap, const int64_t *__restrict__ counts, int nq,
                 QMeta *__restrict__ meta, Tables T, const uint32_t *__restrict__ qflag, const int32_t *__restrict__ n_flagged,
                 const uint32_t *__restrict__ qsel, int topn, const int32_t *__restrict__ out_song, const int32_t *__restrict__ out_nres,
                 int32_t *__restrict__ out_rows, int32_t *__restrict__ flags) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (PASS == PASS_VOTE && (*flags & 32)) return;
  if (PASS == PASS_SINGLES && *n_flagged == 0) return;
  int64_t n;
  const uint64_t *__restrict__ kk = slot_keys(keys, cap, counts, blockIdx.y, n);
  const uint32_t qmask = (1u << kQidBits) - 1u;
  __shared__ unsigned long long s_cand[PASS == PASS_VOTE ? 8 * kCandBuf : 1];
  unsigned long long *cbuf = s_cand + (PASS == PASS_VOTE ? warp * kCandBuf : 0);
  const int64_t n_pieces = (n + 511) >> 9;
  for (int64_t piece = (int64_t)blockIdx.x * 8 + warp; piece < n_pieces; piece += (int64_t)gridDim.x * 8) {
    const int64_t i_lo = piece << 9, i_hi = min(n, i_lo + 512);
    uint32_t cur_q = 0xffffffffu, acc = 0;
    int ncand = 0;
    for (int64_t i0 = i_lo; i0 < i_hi; i0 += 64) {
      __syncwarp();
      const int64_t ia = i0 + lane, ib = ia + 32;
      bool va = ia < i_hi, vb = ib < i_hi;
      const uint64_t ka = va ? __ldcs(kk + ia) : 0, kb = vb ? __ldcs(kk + ib) : 0;
      const uint32_t qa = (uint32_t)(ka >> (kSongBits + kDiffBits)) & qmask, qb = (uint32_t)(kb >> (kSongBits + kDiffBits)) & qmask;
      if (va && qa >= (uint32_t)nq) { atomicOr(flags, 2); va = false; }
      if (vb && qb >= (uint32_t)nq) { atomicOr(flags, 2); vb = false; }
      const uint32_t song_a = (uint32_t)(ka >> kDiffBits) & 0xffffffu, song_b = (uint32_t)(kb >> kDiffBits) & 0xffffffu;
      const uint32_t db_a = (uint32_t)(ka & kDiffMask), db_b = (uint32_t)(kb & kDiffMask);
      if (PASS == PASS_ROWS) { va = va && (ka >> 63); vb = vb && (kb >> 63); }      // head keys count as matched rows
      uint32_t todo_a = __ballot_sync(0xffffffffu, va), todo_b = __ballot_sync(0xffffffffu, vb);
      while (todo_a | todo_b) {                          // one iteration per query present in the step (normally one)
        const uint32_t qq = todo_a ? __shfl_sync(0xffffffffu, qa, __ffs(todo_a) - 1) : __shfl_sync(0xffffffffu, qb, __ffs(todo_b) - 1);
        const bool ma = va && qa == qq, mb = vb && qb == qq;
        todo_a &= ~__ballot_sync(0xffffffffu, ma);
        todo_b &= ~__ballot_sync(0xffffffffu, mb);
        if (qsel && !qsel[qq]) continue;                 // only the queries the partitioned vote left over
        if (PASS == PASS_ROWS) {
          const int64_t obase = (int64_t)qq * topn;
          const int nwin = out_nres[qq];
          rows_pass(0xffffffffu, ma, song_a, out_song + obase, nwin, out_rows + obase, lane);
          rows_pass(0xffffffffu, mb, song_b, out_song + obase, nwin, out_rows + obase, lane);
          continue;
        }
        if (PASS == PASS_SINGLES && !qflag[qq]) continue;
        if (qq != cur_q) {
          leave_query<PASS>(cur_q, acc, cbuf, ncand, meta, T, lane, flags);
          cur_q = qq;
        }
        const QMeta m = meta[qq];
        bool ca, cb;
        tuple_pair_pass<DENSE, PASS>(m, ma, song_a, db_a, mb, song_b, db_b, T, acc, ca, cb, flags);
        if (PASS == PASS_VOTE) {
          if (ncand > kCandBuf - 64) cand_flush(cbuf, ncand, qq, meta, T.cand, lane, flags);
          cand_push(cbuf, ncand, ca, cand_key(qq, song_a, db_a), cb, cand_key(qq, song_b, db_b), lane);
        }
        __syncwarp();
      }
    }
    leave_query<PASS>(cur_q, acc, cbuf, ncand, meta, T, lane, flags);
  }
}

// keys per query (keys arrive grouped by query: one atomic per run inside the warp)
__global__ void __launch_bounds__(256)
count_keys_kernel(const uint64_t *__restrict__ keys, int64_t cap, const int64_t *__restrict__ counts, int nq,
                  const uint32_t *__restrict__ qsel, uint32_t *__restrict__ cnt, int32_t *__restrict__ flags) {
  int64_t n;
  const uint64_t *__restrict__ kk = slot_keys(keys, cap, counts, blockIdx.y, n);
  for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x; i0 < n; i0 += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = i0 + threadIdx.x;
    bool valid = i < n;
    const uint64_t k = valid ? kk[i] : 0;
    const uint32_t q = (uint32_t)(k >> (kSongBits + kDiffBits)) & ((1u << kQidBits) - 1u);
    if (valid && q >= (uint32_t)nq) { atomicOr(flags, 2); valid = false; }
    if (valid && qsel && !qsel[q]) valid = false;
    const uint32_t active = __ballot_sync(0xffffffffu, valid);
    if (valid) {
      const uint32_t peers = __match_any_sync(active, q);
      if ((peers & ((1u << (threadIdx.x & 31)) - 1u)) == 0) atomicAdd(&cnt[q], (uint32_t)__popc(peers));
    }
  }
}

// single block: table layout of the keys path from the per-query key counts (filter, songs), cand zeroed
__global__ void __launch_bounds__(1024)
layout_keys_kernel(const uint32_t *__restrict__ cnt, int nq, int64_t dense_span, const uint32_t *__restrict__ qsel,
                   QMeta *__restrict__ meta) {
  __shared__ int64_t s_f[1024], s_s[1024];
  const int per = (nq + 1023) / 1024;
  const int a = min(nq, (int)threadIdx.x * per), b = min(nq, a + per);
  int64_t sf = 0, ss = 0;
  for (int q = a; q < b; ++q) {
    sf += (int64_t)cnt[q] + 1;
    ss += (qsel && !qsel[q]) ? 0 : dense_span > 0 ? dense_span : 2 * (int64_t)cnt[q] + 32;
  }
  s_f[threadIdx.x] = sf; s_s[threadIdx.x] = ss;
  __syncthreads();
  if (threadIdx.x == 0) {
    int64_t rf = 0, rs = 0;
    for (int i = 0; i < 1024; ++i) { const int64_t x = s_f[i], y = s_s[i]; s_f[i] = rf; s_s[i] = rs; rf += x; rs += y; }
  }
  __syncthreads();
  sf = s_f[threadIdx.x]; ss = s_s[threadIdx.x];
  for (int q = a; q < b; ++q) {
    QMeta m;
    m.bin_base = 0; m.bin_cap = 0; m.cand = 0; m.cand_base = 0; m.cursor = 0; m.pad_ = 0;
    m.filt_base = sf; m.filt_words = cnt[q] + 1u;
    m.song_base = ss; m.song_cap = (qsel && !qsel[q]) ? 0u : dense_span > 0 ? (uint32_t)dense_span : 2u * cnt[q] + 32u;
    meta[q] = m;
    sf += m.filt_words; ss += m.song_cap;
  }
}

// single block: bin tables from the candidate counts of pass 1 (2 slots per candidate tuple); *total = slots in use
__global__ void __launch_bounds__(1024)
layout_bins_kernel(QMeta *__restrict__ meta, int q_lo, int q_hi, int64_t *__restrict__ total) {
  __shared__ int64_t s_b[1024];
  const int nq = q_hi - q_lo;
  const int per = (nq + 1023) / 1024;
  const int a = q_lo + min(nq, (int)threadIdx.x * per), b = min(q_hi, a + per);
  int64_t sb = 0;
  for (int q = a; q < b; ++q) sb += 2 * (int64_t)meta[q].cand + 32;
  s_b[threadIdx.x] = sb;
  __syncthreads();
  if (threadIdx.x == 0) {
    int64_t rb = 0;
    for (int i = 0; i < 1024; ++i) { const int64_t x = s_b[i]; s_b[i] = rb; rb += x; }
    *total = rb;
  }
  __syncthreads();
  sb = s_b[threadIdx.x];
  for (int q = a; q < b; ++q) {
    meta[q].bin_base = sb;
    // the candidate lists follow the same scan: slots before this query = 2 * candidates + 32 per query
    meta[q].cand_base = (sb - 32ll * (q - q_lo)) >> 1;
    meta[q].cursor = 0;
    const int64_t c = 2 * (int64_t)meta[q].cand + 32;
    meta[q].bin_cap = (uint32_t)c;
    sb += c;
  }
}

// zero the bin tables actually in use (the size is only known on the device)
__global__ void __launch_bounds__(256)
zero_bins_kernel(unsigned long long *__restrict__ bins, uint32_t *__restrict__ bin_cnt, const int64_t *__restrict__ total,
                 int64_t cap, int32_t *__restrict__ flags) {
  int64_t n = *total;
  if (n > cap) { if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(flags, 32); n = cap; }
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    bins[i] = 0ull; bin_cnt[i] = 0u;
  }
}

// one block per query: top-n songs by (count desc, song asc), kTopK results per scan of the query's song table.
// Sets qflag[q] = 1 when the n-th result is not settled by the bins of count >= 2 (singles pass needed); with
// ONLY_FLAGGED the kernel redoes just those queries.
template <bool DENSE, bool ONLY_FLAGGED>
__global__ void __launch_bounds__(256)
topn_kernel(const Tables T, const QMeta *__restrict__ meta, int q_lo, int qid_base, int topn, uint32_t *__restrict__ qflag,
            int32_t *__restrict__ n_flagged, const uint32_t *__restrict__ qsel, int32_t *__restrict__ out_song, int32_t *__restrict__ out_diff, int32_t *__restrict__ out_count,
            int32_t *__restrict__ out_rows, int32_t *__restrict__ out_nres) {
  __shared__ unsigned long long s_key[8];
  __shared__ uint32_t s_slot[8];
  __shared__ unsigned long long s_win;
  const int q = (int)blockIdx.x + q_lo;
  if (ONLY_FLAGGED && (*n_flagged == 0 || !qflag[q])) return;
  if (qsel && !qsel[q]) return;           // the partitioned vote settled this query
  const QMeta m = meta[q];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long prev = ~0ull;
  int nres = 0;
  unsigned long long last_count = 0;
  while (nres < topn) {
    // rank key: count (high) then inverted song id, so equal counts order by ascending song id
    unsigned long long tk[kTopK];
    uint32_t ts[kTopK];
#pragma unroll
    for (int i = 0; i < kTopK; ++i) { tk[i] = 0; ts[i] = 0; }
    for (uint32_t s = threadIdx.x; s < m.song_cap; s += 256) {
      const unsigned long long best = T.song_best[m.song_base + s];
      if (best == 0ull) continue;          // empty slot / song without a match
      const uint32_t song = DENSE ? s : T.song_key[m.song_base + s] - 1u;
      unsigned long long k = ((best >> kDiffBits) << kSongBits) | (kM24 - song);
      if (k >= prev || k <= tk[kTopK - 1]) continue;
      uint32_t sl = s;
#pragma unroll
      for (int i = 0; i < kTopK; ++i)
        if (k > tk[i]) { const unsigned long long a = tk[i]; const uint32_t b = ts[i]; tk[i] = k; ts[i] = sl; k = a; sl = b; }
    }
    int got = 0;
    for (int r = 0; r < kTopK && nres < topn; ++r) {
      unsigned long long bk = tk[0];
      uint32_t bs = ts[0];
#pragma unroll
      for (int d = 16; d; d >>= 1) {
        const unsigned long long ok = __shfl_xor_sync(0xffffffffu, bk, d);
        const uint32_t os = __shfl_xor_sync(0xffffffffu, bs, d);
        if (ok > bk) { bk = ok; bs = os; }
      }
      if (lane == 0) { s_key[warp] = bk; s_slot[warp] = bs; }
      __syncthreads();
      if (threadIdx.x == 0) {
        unsigned long long w = 0; uint32_t ws = 0;
        for (int i = 0; i < 8; ++i) if (s_key[i] > w) { w = s_key[i]; ws = s_slot[i]; }
        s_win = w;
        if (w) {
          const unsigned long long v = T.song_best[m.song_base + ws];
          const int64_t o = ((int64_t)q + qid_base) * topn + nres;
          out_song[o] = (int32_t)(kM24 - (w & kM24));
          out_count[o] = (int32_t)(v >> kDiffBits);
          out_diff[o] = (int32_t)(kDiffMask - (v & kDiffMask)) - SIA_DIFF_BIAS;
          out_rows[o] = 0;
        }
      }
      __syncthreads();
      const unsigned long long w = s_win;
      if (w == 0) break;
      if (tk[0] == w) {                   // the winner leaves its owner's list
#pragma unroll
        for (int i = 0; i + 1 < kTopK; ++i) { tk[i] = tk[i + 1]; ts[i] = ts[i + 1]; }
        tk[kTopK - 1] = 0;
      }
      prev = w;
      last_count = w >> kSongBits;
      ++nres; ++got;
      __syncthreads();
    }
    if (got < kTopK) break;               // the table is exhausted
  }
  if (threadIdx.x == 0) {
    out_nres[q + qid_base] = nres;
    for (int r = nres; r < topn; ++r) {       // unused slots read as zero whatever ran before
      const int64_t o = ((int64_t)q + qid_base) * topn + r;
      out_song[o] = 0; out_diff[o] = 0; out_count[o] = 0; out_rows[o] = 0;
    }
    if (!ONLY_FLAGGED) {
      const bool f = m.filt_words > 1 && (nres < topn || last_count < 2);    // a query without tuples has nothing to add
      qflag[q] = f ? 1u : 0u;
      if (f) atomicAdd(n_flagged, 1);
    }
  }
}

int set_device(const sia_index *ix) {
  SIA_CUDA(cudaSetDevice(ix->device));
  return SIA_OK;
}

// read-and-clear of selected status flags (other flags stay)
__global__ void clear_flags_kernel(int32_t *status, int mask) { atomicAnd(status, ~mask); }

int check_status(sia_index *ix, cudaStream_t s, int mask, const char *msg) {
  int32_t st = 0;
  SIA_CUDA(cudaMemcpyAsync(&st, ix->status, sizeof st, cudaMemcpyDeviceToHost, s));
  SIA_CUDA(cudaStreamSynchronize(s));
  if (st & mask) {
    clear_flags_kernel<<<1, 1, 0, s>>>(ix->status, mask);
    set_error(msg);
    return SIA_E_INVALID;
  }
  return SIA_OK;
}

// scratch of the handle-less vote entry point, kept per device (cudaMalloc of GBs per call is slow)
Arena g_vote_tables[64];

// ---- the table vote: one attempt over one set of tables ---------------------------------------------------------
// bin slots reserved for `tuples` tuples over nq queries: first for up to a quarter of the tuples landing in twice-hit
// buckets (12 % on the benchmark's index), then — if pass 1 counted more — for all of them
int64_t bin_slots_for(int64_t tuples, int64_t nq, int attempt) {
  return (attempt == 0 ? tuples / 2 : 2 * tuples) + 32 * nq;
}

// bytes of the tables of group g for `tuples` tuples: filter + worst-case bins of the attempt (every tuple a
// candidate) + songs + the pieces of the entries path
size_t table_bytes(const Group &g, int64_t tuples, int attempt) {
  const int64_t nq = g.qb - g.qa;
  return (size_t)(tuples + nq) * 4 + (size_t)bin_slots_for(tuples, nq, attempt) * 16 + (size_t)g.ns * (g.dense ? 8 : 12) +
         (size_t)(tuples / (kVoteTuples >> 3) + 16) * 4 + 8192;
}

// what a table vote reads and writes besides its tables
struct TableVoteArgs {
  QMeta *meta;                    // indexed by the query id of the tuples
  uint32_t *qflag;                // per query: needs the singles pass
  int64_t *total;                 // bin slots in use
  int32_t *flags;                 // [0] device flags of the attempt, [1] queries of the group that need the singles pass
  unsigned long long *n_bins;     // NULL, or += the distinct bins of count >= 2
  const uint32_t *qsel;           // NULL, or only these queries (the ones the partitioned vote left over)
  int qid_base, topn;             // output row of query q: q + qid_base
  PvOut out;
};

template <int P> using PassTag = std::integral_constant<int, P>;

template <bool D, class Pass>
void table_vote_launches(const Pass &pass, const Group &g, const Tables &T, int64_t nb_cap, const TableVoteArgs &a,
                         StageEvents &tm, cudaStream_t s) {
  const std::bool_constant<D> dense{};
  const int gq = g.qb - g.qa;
  pass(dense, PassTag<PASS_MARK>{}, T);
  tm.mark(2, s);
  layout_bins_kernel<<<1, 1024, 0, s>>>(a.meta, g.qa, g.qb, a.total);
  zero_bins_kernel<<<kNumSMs * 8, 256, 0, s>>>(T.bins, T.bin_cnt, a.total, nb_cap, a.flags);
  tm.mark(3, s);
  pass(dense, PassTag<PASS_VOTE>{}, T);
  tm.mark(4, s);
  cand_vote_kernel<D><<<kNumSMs * 8, 256, 0, s>>>(T.cand, a.meta, g.qa, g.qb, T, a.n_bins, a.flags);
  tm.mark(5, s);
  topn_kernel<D, false><<<gq, 256, 0, s>>>(T, a.meta, g.qa, a.qid_base, a.topn, a.qflag, a.flags + 1, a.qsel, a.out.song,
                                           a.out.diff, a.out.count, a.out.rows, a.out.nres);
  tm.mark(6, s);
  pass(dense, PassTag<PASS_SINGLES>{}, T);
  topn_kernel<D, true><<<gq, 256, 0, s>>>(T, a.meta, g.qa, a.qid_base, a.topn, a.qflag, a.flags + 1, a.qsel, a.out.song,
                                          a.out.diff, a.out.count, a.out.rows, a.out.nres);
  tm.mark(7, s);
  pass(dense, PassTag<PASS_ROWS>{}, T);
  tm.mark(8, s);
}

// One attempt of the table vote over the queries [g.qa, g.qb) of `tuples` vote tuples: carves the group's tables from
// `ar` (bin slots for `attempt`), zeroes them, lays out the queries' QMeta on the device (layout()), then enqueues
// mark → bin layout → zero bins → collect → candidate vote → top-n → singles → top-n → rows.  pass(dense, PassTag<P>,
// tables) launches the walk of pass P over the caller's tuples (entries or vote keys; PASS_ROWS: the winners' rows).
// tm gets marks 0..8: start, after the layout, then after each stage.
template <class Layout, class Pass>
int table_vote(Arena &ar, const Group &g, int64_t tuples, int attempt, const TableVoteArgs &a, const Layout &layout,
               const Pass &pass, StageEvents &tm, cudaStream_t s) {
  const int64_t nb_cap = bin_slots_for(tuples, g.qb - g.qa, attempt);
  Tables T{};
  T.filter = ar.take<uint32_t>(g.nf);
  T.song_best = ar.take<unsigned long long>(g.ns);
  T.song_key = g.dense ? nullptr : ar.take<uint32_t>(g.ns);
  T.bins = ar.take<unsigned long long>(nb_cap);
  T.bin_cnt = ar.take<uint32_t>(nb_cap);
  T.cand = ar.take<unsigned long long>(nb_cap / 2 + 16);
  SIA_REQUIRE(T.filter && T.song_best && (g.dense || T.song_key) && T.bins && T.bin_cnt && T.cand, SIA_E_NOMEM,
              "index scratch arena too small (vote tables)");
  tm.mark(0, s);
  SIA_CUDA(cudaMemsetAsync(a.flags + 1, 0, sizeof(int32_t), s));
  SIA_CUDA(cudaMemsetAsync(T.filter, 0, sizeof(uint32_t) * g.nf, s));
  SIA_CUDA(cudaMemsetAsync(T.song_best, 0, sizeof(unsigned long long) * g.ns, s));
  if (!g.dense) SIA_CUDA(cudaMemsetAsync(T.song_key, 0, sizeof(uint32_t) * g.ns, s));
  int rc = layout();
  if (rc) return rc;
  tm.mark(1, s);
  if (g.dense) table_vote_launches<true>(pass, g, T, nb_cap, a, tm, s);
  else table_vote_launches<false>(pass, g, T, nb_cap, a, tm, s);
  SIA_CHECK_LAUNCH();
  return SIA_OK;
}

// after an attempt, from its device flags: retry when the bin tables outgrew attempt 0's reservation (tie-heavy
// queries), to be voted again with attempt 1; a full table (flag 8) is an error, `overflow` says why
int attempt_retry(int32_t h_flags, int attempt, const char *overflow, bool &retry) {
  SIA_REQUIRE(!(h_flags & 8), SIA_E_CUDA, overflow);
  retry = (h_flags & 32) != 0;
  SIA_REQUIRE(!retry || attempt == 0, SIA_E_CUDA, "vote: bin table overflow (internal error)");
  return SIA_OK;
}

// vote tuples per group of queries: SIA_VOTE_GROUP_TUPLES (default 2^29), bounded by what the device has left
int group_tuple_budget(::sia_index *ix, int64_t &budget) {
  budget = getenv("SIA_VOTE_GROUP_TUPLES") ? std::max(1ll, atoll(getenv("SIA_VOTE_GROUP_TUPLES"))) : (512ll << 20);
  size_t free_b = 0, total_b = 0;
  SIA_CUDA(cudaMemGetInfo(&free_b, &total_b));
  budget = std::max<int64_t>(1 << 20, std::min<int64_t>(budget, (int64_t)((free_b + ix->arena3.cap) * 0.6 / 40)));
  return SIA_OK;
}

}  // namespace

namespace sia {

size_t lookup_bytes(int64_t n) {
  return (size_t)n * (16 * 2 + 8 + 4 * 2) + (size_t)(n + 1) * 16 + radix_sort_tmp_bytes(n) + 16384;
}

int lookup_sorted(::sia_index *ix, Arena &ar, ulonglong2 *a, ulonglong2 *b, int64_t n, const int64_t *d_query_starts,
                  int64_t i0, int n_queries, int64_t max_query_entries, Lookup &L, cudaStream_t s) {
  ix->dist_nq = 0;                 // any new lookup reuses the arena: a pending sia_index_lookup_slots is void
  L = Lookup();
  L.n = n;
  if (n == 0) return SIA_OK;
  void *stmp = ar.take<char>(radix_sort_tmp_bytes(n));
  int64_t *first = ar.take<int64_t>(n);
  uint32_t *c_all = ar.take<uint32_t>(n), *c_head = ar.take<uint32_t>(n);
  int64_t *off_all = ar.take<int64_t>(n + 1), *off_head = ar.take<int64_t>(n + 1);
  SIA_REQUIRE(stmp && first && c_all && c_head && off_all && off_head, SIA_E_NOMEM, "index scratch arena too small (lookup)");
  bool in_b = false;
  int rc = SIA_OK;
  if (d_query_starts && max_query_entries > 0 && max_query_entries <= kSmemSortMax) {
    int P = 2;
    while (P < max_query_entries) P <<= 1;
    const size_t smem = (size_t)P * sizeof(ulonglong2);
    SIA_CUDA(cudaFuncSetAttribute(sort_queries_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    sort_queries_kernel<<<(unsigned)n_queries, kSmemSortThreads, smem, s>>>(a, d_query_starts, i0);
    SIA_CHECK_LAUNCH();
  } else if ((rc = radix_sort(a, b, n, 16, 0, 16, stmp, s, &in_b))) {
    return rc;
  }
  L.ent = in_b ? b : a;
  lookup_kernel<<<grid_for(n), 256, 0, s>>>(L.ent, n, ix->keys[ix->cur], ix->n_keys, ix->dir, ix->dir_bits, first, c_all,
                                           c_head, ix->status);
  SIA_CHECK_LAUNCH();
  if ((rc = exclusive_scan_u32(c_all, off_all, n, stmp, s))) return rc;
  if ((rc = exclusive_scan_u32(c_head, off_head, n, stmp, s))) return rc;
  int64_t tot[2];
  SIA_CUDA(cudaMemcpyAsync(&tot[0], off_all + n, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  SIA_CUDA(cudaMemcpyAsync(&tot[1], off_head + n, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  SIA_CUDA(cudaStreamSynchronize(s));
  L.first = first; L.cnt_head = c_head; L.off_all = off_all; L.off_head = off_head; L.tuples = tot[0]; L.head_rows = tot[1];
  return SIA_OK;
}

Arena &vote_arena(int device) { return g_vote_tables[device]; }

void vote_scratch_release(int device) {
  if (device >= 0 && device < 64) g_vote_tables[device].release();
}

// one vote over slotted keys: everything a retry or a deferred completion needs
struct KeyVote {
  bool pending = false;
  int device = 0;
  const uint64_t *d_keys = nullptr;
  int n_slots = 0;
  int64_t cap = 0;
  const int64_t *d_counts = nullptr;
  int32_t n_queries = 0, topn = 0, max_song = 0;
  int32_t *o_song = nullptr, *o_diff = nullptr, *o_count = nullptr, *o_rows = nullptr, *o_nres = nullptr;
  cudaStream_t s = nullptr;
  int32_t *d_flags = nullptr;      // device flags of the attempt in flight
  int stage = 1;                   // 0: the partitioned vote is in flight; 1: the table vote
  uint32_t *d_small = nullptr;     // per device, allocated once: [0] unsorted, [1] flagged queries, [64..] per-query flags
  const uint32_t *qsel = nullptr;  // table vote: only these queries (the ones the partitioned vote left over)
  StageEvents ev;                  // SIA_QUERY_TIMING
};
static KeyVote g_key_vote[64];

// enqueue every launch of one attempt (0: bin slots for a quarter of the keys being candidates; 1: for all of them)
static int key_vote_enqueue(KeyVote &v, int attempt) {
  const int nq = v.n_queries;
  const int64_t n_keys = (int64_t)v.n_slots * v.cap;     // upper bound of the keys
  Arena &ar = g_vote_tables[v.device];
  // song tables: dense (slot = song id) when that is the smaller layout, else open addressing
  const int64_t span = (int64_t)v.max_song + 1, ns_hashed = 2 * n_keys + 32ll * nq;
  const bool dense = span * nq * 8 <= ns_hashed * 12;
  const Group g{0, nq, dense, n_keys + nq, dense ? span * nq : ns_hashed};
  int rc = ar.reserve(table_bytes(g, n_keys, attempt) + (size_t)nq * (sizeof(QMeta) + 8) + 65536);
  if (rc) return rc;
  QMeta *meta = ar.take<QMeta>(nq);
  uint32_t *cnt = ar.take<uint32_t>(nq), *qflag = ar.take<uint32_t>(nq);
  int64_t *total = ar.take<int64_t>(1);
  int32_t *flags = ar.take<int32_t>(2);
  SIA_REQUIRE(meta && cnt && qflag && total && flags, SIA_E_NOMEM, "vote: scratch");
  v.d_flags = flags;
  v.ev.on = getenv("SIA_QUERY_TIMING") != nullptr;
  SIA_CUDA(cudaMemsetAsync(flags, 0, sizeof(int32_t), v.s));
  // blockIdx.y = slot; the x blocks of a slot stride over its keys (~32 resident blocks per SM in all)
  const dim3 grid((unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div(v.cap, 512), (kNumSMs * 32) / v.n_slots + 1)),
                  (unsigned)v.n_slots);
  const TableVoteArgs a{meta, qflag, total, flags, nullptr, v.qsel, 0, v.topn, {v.o_song, v.o_diff, v.o_count, v.o_rows, v.o_nres}};
  const auto layout = [&]() -> int {
    SIA_CUDA(cudaMemsetAsync(cnt, 0, sizeof(uint32_t) * nq, v.s));
    count_keys_kernel<<<grid, 256, 0, v.s>>>(v.d_keys, v.cap, v.d_counts, nq, v.qsel, cnt, flags);
    layout_keys_kernel<<<1, 1024, 0, v.s>>>(cnt, nq, dense ? span : 0, v.qsel, meta);
    return SIA_OK;
  };
  const auto pass = [&](auto d, auto p, const Tables &T) {
    keys_pass_kernel<decltype(d)::value, decltype(p)::value><<<grid, 256, 0, v.s>>>(
        v.d_keys, v.cap, v.d_counts, nq, meta, T, qflag, flags + 1, v.qsel, v.topn, v.o_song, v.o_nres, v.o_rows, flags);
  };
  return table_vote(ar, g, n_keys, attempt, a, layout, pass, v.ev, v.s);
}

// the partitioned vote of the keys (index_pvote.cu): shared-memory tables, streaming traffic only
static int key_pvote_enqueue(KeyVote &v) {
  if (!v.d_small) SIA_CUDA(cudaMalloc(&v.d_small, sizeof(uint32_t) * (64 + kMaxQueriesPerPass)));
  Arena &ar = g_vote_tables[v.device];
  int rc = ar.reserve(pvote_bytes((int64_t)v.n_slots * v.cap, v.n_queries, v.n_slots, v.topn) + 65536);
  if (rc) return rc;
  SIA_CUDA(cudaMemsetAsync(v.d_small, 0, sizeof(uint32_t) * (64 + (size_t)v.n_queries), v.s));
  v.ev.on = getenv("SIA_QUERY_TIMING") != nullptr;
  v.ev.mark(0, v.s);
  const PvOut po{v.o_song, v.o_diff, v.o_count, v.o_rows, v.o_nres};
  rc = pvote_key_slots(ar, v.d_keys, v.n_slots, v.cap, v.d_counts, v.n_queries, v.topn, po, v.d_small + 64, v.d_small, v.s);
  if (rc) return rc;
  v.ev.mark(1, v.s);
  return SIA_OK;
}

// wait for the vote in flight on this device, check its flags, redo it with the larger bin reservation if it asked
int vote_key_slots_finish(int device) {
  SIA_REQUIRE(device >= 0 && device < 64, SIA_E_INVALID, "device index");
  KeyVote &v = g_key_vote[device];
  if (!v.pending) return SIA_OK;
  v.pending = false;
  SIA_CUDA(cudaSetDevice(device));
  if (v.stage == 0) {
    uint32_t h2[2] = {0, 0};
    SIA_CUDA(cudaMemcpyAsync(h2, v.d_small, sizeof h2, cudaMemcpyDeviceToHost, v.s));
    SIA_CUDA(cudaStreamSynchronize(v.s));
    if (v.ev.on)
      fprintf(stderr, "[sia] key vote (partitioned): %d queries, %d slots x %lld: %.2f ms, unsorted %u, flagged queries %u\n",
              v.n_queries, v.n_slots, (long long)v.cap, v.ev.ms(0, 1), h2[0], h2[1]);
    if (!h2[0] && !h2[1]) return SIA_OK;
    // keys not grouped by query (any order is allowed): everything goes to the table vote; else only the flagged queries
    v.qsel = h2[0] ? nullptr : v.d_small + 64;
    v.stage = 1;
    int rc = key_vote_enqueue(v, 0);
    if (rc) return rc;
  }
  for (int attempt = 0;; ++attempt) {
    int32_t h_flags = 0;
    SIA_CUDA(cudaMemcpyAsync(&h_flags, v.d_flags, sizeof h_flags, cudaMemcpyDeviceToHost, v.s));
    SIA_CUDA(cudaStreamSynchronize(v.s));
    SIA_REQUIRE(!(h_flags & 2), SIA_E_INVALID, "vote: query id outside 0..n_queries-1");
    bool retry = false;
    int rc = attempt_retry(h_flags, attempt, "vote: table overflow (internal error, or song id above max_song)", retry);
    if (rc) return rc;
    StageEvents &e = v.ev;
    if (e.on)
      fprintf(stderr, "[sia] key vote: %d queries, %d slots x %lld: memsets + count + layout %.2f ms, mark %.2f, bin layout + collect %.2f, "
              "candidate vote %.2f, topn + singles %.2f, rows %.2f\n", v.n_queries, v.n_slots, (long long)v.cap, e.ms(0, 1),
              e.ms(1, 2), e.ms(2, 4), e.ms(4, 5), e.ms(5, 7), e.ms(7, 8));
    if (!retry) return SIA_OK;
    if ((rc = key_vote_enqueue(v, 1))) return rc;
  }
}

// defer != 0: return once everything is enqueued; vote_key_slots_finish(device) completes the call (one vote in flight
// per device; the key slots and outputs must stay alive until then)
int vote_key_slots(int device, const uint64_t *d_keys, int n_slots, int64_t cap, const int64_t *d_counts, int32_t n_queries,
                   int32_t topn, int32_t max_song, int32_t *d_out_song, int32_t *d_out_diff, int32_t *d_out_count,
                   int32_t *d_out_rows, int32_t *d_out_nres, cudaStream_t s, int defer) {
  SIA_REQUIRE(n_queries >= 0 && n_queries <= kMaxQueriesPerPass && topn >= 1, SIA_E_INVALID,
              "vote: 0..16384 queries per call, topn >= 1");
  SIA_REQUIRE(n_slots >= 1 && cap >= 0 && max_song >= 0 && max_song <= (int32_t)kM24, SIA_E_INVALID, "vote: bad sizes");
  if (n_queries == 0) return SIA_OK;
  SIA_REQUIRE(d_out_song && d_out_diff && d_out_count && d_out_rows && d_out_nres, SIA_E_INVALID, "NULL output");
  SIA_REQUIRE(device >= 0 && device < 64, SIA_E_INVALID, "device index");
  SIA_CUDA(cudaSetDevice(device));
  SIA_REQUIRE((int64_t)n_slots * cap < (1ll << 31), SIA_E_UNSUPPORTED, "vote: more than 2^31 key slots in one call");
  int rc = vote_key_slots_finish(device);               // a vote left in flight by the caller
  if (rc) return rc;
  KeyVote &v = g_key_vote[device];
  v.device = device; v.d_keys = d_keys; v.n_slots = n_slots; v.cap = cap; v.d_counts = d_counts;
  v.n_queries = n_queries; v.topn = topn; v.max_song = max_song;
  v.o_song = d_out_song; v.o_diff = d_out_diff; v.o_count = d_out_count; v.o_rows = d_out_rows; v.o_nres = d_out_nres;
  v.s = s;
  v.qsel = nullptr;
  if (topn <= kPvMaxTopn) {
    v.stage = 0;
    rc = key_pvote_enqueue(v);
  } else {
    v.stage = 1;
    rc = key_vote_enqueue(v, 0);
  }
  if (rc) return rc;
  v.pending = true;
  return defer ? SIA_OK : vote_key_slots_finish(device);
}

// completes a vote left in flight on the device (it owns the arena), then sizes the arena for a new user
int vote_scratch_finish_and_reserve(int device, size_t bytes) {
  int rc = vote_key_slots_finish(device);
  if (rc) return rc;
  return g_vote_tables[device].reserve(bytes);
}

namespace tvote {

Group make_group(int qa, int qb, const int64_t *h_off_all, const int64_t *h_off_head, int64_t span, QMeta *h_meta) {
  Group g{qa, qb, false, 0, 0};
  const int64_t h_all = h_off_head[qb] - h_off_head[qa];
  const int64_t ns_hashed = 2 * h_all + 32ll * (qb - qa);
  g.dense = span * (qb - qa) * 8 <= ns_hashed * 12 * 2;
  int64_t fb = 0, sb = 0;
  for (int q = qa; q < qb; ++q) {
    const int64_t t = h_off_all[q + 1] - h_off_all[q], h = h_off_head[q + 1] - h_off_head[q];
    QMeta &m = h_meta[q];
    m.bin_base = 0; m.bin_cap = 0; m.cand = 0; m.cand_base = 0; m.cursor = 0; m.pad_ = 0;
    m.filt_base = fb; m.filt_words = (uint32_t)(t + 1);
    m.song_base = sb; m.song_cap = g.dense ? (uint32_t)span : (uint32_t)(2 * h + 32);
    fb += m.filt_words; sb += m.song_cap;
  }
  g.nf = fb; g.ns = sb;
  return g;
}

std::vector<std::pair<int, int>> split_groups(const int64_t *h_off_all, int nq, int64_t budget, const uint32_t *keep) {
  std::vector<std::pair<int, int>> groups;
  for (int qa = 0; qa < nq;) {
    if (keep && !keep[qa]) { ++qa; continue; }
    int qb = qa + 1;
    while (qb < nq && (!keep || keep[qb]) && h_off_all[qb + 1] - h_off_all[qa] <= budget) ++qb;
    if (h_off_all[qb] > h_off_all[qa]) groups.emplace_back(qa, qb);
    qa = qb;
  }
  return groups;
}

}  // namespace tvote

// pack the pairs [h_query_starts[0], h_query_starts[nq]) of nq queries (d_qs: the same starts on the device) into
// ea (alt buffer eb), sort and look them up (lookup_sorted), check the offsets / ids.
static int lookup_queries(::sia_index *ix, const uint8_t *d_hash, const int32_t *d_qoff, const int64_t *h_query_starts,
                          const int64_t *d_qs, int nq, ulonglong2 *ea, ulonglong2 *eb, Lookup &L, cudaStream_t s) {
  const int64_t i0 = h_query_starts[0], n = h_query_starts[nq] - i0;
  int64_t max_entries = 0;
  for (int q = 0; q < nq; ++q) max_entries = std::max(max_entries, h_query_starts[q + 1] - h_query_starts[q]);
  pack_queries_kernel<<<grid_for(n), 256, 0, s>>>(d_hash, d_qoff, nullptr, d_qs, nq, i0, n, ea, ix->status);
  SIA_CHECK_LAUNCH();
  int rc = lookup_sorted(ix, ix->arena, ea, eb, n, d_qs, i0, nq, max_entries, L, s);
  if (rc) return rc;
  return check_status(ix, s, 2 | 4, "query: offset outside 0..2^24-1 (or a posting run of 2^32 rows)");
}

// scanned tuple / head-row offsets at the queries' first entries: h_goff[0..nq] = off_all, h_goff[nq+1..] = off_head
// (d_goff: 2 * (nq + 1) device scratch).  Synchronises the stream.
static int query_offsets(const Lookup &L, const int64_t *d_qs, int64_t i0, int nq, int64_t *d_goff, std::vector<int64_t> &h_goff,
                         cudaStream_t s) {
  h_goff.assign(2 * (size_t)(nq + 1), 0);
  gather_offsets_kernel<<<grid_for(nq + 1), 256, 0, s>>>(L.off_all, L.off_head, d_qs, i0, nq, d_goff);
  SIA_CHECK_LAUNCH();
  SIA_CUDA(cudaMemcpyAsync(h_goff.data(), d_goff, h_goff.size() * 8, cudaMemcpyDeviceToHost, s));
  SIA_CUDA(cudaStreamSynchronize(s));
  return SIA_OK;
}

int query_passes(::sia_index *ix, const uint8_t *d_hash, const int32_t *d_qoff, const int64_t *h_query_starts,
                 int32_t n_queries, int32_t topn, const QueryOut &out, int64_t *h_stats, cudaStream_t s, bool timing,
                 size_t (*extra_bytes)(int nq, int64_t n), const std::function<int(QueryPass &)> &vote) {
  SIA_REQUIRE(ix && h_query_starts, SIA_E_INVALID, "NULL argument");
  SIA_REQUIRE(n_queries >= 0 && topn >= 1, SIA_E_INVALID, "n_queries >= 0 and topn >= 1 required");
  SIA_REQUIRE(ix->n_pending == 0, SIA_E_INVALID, "index has pending rows: call sia_index_finalize first");
  if (h_stats) h_stats[0] = h_stats[1] = h_stats[2] = h_stats[3] = 0;
  if (n_queries == 0) return SIA_OK;
  SIA_REQUIRE(out.song && out.diff && out.count && out.rows && out.nres, SIA_E_INVALID, "NULL output");
  int rc = set_device(ix);
  if (rc) return rc;
  for (int q = 0; q < n_queries; ++q)
    SIA_REQUIRE(h_query_starts[q] <= h_query_starts[q + 1], SIA_E_INVALID, "query_starts must be non-decreasing");
  SIA_REQUIRE(h_query_starts[n_queries] == h_query_starts[0] || (d_hash && d_qoff), SIA_E_INVALID, "NULL input");
  for (int32_t *o : {out.nres, out.batches, out.exit})
    if (o) SIA_CUDA(cudaMemsetAsync(o, 0, sizeof(int32_t) * n_queries, s));
  for (int32_t *o : {out.song, out.diff, out.count, out.rows})
    SIA_CUDA(cudaMemsetAsync(o, 0, sizeof(int32_t) * (size_t)n_queries * topn, s));
  QueryPass p;
  p.s = s;
  if ((rc = group_tuple_budget(ix, p.budget))) return rc;
  for (auto &e : ix->ev_q) if (!e) SIA_CUDA(cudaEventCreate(&e));
  ix->last_lookup_ms = ix->last_vote_ms = 0;
  for (int64_t q0 = 0; q0 < n_queries; q0 += kMaxQueriesPerPass) {
    const int nq = (int)std::min<int64_t>(kMaxQueriesPerPass, n_queries - q0);
    const int64_t i0 = h_query_starts[q0], n = h_query_starts[q0 + nq] - i0;
    if (h_stats) h_stats[0] += n;
    if (n == 0) continue;    // the outputs of these queries stay zero
    if ((rc = ix->arena.reserve((size_t)(nq + 1) * 8 * 3 + (size_t)n * 32 + lookup_bytes(n) + extra_bytes(nq, n) + (1 << 20))))
      return rc;
    int64_t *d_qs = ix->arena.take<int64_t>(nq + 1);
    int64_t *d_goff = ix->arena.take<int64_t>(2 * (size_t)(nq + 1));
    ulonglong2 *ea = ix->arena.take<ulonglong2>(n), *eb = ix->arena.take<ulonglong2>(n);
    SIA_REQUIRE(d_qs && d_goff && ea && eb, SIA_E_NOMEM, "index scratch arena too small (query)");
    SIA_CUDA(cudaMemcpyAsync(d_qs, h_query_starts + q0, sizeof(int64_t) * (nq + 1), cudaMemcpyHostToDevice, s));
    const auto h0 = std::chrono::steady_clock::now();
    SIA_CUDA(cudaEventRecord(ix->ev_q[0], s));
    if ((rc = lookup_queries(ix, d_hash, d_qoff, h_query_starts + q0, d_qs, nq, ea, eb, p.L, s))) return rc;
    SIA_CUDA(cudaEventRecord(ix->ev_q[1], s));
    // After the sort query q still owns entries [starts[q]-i0, starts[q+1]-i0) (duplicates stay, with no
    // postings), so the scanned offsets at those positions split the pass into groups that fit the budget.
    std::vector<int64_t> h_goff;
    if ((rc = query_offsets(p.L, d_qs, i0, nq, d_goff, h_goff, s))) return rc;
    for (int q = 0; q < nq; ++q)
      SIA_REQUIRE(h_goff[q + 1] - h_goff[q] < (1ll << 31), SIA_E_UNSUPPORTED, "query: more than 2^31 vote tuples in one query");
    p.q0 = q0; p.i0 = i0; p.n = n; p.nq = nq;
    p.h_qs = h_query_starts + q0; p.d_qs = d_qs;
    p.h_off_all = h_goff.data(); p.h_off_head = h_goff.data() + nq + 1; p.d_goff = d_goff;
    p.groups = 0;
    if ((rc = vote(p))) return rc;
    SIA_CUDA(cudaEventRecord(ix->ev_q[2], s));
    SIA_CUDA(cudaStreamSynchronize(s));
    float t_lookup = 0, t_vote = 0;
    cudaEventElapsedTime(&t_lookup, ix->ev_q[0], ix->ev_q[1]); cudaEventElapsedTime(&t_vote, ix->ev_q[1], ix->ev_q[2]);
    ix->last_lookup_ms += t_lookup; ix->last_vote_ms += t_vote;
    if (timing) {
      const double host_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - h0).count();
      fprintf(stderr, "[sia] query pass: %d queries, %lld entries, %lld tuples, %zu groups: lookup %.2f ms, vote %.2f ms, host wall %.2f ms\n",
              nq, (long long)n, (long long)p.L.tuples, p.groups, t_lookup, t_vote, host_ms);
    }
  }
  return SIA_OK;
}

}  // namespace sia

extern "C" {

int sia_index_select_host(sia_index *ix, const uint8_t *h_hash, int64_t n, int32_t *h_row_hashidx, int32_t *h_row_song,
                          int32_t *h_row_off, int64_t cap, int64_t *h_nrows) {
  SIA_REQUIRE(ix && h_nrows, SIA_E_INVALID, "NULL argument");
  SIA_REQUIRE(ix->n_pending == 0, SIA_E_INVALID, "index has pending rows: call sia_index_finalize first");
  *h_nrows = 0;
  if (n == 0) return SIA_OK;
  SIA_REQUIRE(h_hash && n > 0 && n <= (int64_t)kM24, SIA_E_INVALID, "select: 1..2^24-1 hashes per call");
  int rc = set_device(ix);
  if (rc) return rc;
  cudaStream_t s = nullptr;
  SIA_CUDA(cudaDeviceSynchronize());
  // position of each hash rides in the qoff field, qid = 0 -> sorted by (digest, position)
  std::vector<int32_t> pos(n);
  for (int64_t i = 0; i < n; ++i) pos[i] = (int32_t)i;
  const size_t in_bytes = (size_t)n * (SIA_HASH_BYTES + 4 + 4) + 4096;
  if ((rc = ix->arena.reserve(in_bytes + lookup_bytes(n) + (size_t)cap * 12 + 4096))) return rc;
  uint8_t *dh = ix->arena.take<uint8_t>((size_t)n * SIA_HASH_BYTES);
  int32_t *dpos = ix->arena.take<int32_t>(n), *dq = ix->arena.take<int32_t>(n);
  ulonglong2 *a = ix->arena.take<ulonglong2>(n), *b = ix->arena.take<ulonglong2>(n);
  SIA_REQUIRE(dh && dpos && dq && a && b, SIA_E_NOMEM, "index scratch arena too small (select)");
  SIA_CUDA(cudaMemcpyAsync(dh, h_hash, (size_t)n * SIA_HASH_BYTES, cudaMemcpyHostToDevice, s));
  SIA_CUDA(cudaMemcpyAsync(dpos, pos.data(), (size_t)n * 4, cudaMemcpyHostToDevice, s));
  SIA_CUDA(cudaMemsetAsync(dq, 0, (size_t)n * 4, s));
  pack_queries_kernel<<<grid_for(n), 256, 0, s>>>(dh, dpos, dq, nullptr, 1, 0, n, a, ix->status);
  SIA_CHECK_LAUNCH();
  Lookup L;
  if ((rc = lookup_sorted(ix, ix->arena, a, b, n, nullptr, 0, 1, 0, L, s))) return rc;
  *h_nrows = L.tuples;
  const int64_t m = std::min(L.tuples, cap);
  if (m > 0) {
    SIA_REQUIRE(h_row_hashidx && h_row_song && h_row_off, SIA_E_INVALID, "NULL output");
    int32_t *o1 = ix->arena.take<int32_t>(m), *o2 = ix->arena.take<int32_t>(m), *o3 = ix->arena.take<int32_t>(m);
    SIA_REQUIRE(o1 && o2 && o3, SIA_E_NOMEM, "index scratch arena too small (select)");
    select_rows_kernel<<<grid_for(n), 256, 0, s>>>(L.ent, n, L.first, L.off_all, ix->post, o1, o2, o3, m);
    SIA_CHECK_LAUNCH();
    SIA_CUDA(cudaMemcpyAsync(h_row_hashidx, o1, (size_t)m * 4, cudaMemcpyDeviceToHost, s));
    SIA_CUDA(cudaMemcpyAsync(h_row_song, o2, (size_t)m * 4, cudaMemcpyDeviceToHost, s));
    SIA_CUDA(cudaMemcpyAsync(h_row_off, o3, (size_t)m * 4, cudaMemcpyDeviceToHost, s));
  }
  SIA_CUDA(cudaStreamSynchronize(s));
  return SIA_OK;
}

int sia_index_query_batch(sia_index *ix, const uint8_t *d_hash, const int32_t *d_qoff, const int64_t *h_query_starts,
                          int32_t n_queries, int32_t topn, int32_t *d_out_song, int32_t *d_out_diff,
                          int32_t *d_out_count, int32_t *d_out_rows, int32_t *d_out_nres, int64_t *h_stats, void *stream) {
  const QueryOut out{{d_out_song, d_out_diff, d_out_count, d_out_rows, d_out_nres}, nullptr, nullptr};
  const bool timing = getenv("SIA_QUERY_TIMING") != nullptr;       // stage times of every pass on stderr
  double stage_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};                   // table vote, summed over the call's groups
  const auto vote = [&](QueryPass &p) -> int {
    const int nq = p.nq;
    const int64_t *h_off_all = p.h_off_all;
    const Lookup &L = p.L;
    cudaStream_t s = p.s;
    StageEvents &tm = ix->ev_stage;
    tm.on = timing;
    if (h_stats) { h_stats[1] += L.head_rows; h_stats[2] += L.tuples; }
    int rc = SIA_OK;
    std::vector<std::pair<int, int>> table_groups;    // what the table vote has to do
    unsigned long long h_nb_pv = 0;
    if (topn <= kPvMaxTopn) {
      // ---- partitioned vote (index_pvote.cu): shared-memory tables, streaming traffic only --------------------------
      const auto pg = split_groups(h_off_all, nq, p.budget, nullptr);
      size_t max_bytes = 0;
      for (const auto &[qa, qb] : pg) max_bytes = std::max(max_bytes, pvote_bytes(h_off_all[qb] - h_off_all[qa], qb - qa, 1, topn));
      if ((rc = ix->arena3.reserve(max_bytes + (size_t)nq * 8 + 65536))) return rc;
      uint32_t *d_qover = ix->arena3.take<uint32_t>(2 * (size_t)nq), *d_qbins = d_qover + nq;
      unsigned long long *d_nbins = ix->arena3.take<unsigned long long>(1);
      SIA_REQUIRE(d_qover && d_nbins, SIA_E_NOMEM, "index scratch arena too small (vote)");
      const size_t fixed = ix->arena3.used;
      SIA_CUDA(cudaMemsetAsync(d_qover, 0, sizeof(uint32_t) * 2 * nq, s));
      SIA_CUDA(cudaMemsetAsync(d_nbins, 0, sizeof(unsigned long long), s));
      double pv_ms[3] = {0, 0, 0};
      longlong2 *d_info = ix->arena.take<longlong2>(p.n);
      uint32_t *d_qh = ix->arena.take<uint32_t>(p.n);
      SIA_REQUIRE(d_info && d_qh, SIA_E_NOMEM, "index scratch arena too small (entry info)");
      if ((rc = pvote_entry_info(L, d_info, d_qh, s))) return rc;
      for (const auto &[qa, qb] : pg) {
        ix->arena3.used = fixed;
        if ((rc = pvote_entries(ix->arena3, L, d_info, d_qh, ix->post, p.d_qs, p.i0, p.d_goff, h_off_all, qa, qb, (int)p.q0, topn, out,
                                d_qover, d_qbins, h_stats ? d_nbins : nullptr, s, tm)))
          return rc;
        if (tm.on) for (int k = 0; k < 3; ++k) pv_ms[k] += tm.ms(k, k + 1);
        const int64_t e0 = p.h_qs[qa] - p.i0, ne = p.h_qs[qb] - p.i0 - e0;
        entries_rows_kernel<<<grid_for(ne * 32), 256, 0, s>>>(L.ent, e0, ne, L.first, L.cnt_head, ix->post, (int)p.q0, topn,
                                                             out.song, out.nres, out.rows);
        SIA_CHECK_LAUNCH();
      }
      std::vector<uint32_t> h_qover(nq);
      SIA_CUDA(cudaMemcpyAsync(h_qover.data(), d_qover, sizeof(uint32_t) * nq, cudaMemcpyDeviceToHost, s));
      SIA_CUDA(cudaMemcpyAsync(&h_nb_pv, d_nbins, sizeof h_nb_pv, cudaMemcpyDeviceToHost, s));
      SIA_CUDA(cudaStreamSynchronize(s));
      // queries that did not fit their partitions (a bin of thousands of matches, > 2048 partitions): table vote
      table_groups = split_groups(h_off_all, nq, p.budget, h_qover.data());
      if (timing)
        fprintf(stderr, "[sia]   partitioned vote, %zu group(s): layout %.2f ms, scatter %.2f, count + merge %.2f; %zu group(s) of flagged "
                "queries go to the table vote\n", pg.size(), pv_ms[0], pv_ms[1], pv_ms[2], table_groups.size());
    } else {
      table_groups = split_groups(h_off_all, nq, p.budget, nullptr);
    }
    std::vector<QMeta> h_meta(nq);
    std::vector<Group> groups;
    for (const auto &[qa, qb] : table_groups)
      groups.push_back(make_group(qa, qb, h_off_all, p.h_off_head, (int64_t)ix->max_song + 1, h_meta.data()));
    p.groups = groups.size();
    unsigned long long h_nb = 0;
    for (int attempt = 0; !groups.empty(); ++attempt) {
      size_t max_bytes = 0;
      for (const Group &g : groups) max_bytes = std::max(max_bytes, table_bytes(g, h_off_all[g.qb] - h_off_all[g.qa], attempt));
      if ((rc = ix->arena3.reserve(max_bytes + (size_t)nq * (sizeof(QMeta) + 4) + 65536))) return rc;
      QMeta *d_meta = ix->arena3.take<QMeta>(nq);
      uint32_t *qflag = ix->arena3.take<uint32_t>(nq);
      int64_t *d_total = ix->arena3.take<int64_t>(1);
      unsigned long long *d_nbins = ix->arena3.take<unsigned long long>(1);
      int32_t *d_flags = ix->arena3.take<int32_t>(2);
      const size_t fixed = ix->arena3.used;
      SIA_REQUIRE(d_meta && qflag && d_total && d_nbins && d_flags, SIA_E_NOMEM, "index scratch arena too small (vote)");
      SIA_CUDA(cudaMemsetAsync(d_nbins, 0, sizeof(unsigned long long), s));
      SIA_CUDA(cudaMemsetAsync(d_flags, 0, sizeof(int32_t), s));
      const TableVoteArgs a{d_meta, qflag, d_total, d_flags, d_nbins, nullptr, (int)p.q0, topn, out};
      for (const Group &g : groups) {
        const int64_t e0 = p.h_qs[g.qa] - p.i0, ne = p.h_qs[g.qb] - p.i0 - e0;
        const int64_t tuples = h_off_all[g.qb] - h_off_all[g.qa];
        ix->arena3.used = fixed;
        const unsigned blocks = (unsigned)ceil_div(tuples, kVoteTuples);
        const int64_t n_pieces = (int64_t)blocks * 8;
        uint32_t *piece_ent = ix->arena3.take<uint32_t>(n_pieces);
        SIA_REQUIRE(piece_ent != nullptr, SIA_E_NOMEM, "index scratch arena too small (vote pieces)");
        piece_entries_kernel<<<grid_for(n_pieces), 256, 0, s>>>(L.off_all, e0, ne, n_pieces, piece_ent);
        const auto layout = [&]() -> int {
          SIA_CUDA(cudaMemcpyAsync(d_meta + g.qa, h_meta.data() + g.qa, sizeof(QMeta) * (g.qb - g.qa), cudaMemcpyHostToDevice, s));
          return SIA_OK;
        };
        const auto pass = [&](auto d, auto pt, const Tables &T) {
          if constexpr (decltype(pt)::value == PASS_ROWS)
            entries_rows_kernel<<<grid_for(ne * 32), 256, 0, s>>>(L.ent, e0, ne, L.first, L.cnt_head, ix->post, (int)p.q0, topn,
                                                                 out.song, out.nres, out.rows);
          else
            entries_pass_kernel<decltype(d)::value, decltype(pt)::value><<<blocks, 256, 0, s>>>(
                L.ent, e0, ne, L.first, L.off_all, piece_ent, ix->post, d_meta, T, qflag, d_flags + 1, d_nbins, d_flags);
        };
        if ((rc = table_vote(ix->arena3, g, tuples, attempt, a, layout, pass, tm, s))) return rc;
        if (tm.on) {      // memsets, mark, bin layout + zero, collect + candidate vote, candidate vote, topn, singles + topn, rows
          const int to[8] = {1, 2, 3, 5, 5, 6, 7, 8};
          for (int k = 0; k < 8; ++k) stage_ms[k] += tm.ms(k, to[k]);
        }
      }
      int32_t h_flags = 0;
      SIA_CUDA(cudaMemcpyAsync(&h_flags, d_flags, sizeof h_flags, cudaMemcpyDeviceToHost, s));
      SIA_CUDA(cudaMemcpyAsync(&h_nb, d_nbins, sizeof h_nb, cudaMemcpyDeviceToHost, s));
      SIA_CUDA(cudaStreamSynchronize(s));      // the lookup scratch and the tables are reused by the next pass / call
      bool retry = false;
      if ((rc = attempt_retry(h_flags, attempt, "query: vote table overflow (internal error)", retry))) return rc;
      if (!retry) break;
    }
    if (h_stats) h_stats[3] += (int64_t)(h_nb + h_nb_pv);
    if (timing)
      fprintf(stderr, "[sia]   vote stages (ms): table memsets %.2f, mark %.2f, bin layout + zero %.2f, collect + candidate vote %.2f "
              "(candidate vote %.2f), topn %.2f, singles + topn %.2f, rows %.2f\n", stage_ms[0], stage_ms[1], stage_ms[2],
              stage_ms[3], stage_ms[4], stage_ms[5], stage_ms[6], stage_ms[7]);
    return SIA_OK;
  };
  return query_passes(ix, d_hash, d_qoff, h_query_starts, n_queries, topn, out, h_stats, (cudaStream_t)stream, timing,
                      [](int, int64_t n) { return (size_t)n * 20; }, vote);   // the partitioned vote's entry info
}

int sia_index_query_timing(const sia_index *ix, double *h_ms2) {
  SIA_REQUIRE(ix && h_ms2, SIA_E_INVALID, "NULL argument");
  h_ms2[0] = ix->last_lookup_ms; h_ms2[1] = ix->last_vote_ms;
  return SIA_OK;
}

int sia_vote_tuples(int device, const uint64_t *d_key, int64_t n_keys, int32_t n_queries, int32_t topn, int32_t max_song,
                    int32_t *d_out_song, int32_t *d_out_diff, int32_t *d_out_count, int32_t *d_out_rows,
                    int32_t *d_out_nres, void *stream) {
  SIA_REQUIRE(n_keys >= 0, SIA_E_INVALID, "negative size");
  SIA_REQUIRE(device >= 0 && device < 64, SIA_E_INVALID, "device index");
  SIA_CUDA(cudaSetDevice(device));
  cudaStream_t s = (cudaStream_t)stream;
  static int64_t *d_count[64] = {nullptr};                      // one device scalar per device
  if (!d_count[device]) SIA_CUDA(cudaMalloc(&d_count[device], sizeof(int64_t)));
  SIA_CUDA(cudaMemcpyAsync(d_count[device], &n_keys, sizeof n_keys, cudaMemcpyHostToDevice, s));
  SIA_CUDA(cudaStreamSynchronize(s));                           // n_keys is a stack variable
  if (n_queries > 0 && d_out_nres) {
    SIA_CUDA(cudaMemsetAsync(d_out_nres, 0, sizeof(int32_t) * n_queries, s));
    for (int32_t *o : {d_out_song, d_out_diff, d_out_count, d_out_rows})
      if (o) SIA_CUDA(cudaMemsetAsync(o, 0, sizeof(int32_t) * (size_t)n_queries * topn, s));
  }
  return vote_key_slots(device, d_key, 1, std::max<int64_t>(n_keys, 1), d_count[device], n_queries, topn, max_song, d_out_song,
                        d_out_diff, d_out_count, d_out_rows, d_out_nres, s, 0);
}

}  // extern "C"
