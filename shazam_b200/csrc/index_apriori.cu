// K4, query side — the a-priori early exit of recognizer_apriori.py:246-310 on the device (sia_index_query_apriori).
//
// The reference reads a query's distinct hashes in batches of B, aligns what it has read after every batch and stops
// once the best song has more than twice the matched DB rows of the runner-up.  Here the batches follow ascending
// digest order (the reference's order is that of a Python set, which is undefined), so that batch k of a query is one
// contiguous range of its lookup entries, which arrive sorted by (query, hash, offset).
//
// Per pass of queries: the lookup of index_query.cu (pack, sort, posting runs, scanned tuple / head-row offsets), then
// an exclusive scan of the head flags (first entry of each (query, hash)) gives every entry its distinct-hash rank and
// so its batch.  Queries are grouped under the tuple budget of the table vote; per group:
//   layout   every query owns an exact bin table (2 slots per tuple it can read, no singleton filter: a count-1 bin
//            can still grow), a song table (dense or open addressing, make_group) with best key, rows and round stamp
//            per song, and a changed list; the entries with postings are bucketed by batch (counting sort), so round
//            k's work is one contiguous range of that list;
//   rounds   k = 0 .. K_max-1, launched back to back with no host synchronisation:
//            vote    one warp per entry of batch k whose query is still active: every posting is one vote tuple, read
//                    once — bin count, song best (atomicMax of count | inverted diff), rows (head entries); a song
//                    whose best rose is pushed once per round onto its query's changed list (round stamp);
//            decide  one warp per active query: best keys only grow, so the new top max(topn, 2) is found among the
//                    previous top list and the changed list; the exit rule is checked on the top two, and on exit or
//                    after the query's last batch the outputs are written and the query retires.
// One host synchronisation per group (overflow flags, which the sizing rules out).
#include "index.cuh"

using namespace sia;
using namespace sia::tvote;

namespace {

constexpr int kRoundBlocks = kNumSMs * 16;     // blocks of the round vote (grid-stride over the round's entries)

// per entry: 1 if it is the first of its (query, hash)
__global__ void __launch_bounds__(256)
head_flags_kernel(const ulonglong2 *__restrict__ ent, int64_t n, uint32_t *__restrict__ head) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    bool h = true;
    if (i > 0) {
      const ulonglong2 e = ent[i], p = ent[i - 1];
      h = !(p.y == e.y && (p.x >> 24) == (e.x >> 24));
    }
    head[i] = h ? 1u : 0u;
  }
}

// per query of the pass: batches K_q = ceil(distinct hashes / B); out_batches starts at K_q (the value of a query
// whose exit never fires)
__global__ void __launch_bounds__(256)
query_batches_kernel(const int64_t *__restrict__ hr, const int64_t *__restrict__ qs, int64_t i0, int nq, int64_t B,
                     uint32_t *__restrict__ nb, int32_t *__restrict__ out_batches) {
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += gridDim.x * blockDim.x) {
    const int64_t distinct = hr[qs[q + 1] - i0] - hr[qs[q] - i0];
    const uint32_t k = (uint32_t)((distinct + B - 1) / B);
    nb[q] = k;
    out_batches[q] = (int32_t)k;
  }
}

// batch of entry i (hash rank inside its query / B), -1 for an entry without postings
__device__ __forceinline__ int entry_batch(const ulonglong2 *__restrict__ ent, const int64_t *__restrict__ off_all,
                                           const int64_t *__restrict__ hr, const int64_t *__restrict__ qs, int64_t i0,
                                           int64_t i, int64_t B) {
  if (off_all[i + 1] == off_all[i]) return -1;
  const uint32_t q = (uint32_t)(ent[i].y >> 40);
  return (int)((hr[i + 1] - 1 - hr[qs[q] - i0]) / B);
}

// counting sort of the group's entries [e0, e0 + ne) by batch.  SCATTER = false: count per batch; true: write the
// entry (relative to e0) at boff[b] + its place.  Entries of one warp mostly share a batch: one atomic per batch and warp.
template <bool SCATTER>
__global__ void __launch_bounds__(256)
bucket_entries_kernel(const ulonglong2 *__restrict__ ent, const int64_t *__restrict__ off_all, const int64_t *__restrict__ hr,
                      const int64_t *__restrict__ qs, int64_t i0, int64_t e0, int64_t ne, int64_t B, uint32_t *__restrict__ bcnt,
                      const int64_t *__restrict__ boff, uint32_t *__restrict__ perm) {
  const int lane = threadIdx.x & 31;
  for (int64_t j0 = (int64_t)blockIdx.x * blockDim.x; j0 < ne; j0 += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = j0 + threadIdx.x;
    const int b = j < ne ? entry_batch(ent, off_all, hr, qs, i0, e0 + j, B) : -1;
    const uint32_t active = __ballot_sync(0xffffffffu, b >= 0);
    if (b >= 0) {
      const uint32_t peers = __match_any_sync(active, b);
      const int leader = __ffs(peers) - 1;
      uint32_t base = 0;
      if (lane == leader) base = atomicAdd(&bcnt[b], (uint32_t)__popc(peers));
      if (SCATTER) {
        base = __shfl_sync(peers, base, leader);
        perm[boff[b] + base + __popc(peers & ((1u << lane) - 1u))] = (uint32_t)j;
      }
    }
    __syncwarp();
  }
}

// round k, vote: one warp per entry of batch k (perm[boff[k] .. boff[k+1])) whose query is still active
template <bool DENSE>
__global__ void __launch_bounds__(256)
round_vote_kernel(int k, const ulonglong2 *__restrict__ ent, int64_t e0, const int64_t *__restrict__ first,
                  const uint32_t *__restrict__ cnt_head, const int64_t *__restrict__ off_all, const uint32_t *__restrict__ perm,
                  const int64_t *__restrict__ boff, const uint64_t *__restrict__ post, QMeta *__restrict__ meta, int qa,
                  Tables T, uint32_t *__restrict__ rows, uint32_t *__restrict__ stamp, uint32_t *__restrict__ chg,
                  const uint32_t *__restrict__ done, unsigned long long *__restrict__ stats, int32_t *__restrict__ flags) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int64_t j_hi = boff[k + 1];
  unsigned long long n_tup = 0, n_rows = 0;          // lane 0: tuples / head tuples this warp voted
  uint32_t fresh = 0;
  for (int64_t j = boff[k] + (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); j < j_hi; j += warps) {
    const int64_t ei = e0 + perm[j];
    const ulonglong2 e = ent[ei];
    const uint32_t q = (uint32_t)(e.y >> 40) - (uint32_t)qa;
    if (done[q]) continue;
    const QMeta m = meta[q];
    const uint32_t qoff = (uint32_t)(e.x & kM24);
    const bool head = cnt_head[ei] != 0;
    const uint64_t *__restrict__ run = post + first[ei];
    const uint32_t c = (uint32_t)(off_all[ei + 1] - off_all[ei]);
    n_tup += c;
    if (head) n_rows += c;
    for (uint32_t kw = 0; kw < c; kw += 32) {
      const uint32_t i = kw + lane;
      bool push = false;
      int64_t ss = -1;
      if (i < c) {
        const uint64_t r = __ldcs(run + i);
        const uint32_t song = (uint32_t)(r >> 24) & 0xffffffu, dbits = (uint32_t)(r & kM24) - qoff + SIA_DIFF_BIAS;
        const unsigned long long cnt = bin_count(m, song, dbits, T, fresh, flags);
        ss = song_slot<DENSE>(m, song, T.song_key);
        if (ss < 0) {
          atomicOr(flags, 8);
        } else {
          if (head) atomicAdd(&rows[ss], 1u);
          push = cnt && best_raise(&T.song_best[ss], best_key(cnt, dbits)) && __ldcg(&stamp[ss]) != (uint32_t)k + 1u &&
                 atomicExch(&stamp[ss], (uint32_t)k + 1u) != (uint32_t)k + 1u;
        }
      }
      const uint32_t pm = __ballot_sync(0xffffffffu, push);
      if (pm) {
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(&meta[q].cursor, (uint32_t)__popc(pm));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (push) {
          const uint32_t at = base + __popc(pm & ((1u << lane) - 1u));
          if (at < m.cand) chg[m.cand_base + at] = (uint32_t)(ss - m.song_base);
          else atomicOr(flags, 8);
        }
      }
    }
  }
  if (lane == 0 && n_tup) { atomicAdd(&stats[0], n_tup); atomicAdd(&stats[1], n_rows); }
}

// round k, decide: one warp per query of the group.  top[2][gq][L] double-buffers the song slots of the ranked list.
template <bool DENSE>
__global__ void __launch_bounds__(256)
round_decide_kernel(int k, int gq, int qbase, int topn, int L, QMeta *__restrict__ meta, Tables T,
                    const uint32_t *__restrict__ rows, const uint32_t *__restrict__ chg, uint32_t *__restrict__ top,
                    uint32_t *__restrict__ ntop, uint32_t *__restrict__ done, const uint32_t *__restrict__ nb,
                    int32_t *__restrict__ out_song, int32_t *__restrict__ out_diff, int32_t *__restrict__ out_count,
                    int32_t *__restrict__ out_rows, int32_t *__restrict__ out_nres, int32_t *__restrict__ out_batches,
                    int32_t *__restrict__ out_exit) {
  const int lane = threadIdx.x & 31;
  const int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (q >= gq || done[q] || (uint32_t)k >= nb[q]) return;
  const QMeta m = meta[q];
  const uint32_t *__restrict__ old_top = top + ((size_t)((k + 1) & 1) * gq + q) * L;
  uint32_t *__restrict__ new_top = top + ((size_t)(k & 1) * gq + q) * L;
  const uint32_t n_old = k ? ntop[(size_t)((k + 1) & 1) * gq + q] : 0u, n_cand = n_old + min(m.cursor, m.cand);
  // candidates: the previous list, then the songs whose best rose this round (a song may be in both: equal rank keys
  // are kept once per lane, and the winner leaves every lane's list)
  unsigned long long prev = ~0ull;
  int nres = 0;
  while (nres < L) {
    unsigned long long tk[kTopK];
    uint32_t ts[kTopK];
#pragma unroll
    for (int i = 0; i < kTopK; ++i) { tk[i] = 0; ts[i] = 0; }
    for (uint32_t i = lane; i < n_cand; i += 32) {
      uint32_t sl = i < n_old ? old_top[i] : chg[m.cand_base + i - n_old];
      const unsigned long long best = __ldcg(&T.song_best[m.song_base + sl]);
      const uint32_t song = DENSE ? sl : __ldcg(&T.song_key[m.song_base + sl]) - 1u;
      unsigned long long key = ((best >> kDiffBits) << kSongBits) | (kM24 - song);   // count desc, then song id asc
      if (key >= prev || key <= tk[kTopK - 1]) continue;
      bool seen = false;
#pragma unroll
      for (int t = 0; t < kTopK; ++t) seen = seen || tk[t] == key;
      if (seen) continue;
#pragma unroll
      for (int t = 0; t < kTopK; ++t)
        if (key > tk[t]) { const unsigned long long a = tk[t]; const uint32_t b = ts[t]; tk[t] = key; ts[t] = sl; key = a; sl = b; }
    }
    int got = 0;
    for (; got < kTopK && nres < L; ++got) {
      unsigned long long bk = tk[0];
      uint32_t bs = ts[0];
#pragma unroll
      for (int d = 16; d; d >>= 1) {
        const unsigned long long ok = __shfl_xor_sync(0xffffffffu, bk, d);
        const uint32_t os = __shfl_xor_sync(0xffffffffu, bs, d);
        if (ok > bk) { bk = ok; bs = os; }
      }
      if (bk == 0) break;
      if (lane == 0) new_top[nres] = bs;
      if (tk[0] == bk) {
#pragma unroll
        for (int t = 0; t + 1 < kTopK; ++t) { tk[t] = tk[t + 1]; ts[t] = ts[t + 1]; }
        tk[kTopK - 1] = 0;
      }
      prev = bk;
      ++nres;
    }
    if (got < kTopK) break;
  }
  __syncwarp();
  if (lane != 0) return;
  ntop[(size_t)(k & 1) * gq + q] = (uint32_t)nres;
  meta[q].cursor = 0;
  // recognizer_apriori.py:305: songs_arr[0][HASHES_MATCHED] / 2 > songs_arr[1][HASHES_MATCHED]
  const bool fire = nres >= 2 && (uint64_t)rows[m.song_base + new_top[0]] > 2ull * rows[m.song_base + new_top[1]];
  if (!fire && (uint32_t)k + 1 < nb[q]) return;
  const int qo = qbase + q;
  const int nout = min(nres, topn);
  for (int r = 0; r < nout; ++r) {
    const uint32_t sl = new_top[r];
    const unsigned long long best = T.song_best[m.song_base + sl];
    const int64_t o = (int64_t)qo * topn + r;
    out_song[o] = (int32_t)(DENSE ? sl : T.song_key[m.song_base + sl] - 1u);
    out_diff[o] = (int32_t)(kDiffMask - (best & kDiffMask)) - SIA_DIFF_BIAS;
    out_count[o] = (int32_t)(best >> kDiffBits);
    out_rows[o] = (int32_t)rows[m.song_base + sl];
  }
  out_nres[qo] = nout;
  out_batches[qo] = k + 1;
  out_exit[qo] = fire ? 1 : 0;
  done[q] = 1;
}

}  // namespace

extern "C" int sia_index_query_apriori(sia_index *ix, const uint8_t *d_hash, const int32_t *d_qoff, const int64_t *h_query_starts,
                                       int32_t n_queries, int32_t topn, int32_t batch_hashes, int32_t *d_out_song,
                                       int32_t *d_out_diff, int32_t *d_out_count, int32_t *d_out_rows, int32_t *d_out_nres,
                                       int32_t *d_out_batches, int32_t *d_out_exit, int64_t *h_stats, void *stream) {
  SIA_REQUIRE(n_queries >= 0 && topn >= 1 && batch_hashes >= 1, SIA_E_INVALID,
              "n_queries >= 0, topn >= 1 and batch_hashes >= 1 required");
  SIA_REQUIRE(n_queries == 0 || (d_out_song && d_out_diff && d_out_count && d_out_rows && d_out_nres && d_out_batches &&
                                 d_out_exit), SIA_E_INVALID, "NULL output");
  const QueryOut out{{d_out_song, d_out_diff, d_out_count, d_out_rows, d_out_nres}, d_out_batches, d_out_exit};
  const int L = std::max(topn, 2);                   // the exit rule always looks at the top two
  const int64_t B = batch_hashes;
  const auto vote = [&](QueryPass &p) -> int {
    const int nq = p.nq;
    const int64_t n = p.n, i0 = p.i0, q0 = p.q0;
    const int64_t *h_off_all = p.h_off_all, *h_off_head = p.h_off_head, *d_qs = p.d_qs;
    const Lookup &Lk = p.L;
    cudaStream_t s = p.s;
    // distinct-hash rank of every entry: hr[i + 1] - 1 - hr[first entry of its query]
    uint32_t *d_nb = ix->arena.take<uint32_t>(nq);
    uint32_t *d_head = ix->arena.take<uint32_t>(n);
    int64_t *d_hr = ix->arena.take<int64_t>(n + 1);
    void *d_stmp = ix->arena.take<char>(scan_tmp_bytes(n));
    SIA_REQUIRE(d_nb && d_head && d_hr && d_stmp, SIA_E_NOMEM, "index scratch arena too small (batches)");
    head_flags_kernel<<<grid_for(n), 256, 0, s>>>(Lk.ent, n, d_head);
    SIA_CHECK_LAUNCH();
    int rc = exclusive_scan_u32(d_head, d_hr, n, d_stmp, s);
    if (rc) return rc;
    query_batches_kernel<<<grid_for(nq), 256, 0, s>>>(d_hr, d_qs, i0, nq, B, d_nb, d_out_batches + q0);
    SIA_CHECK_LAUNCH();
    std::vector<uint32_t> h_nb(nq);
    SIA_CUDA(cudaMemcpyAsync(h_nb.data(), d_nb, sizeof(uint32_t) * nq, cudaMemcpyDeviceToHost, s));
    SIA_CUDA(cudaStreamSynchronize(s));
    std::vector<QMeta> h_meta(nq);
    // queries without matches are in no group: 0 results, out_batches = K_q, no exit
    for (const auto &[qa, qb] : split_groups(h_off_all, nq, p.budget, nullptr)) {
      const int gq = qb - qa;
      uint32_t k_max = 0;
      for (int q = qa; q < qb; ++q) if (h_off_all[q + 1] > h_off_all[q]) k_max = std::max(k_max, h_nb[q]);
      const Group g = make_group(qa, qb, h_off_all, h_off_head, (int64_t)ix->max_song + 1, h_meta.data());
      int64_t nb_slots = 0, nc = 0;
      for (int q = qa; q < qb; ++q) {
        QMeta &m = h_meta[q];
        const int64_t t = h_off_all[q + 1] - h_off_all[q], h = h_off_head[q + 1] - h_off_head[q];
        m.bin_base = nb_slots; m.bin_cap = (uint32_t)(2 * t + 32);
        m.cand_base = nc; m.cand = (uint32_t)std::min<int64_t>(m.song_cap, h + 1);   // a matched song has a head row
        m.cursor = 0;
        nb_slots += m.bin_cap; nc += m.cand;
      }
      const int64_t e0 = p.h_qs[qa] - i0, ne = p.h_qs[qb] - i0 - e0;
      const size_t bytes = (size_t)gq * (sizeof(QMeta) + 4 * 2 + 8 + 4 * 2 * L) + (size_t)nb_slots * 12 +
                           (size_t)g.ns * (8 + 4 + 4 + (g.dense ? 0 : 4)) + (size_t)nc * 4 + (size_t)ne * 4 +
                           (size_t)(k_max + 1) * (4 + 8) + scan_tmp_bytes(k_max) + 64 + (1 << 16);
      if ((rc = ix->arena3.reserve(bytes))) return rc;
      QMeta *d_meta = ix->arena3.take<QMeta>(gq);
      uint32_t *d_done = ix->arena3.take<uint32_t>(gq), *d_ntop = ix->arena3.take<uint32_t>(2 * (size_t)gq);
      uint32_t *d_top = ix->arena3.take<uint32_t>(2 * (size_t)gq * L);
      unsigned long long *d_stats = ix->arena3.take<unsigned long long>(2);   // tuples voted, head tuples (DB rows)
      int32_t *d_flags = ix->arena3.take<int32_t>(1);
      Tables T{};
      T.bins = ix->arena3.take<unsigned long long>(nb_slots);
      T.bin_cnt = ix->arena3.take<uint32_t>(nb_slots);
      T.song_best = ix->arena3.take<unsigned long long>(g.ns);
      T.song_key = g.dense ? nullptr : ix->arena3.take<uint32_t>(g.ns);
      uint32_t *d_rows = ix->arena3.take<uint32_t>(g.ns), *d_stamp = ix->arena3.take<uint32_t>(g.ns);
      uint32_t *d_chg = ix->arena3.take<uint32_t>(nc), *d_perm = ix->arena3.take<uint32_t>(ne);
      uint32_t *d_bcnt = ix->arena3.take<uint32_t>(k_max + 1);
      int64_t *d_boff = ix->arena3.take<int64_t>(k_max + 1);
      void *d_btmp = ix->arena3.take<char>(scan_tmp_bytes(k_max));
      SIA_REQUIRE(d_meta && d_done && d_ntop && d_top && d_stats && d_flags && T.bins && T.bin_cnt && T.song_best &&
                  (g.dense || T.song_key) && d_rows && d_stamp && d_chg && d_perm && d_bcnt && d_boff && d_btmp,
                  SIA_E_NOMEM, "index scratch arena too small (a-priori tables)");
      SIA_CUDA(cudaMemcpyAsync(d_meta, h_meta.data() + qa, sizeof(QMeta) * gq, cudaMemcpyHostToDevice, s));
      SIA_CUDA(cudaMemsetAsync(d_done, 0, sizeof(uint32_t) * gq, s));
      SIA_CUDA(cudaMemsetAsync(d_stats, 0, 2 * sizeof(unsigned long long), s));
      SIA_CUDA(cudaMemsetAsync(d_flags, 0, sizeof(int32_t), s));
      SIA_CUDA(cudaMemsetAsync(T.bins, 0, sizeof(unsigned long long) * nb_slots, s));
      SIA_CUDA(cudaMemsetAsync(T.bin_cnt, 0, sizeof(uint32_t) * nb_slots, s));
      SIA_CUDA(cudaMemsetAsync(T.song_best, 0, sizeof(unsigned long long) * g.ns, s));
      if (!g.dense) SIA_CUDA(cudaMemsetAsync(T.song_key, 0, sizeof(uint32_t) * g.ns, s));
      SIA_CUDA(cudaMemsetAsync(d_rows, 0, sizeof(uint32_t) * g.ns, s));
      SIA_CUDA(cudaMemsetAsync(d_stamp, 0, sizeof(uint32_t) * g.ns, s));
      SIA_CUDA(cudaMemsetAsync(d_bcnt, 0, sizeof(uint32_t) * (k_max + 1), s));
      // round k's entries: d_perm[d_boff[k] .. d_boff[k + 1])
      bucket_entries_kernel<false><<<grid_for(ne), 256, 0, s>>>(Lk.ent, Lk.off_all, d_hr, d_qs, i0, e0, ne, B, d_bcnt, nullptr, nullptr);
      SIA_CHECK_LAUNCH();
      if ((rc = exclusive_scan_u32(d_bcnt, d_boff, k_max, d_btmp, s))) return rc;
      SIA_CUDA(cudaMemsetAsync(d_bcnt, 0, sizeof(uint32_t) * (k_max + 1), s));
      bucket_entries_kernel<true><<<grid_for(ne), 256, 0, s>>>(Lk.ent, Lk.off_all, d_hr, d_qs, i0, e0, ne, B, d_bcnt, d_boff, d_perm);
      SIA_CHECK_LAUNCH();
      const unsigned dblocks = (unsigned)ceil_div(gq, 8);
      for (uint32_t k = 0; k < k_max; ++k) {
        if (g.dense) {
          round_vote_kernel<true><<<kRoundBlocks, 256, 0, s>>>((int)k, Lk.ent, e0, Lk.first, Lk.cnt_head, Lk.off_all, d_perm, d_boff, ix->post,
                                                              d_meta, (int)qa, T, d_rows, d_stamp, d_chg, d_done, d_stats, d_flags);
          round_decide_kernel<true><<<dblocks, 256, 0, s>>>((int)k, gq, (int)(q0 + qa), topn, L, d_meta, T, d_rows, d_chg, d_top, d_ntop,
                                                            d_done, d_nb + qa, d_out_song, d_out_diff, d_out_count, d_out_rows, d_out_nres,
                                                            d_out_batches, d_out_exit);
        } else {
          round_vote_kernel<false><<<kRoundBlocks, 256, 0, s>>>((int)k, Lk.ent, e0, Lk.first, Lk.cnt_head, Lk.off_all, d_perm, d_boff, ix->post,
                                                               d_meta, (int)qa, T, d_rows, d_stamp, d_chg, d_done, d_stats, d_flags);
          round_decide_kernel<false><<<dblocks, 256, 0, s>>>((int)k, gq, (int)(q0 + qa), topn, L, d_meta, T, d_rows, d_chg, d_top, d_ntop,
                                                             d_done, d_nb + qa, d_out_song, d_out_diff, d_out_count, d_out_rows, d_out_nres,
                                                             d_out_batches, d_out_exit);
        }
        SIA_CHECK_LAUNCH();
      }
      int32_t h_flags = 0;
      unsigned long long h_st[2] = {0, 0};
      SIA_CUDA(cudaMemcpyAsync(&h_flags, d_flags, sizeof h_flags, cudaMemcpyDeviceToHost, s));
      SIA_CUDA(cudaMemcpyAsync(h_st, d_stats, sizeof h_st, cudaMemcpyDeviceToHost, s));
      SIA_CUDA(cudaStreamSynchronize(s));      // the tables are reused by the next group
      SIA_REQUIRE(!(h_flags & 8), SIA_E_CUDA, "query_apriori: vote table overflow (internal error)");
      if (h_stats) { h_stats[2] += (int64_t)h_st[0]; h_stats[1] += (int64_t)h_st[1]; }
    }
    std::vector<int32_t> h_batches(nq);
    SIA_CUDA(cudaMemcpyAsync(h_batches.data(), d_out_batches + q0, sizeof(int32_t) * nq, cudaMemcpyDeviceToHost, s));
    SIA_CUDA(cudaStreamSynchronize(s));
    if (h_stats) for (int32_t b : h_batches) h_stats[3] += b;
    return SIA_OK;
  };
  return query_passes(ix, d_hash, d_qoff, h_query_starts, n_queries, topn, out, h_stats, (cudaStream_t)stream, false,
                      [](int nq, int64_t n) { return (size_t)nq * 4 + (size_t)n * (4 + 8) + scan_tmp_bytes(n); }, vote);
}
