// K4, the partitioned vote — align_matches' histogram (recognizer.py:303-310) counted in SHARED memory.
//
// The table vote of index_query.cu counts every (query, song, diff) tuple with atomics on tables that live in HBM:
// a random 32-byte sector per tuple and pass.  Here the tuples of a query are first split by a hash of the BIN
// (song, diff) into partitions of ~10 240 tuples (regions of at most 24 576 slots), so that each partition's repeated
// bins fit a duplicate filter + a small exact table in shared memory:
//
//   scatter  one CTA per block of 8 192 consecutive tuples of ONE query (posting runs walked entry by entry, or a slice
//            of received vote keys): tuple -> (song 24 | diff 25 | head 1), partition = hi16(hash(song, diff)) * np >> 16,
//            counted in a shared histogram, sorted by partition through a shared staging buffer, and written as one
//            contiguous run per partition into the (query, partition) region (one global atomicAdd per block and
//            partition reserves the room; with peer memory the region lives in the query owner's HBM);
//   count    one CTA per region, two passes over its tuples: a 2-bit duplicate filter marks the buckets hit twice, then
//            only the tuples of those buckets go to an exact open-addressing table (one 64-bit word per slot =
//            key 49 | count 15; CAS to claim, 32-bit add to bump); bins that reach count 2 are remembered in a list; the
//            region's top-n songs by (count desc, song asc), per song the largest bin, smallest diff on ties, come
//            from that list (or from a scan of the tuples when fewer than n songs have a repeated bin);
//   merge    one warp per query: top-n over its regions' candidates.  A BIN lives in exactly one partition, so its
//            count is exact; a song's bins are spread over the partitions, so the merge keeps a song's first (= best)
//            occurrence in descending order and skips the later ones.
// All traffic is streaming: 8 B read + 8 B written per tuple (scatter), 8 B read (count; the second pass hits L2).
// Queries that do not fit — one BIN above a region's capacity, more than 4 096 partitions — are flagged and voted by
// the table vote instead; nothing is approximated.
#include "index.cuh"

using namespace sia;

namespace {

constexpr int kDiffBits = SIA_KEY_DIFF_BITS, kSongBits = SIA_KEY_SONG_BITS, kQidBits = SIA_KEY_QID_BITS;
constexpr uint64_t kDiffMask = (1ull << kDiffBits) - 1;

constexpr int kBlk = 8192;            // tuples per scatter block
constexpr int kScThreads = 512;
constexpr int kTpt = kBlk / kScThreads;
constexpr int kCap = 24576;           // tuples a region can hold (a 15-bit count per bin; room for one heavy bin next to the average)
constexpr int kAvg = 10240;           // tuples per partition the layout aims at
constexpr int kMaxParts = 4096;         // partitions of one query (a query of more than ~4096 * 10240 tuples goes to the table vote)
constexpr int kFiltWords = 8192;      // count kernel: duplicate filter, 2 bits per bucket, 16 buckets per word (32 KB)
constexpr int kTabSlots = 4096;       // count kernel: exact table of the tuples in twice-hit buckets (32 KB)
constexpr int kDup = 2048;            // repeated bins a region remembers
constexpr int kCntThreads = 512;
constexpr int kRegionsPerCta = 1;
constexpr size_t kCountSmem = (size_t)kFiltWords * 4 + (size_t)kTabSlots * 8;

struct PvQuery {
  int64_t reg_off;                    // first tuple slot of the query's regions
  uint32_t ridx0, np, cap, nt;        // first region index, partitions, tuple slots per region, tuples
};

struct PvTune { uint32_t cap, avg; };

PvTune pv_tune() {
  PvTune v{kCap, kAvg};
  if (const char *e = getenv("SIA_PVOTE_CAP")) {            // tests: small regions force the fallback to the table vote
    const long c = atol(e);
    if (c >= 2 && c <= kCap) { v.cap = (uint32_t)c & ~1u; v.avg = std::max(1u, (uint32_t)(v.cap * 7ull / 12)); }
  }
  return v;
}

__host__ __device__ inline uint32_t pv_parts(uint64_t t, uint32_t cap, uint32_t avg) {
  if (t <= cap) return 1;
  const uint64_t n = (t + avg - 1) / avg;
  return n > (uint64_t)kMaxParts ? (uint32_t)kMaxParts : (uint32_t)n;
}
__host__ __device__ inline uint32_t pv_region_cap(uint64_t t, uint32_t cap) {
  return t <= cap ? (uint32_t)((t + 1) & ~1ull) : cap;        // a single region holds exactly its query
}

__device__ __forceinline__ uint32_t mix32(uint32_t k) {
  k ^= k >> 16; k *= 0x85ebca6bu; k ^= k >> 13; k *= 0xc2b2ae35u; k ^= k >> 16;
  return k;
}
// partition of a bin (song, biased diff): multiplicative hash, top 16 bits scaled to np.  Partitioning by BIN (not by
// song) spreads a song with tens of thousands of tuples (a long query against its own track) over all partitions.
__device__ __forceinline__ uint32_t pv_part(uint32_t song, uint32_t dbits, uint32_t np) {
  return (((song * 0x9e3779b1u + dbits * 0x7feb352du) >> 16) * np) >> 16;
}

// largest i in [lo, hi) with a[i] <= x, given a[lo] <= x and a non-decreasing; the 32 lanes of a warp call it with the
// same arguments and probe 32 positions per round (3 dependent loads for 2 000 elements instead of 11)
template <typename T, typename X>
__device__ __forceinline__ int64_t warp_search(const T *__restrict__ a, int64_t lo, int64_t hi, X x, int lane) {
  while (hi - lo > 1) {
    const int64_t step = (hi - lo + 31) >> 5;
    const int64_t pos = lo + (int64_t)(lane + 1) * step;
    const bool le = pos < hi && (X)a[pos] <= x;
    const int c = __popc(__ballot_sync(0xffffffffu, le));
    lo += (int64_t)c * step;
    hi = min(hi, lo + step);
  }
  return lo;
}

// ---- layout ---------------------------------------------------------------------------------------------------
// segments: (query, source) -> a range of tuples / keys.  Entries variant: one source, the query's slice of off_all.
// il_world > 0 (peer scatter): segment j is the query of owner (j + il_rank) % il_world, slot j / il_world — consecutive
// blocks go to different owners and every shard starts with a different one, so no owner's NVLink ingress is the
// target of all shards at once
__device__ __forceinline__ int pv_seg_query(int j, int il_world, int il_rank, int qp) {
  return il_world > 0 ? ((j + il_rank) % il_world) * qp + j / il_world : j;
}
__global__ void pv_segs_entries_kernel(const int64_t *__restrict__ goff, int qa, int nq, int64_t *__restrict__ seg_lo,
                                       uint32_t *__restrict__ seg_cnt, int il_world, int il_rank, int qp) {
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < nq; j += gridDim.x * blockDim.x) {
    const int q = pv_seg_query(j, il_world, il_rank, qp);
    seg_lo[j] = goff[qa + q];
    seg_cnt[j] = (uint32_t)(goff[qa + q + 1] - goff[qa + q]);
  }
}

// per entry what the scatter walk needs, in two loads: {end of the entry's tuples, first posting - first tuple} and
// query offset << 1 | head
__global__ void __launch_bounds__(256)
pv_entry_info_kernel(const ulonglong2 *__restrict__ ent, const int64_t *__restrict__ first, const int64_t *__restrict__ off,
                     const uint32_t *__restrict__ cnt_head, int64_t n, longlong2 *__restrict__ info, uint32_t *__restrict__ qh) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    info[e] = make_longlong2(off[e + 1], first[e] - off[e]);
    qh[e] = ((uint32_t)(ent[e].x & kM24) << 1) | (cnt_head[e] != 0 ? 1u : 0u);
  }
}

// keys variant: slot g sorted by query id -> boundaries by binary search; anything inconsistent sets *unsorted
__global__ void pv_segs_keys_kernel(const uint64_t *__restrict__ keys, int64_t cap, const int64_t *__restrict__ counts, int G,
                                    int nq, int64_t *__restrict__ seg_lo, uint32_t *__restrict__ seg_cnt,
                                    uint32_t *__restrict__ unsorted) {
  const uint32_t qmask = (1u << kQidBits) - 1u;
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < nq * G; s += gridDim.x * blockDim.x) {
    const int q = s / G, g = s - q * G;
    int64_t n;
    const uint64_t *__restrict__ kk = slot_keys(keys, cap, counts, g, n);
    int64_t b[2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const uint32_t want = (uint32_t)(q + h);
      int64_t lo = 0, hi = n;
      if (want == 0) hi = 0;
      else if (want >= (uint32_t)nq) lo = n;
      while (lo < hi) {
        const int64_t mid = lo + ((hi - lo) >> 1);
        if (((uint32_t)(kk[mid] >> (kSongBits + kDiffBits)) & qmask) < want) lo = mid + 1; else hi = mid;
      }
      b[h] = lo;
    }
    if (b[1] < b[0] || b[1] - b[0] > 0xffffffffll) { atomicOr(unsorted, 1u); b[1] = b[0]; }
    seg_lo[s] = b[0];
    seg_cnt[s] = (uint32_t)(b[1] - b[0]);
  }
}

// single block: per query partitions / region offsets, per segment first scatter block; tot = {regions, blocks}
__global__ void __launch_bounds__(1024)
pv_layout_kernel(const uint32_t *__restrict__ seg_cnt, int nq, int G, PvTune tune, PvQuery *__restrict__ pq,
                 uint32_t *__restrict__ q_ridx0, uint32_t *__restrict__ seg_blk0, uint32_t *__restrict__ tot) {
  __shared__ int64_t s_reg[1024];
  __shared__ uint32_t s_idx[1024], s_blk[1024];
  const int per = (nq + 1023) / 1024;
  const int a = min(nq, (int)threadIdx.x * per), b = min(nq, a + per);
  int64_t reg = 0;
  uint32_t idx = 0, blk = 0;
  for (int q = a; q < b; ++q) {
    uint64_t t = 0;
    for (int g = 0; g < G; ++g) { const uint32_t c = seg_cnt[q * G + g]; t += c; blk += (c + kBlk - 1) / kBlk; }
    const uint32_t np = t ? pv_parts(t, tune.cap, tune.avg) : 0;
    idx += np;
    reg += (int64_t)np * pv_region_cap(t, tune.cap);
  }
  s_reg[threadIdx.x] = reg; s_idx[threadIdx.x] = idx; s_blk[threadIdx.x] = blk;
  __syncthreads();
  if (threadIdx.x == 0) {
    int64_t r = 0; uint32_t i = 0, k = 0;
    for (int j = 0; j < 1024; ++j) {
      const int64_t x = s_reg[j]; const uint32_t y = s_idx[j], z = s_blk[j];
      s_reg[j] = r; s_idx[j] = i; s_blk[j] = k;
      r += x; i += y; k += z;
    }
    tot[0] = i; tot[1] = k; tot[2] = 0; tot[3] = 0;
    q_ridx0[nq] = i; seg_blk0[nq * G] = k;
  }
  __syncthreads();
  reg = s_reg[threadIdx.x]; idx = s_idx[threadIdx.x]; blk = s_blk[threadIdx.x];
  for (int q = a; q < b; ++q) {
    uint64_t t = 0;
    for (int g = 0; g < G; ++g) {
      const uint32_t c = seg_cnt[q * G + g];
      seg_blk0[q * G + g] = blk;
      t += c; blk += (c + kBlk - 1) / kBlk;
    }
    PvQuery m;
    m.np = t ? pv_parts(t, tune.cap, tune.avg) : 0;
    m.cap = pv_region_cap(t, tune.cap);
    m.nt = (uint32_t)min(t, (uint64_t)0xffffffffu);
    m.reg_off = reg; m.ridx0 = idx;
    pq[q] = m;
    q_ridx0[q] = idx;
    idx += m.np; reg += (int64_t)m.np * m.cap;
  }
}

// scatter block -> segment and region -> query, so that the big kernels start with one load instead of a search
__global__ void __launch_bounds__(256)
pv_maps_kernel(const uint32_t *__restrict__ seg_blk0, int n_seg, const uint32_t *__restrict__ q_ridx0, int nq,
               const uint32_t *__restrict__ tot, uint32_t *__restrict__ blk_seg, uint32_t *__restrict__ reg_q) {
  const uint32_t n_reg = tot[0], n_blk = tot[1];
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_reg + n_blk; i += gridDim.x * blockDim.x) {
    if (i < n_blk) blk_seg[i] = (uint32_t)find_segment(seg_blk0, n_seg, i);
    else reg_q[i - n_blk] = (uint32_t)find_segment(q_ridx0, nq, i - n_blk);
  }
}

// ---- scatter --------------------------------------------------------------------------------------------------
struct ScatterArgs {
  const uint32_t *seg_blk0, *blk_seg; const int64_t *seg_lo; const uint32_t *seg_cnt; int G;
  const PvQuery *pq; const uint32_t *tot;
  uint64_t *regions; uint32_t *fill; uint32_t *qover; int q_lo;
  int maxp;                             // partitions the shared histogram is laid out for (>= every np of the launch)
  // hash-prefix sharding over peer memory: query ql belongs to rank ql / qp_dest, whose regions / counters are written
  // through NVLink (qp_dest = 0: everything is local)
  int qp_dest, il_rank, il_world;
  uint64_t *regions_p[kPvMaxPeers]; uint32_t *fill_p[kPvMaxPeers]; uint32_t *qover_p[kPvMaxPeers];
  // source 0: posting runs of the query's entries
  const int64_t *off; const longlong2 *info; const uint32_t *qh; const uint64_t *post;
  const int64_t *q_ent; int64_t i0;
  // source 1: vote keys in slots
  const uint64_t *keys; int64_t key_cap; const int64_t *counts; uint32_t *unsorted;
};

constexpr size_t scatter_smem(int maxp) { return (size_t)kBlk * 8 + (size_t)kBlk * 2 + (size_t)(2 * maxp + 1) * 4; }
constexpr size_t kScatterSmem = scatter_smem(kMaxParts);

__device__ __forceinline__ void cp_async8(uint32_t dst, const void *src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(dst), "l"(src) : "memory");
}

template <int SRC>
__global__ void __launch_bounds__(kScThreads, 2) pv_scatter_kernel(const ScatterArgs a) {
  extern __shared__ __align__(16) unsigned char pv_smem[];
  uint64_t *stage = reinterpret_cast<uint64_t *>(pv_smem);              // [kBlk] tuples in arrival order
  uint16_t *idx = reinterpret_cast<uint16_t *>(stage + kBlk);            // [kBlk] arrival index of the t-th tuple in partition order
  uint32_t *hist = reinterpret_cast<uint32_t *>(idx + kBlk);             // [np + 1] counts, then exclusive offsets
  int32_t *gdst = reinterpret_cast<int32_t *>(hist + a.maxp + 1);        // [np] region slot of partition order position 0
  __shared__ uint32_t s_warp[kScThreads / 32];
  const uint32_t b = blockIdx.x;
  if (b >= a.tot[1]) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int s = (int)a.blk_seg[b];
  const int ql = a.qp_dest > 0 ? pv_seg_query(s, a.il_world, a.il_rank, a.qp_dest) : s / a.G;
  const int g = a.qp_dest > 0 ? 0 : s - ql * a.G;
  const PvQuery m = a.pq[ql];
  const int64_t lo = a.seg_lo[s];
  const int64_t j0 = lo + (int64_t)(b - a.seg_blk0[s]) * kBlk;
  const int n = (int)min((int64_t)kBlk, lo + (int64_t)a.seg_cnt[s] - j0);
  const uint32_t np = m.np;
  uint64_t *regions_d = a.regions;
  uint32_t *fill_d = a.fill, *qover_d = a.qover + a.q_lo + ql;
  if (a.qp_dest > 0) {
    const int d = ql / a.qp_dest;
    regions_d = a.regions_p[d]; fill_d = a.fill_p[d]; qover_d = a.qover_p[d] + (ql - d * a.qp_dest);
  }
  for (uint32_t p = tid; p <= np; p += kScThreads) hist[p] = 0;

  uint32_t pr[kTpt];                       // first the entry's (query offset, head), then partition << 13 | rank
  const int iw = warp * (kBlk / (kScThreads / 32));
  const uint32_t stage_s = (uint32_t)__cvta_generic_to_shared(stage);
  // the raw postings / keys of the block go straight to the staging buffer (cp.async: all 16 loads of a thread in flight)
  if (SRC == 0) {
    if (iw < n) {
      // entry of the warp's first tuple, then every lane walks on from there by itself
      int64_t e = warp_search(a.off, a.q_ent[a.q_lo + ql] - a.i0, a.q_ent[a.q_lo + ql + 1] - a.i0, j0 + iw, lane);
      longlong2 inf = a.info[e];
      uint32_t qh = a.qh[e];
#pragma unroll
      for (int k = 0; k < kTpt; ++k) {
        const int i = iw + k * 32 + lane;
        pr[k] = 0;
        if (i < n) {
          const int64_t j = j0 + i;
          if (inf.x <= j) {
            do { ++e; inf = a.info[e]; } while (inf.x <= j);
            qh = a.qh[e];
          }
          cp_async8(stage_s + (uint32_t)i * 8u, a.post + inf.y + j);
          pr[k] = qh;
        }
      }
    }
  } else {
    int64_t nk;
    const uint64_t *__restrict__ kk = slot_keys(a.keys, a.key_cap, a.counts, g, nk);
#pragma unroll
    for (int k = 0; k < kTpt; ++k) {
      const int i = iw + k * 32 + lane;
      if (i < n) cp_async8(stage_s + (uint32_t)i * 8u, kk + j0 + i);
    }
  }
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
  __syncthreads();                         // the histogram is zero (every thread reads only its own staged words)
  bool bad = false;
#pragma unroll
  for (int k = 0; k < kTpt; ++k) {
    const int i = iw + k * 32 + lane;
    if (i < n) {
      const uint64_t r = stage[i];
      uint32_t song, dbits;
      uint64_t tup;
      if (SRC == 0) {
        song = (uint32_t)(r >> 24) & 0xffffffu;
        dbits = ((uint32_t)(r & kM24) - (pr[k] >> 1) + SIA_DIFF_BIAS) & (uint32_t)kDiffMask;
        tup = ((uint64_t)song << (kDiffBits + 1)) | ((uint64_t)dbits << 1) | (pr[k] & 1u);
      } else {
        bad = bad || ((uint32_t)(r >> (kSongBits + kDiffBits)) & ((1u << kQidBits) - 1u)) != (uint32_t)ql;
        song = (uint32_t)(r >> kDiffBits) & 0xffffffu;
        dbits = (uint32_t)(r & kDiffMask);
        tup = ((uint64_t)song << (kDiffBits + 1)) | ((uint64_t)dbits << 1) | (r >> 63);
      }
      const uint32_t p = pv_part(song, dbits, np);
      const uint32_t rk = atomicAdd(&hist[p], 1u);
      stage[i] = tup;
      pr[k] = (p << 13) | rk;
    }
  }
  if (SRC == 1 && bad) atomicOr(a.unsorted, 1u);
  __syncthreads();

  // exclusive scan of the histogram (kPpt consecutive partitions per thread), room reserved in the regions
  constexpr int kPpt = kMaxParts / kScThreads;
  static_assert(kPpt * kScThreads == kMaxParts && kMaxParts <= (1 << 19), "partition / rank packing");
  if (np <= (uint32_t)kScThreads) {                    // the usual case: one partition per thread
    const uint32_t pme = (uint32_t)tid;
    const uint32_t c = pme < np ? hist[pme] : 0u;
    uint32_t inc = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      const uint32_t w = lane < kScThreads / 32 ? s_warp[lane] : 0u;
      uint32_t winc = w;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, winc, d); if (lane >= d) winc += t; }
      if (lane < kScThreads / 32) s_warp[lane] = winc - w;
    }
    __syncthreads();
    if (pme < np) {
      const uint32_t base = s_warp[warp] + inc - c;
      hist[pme] = base;
      int32_t d = INT32_MIN;
      if (c) {
        const uint32_t old = atomicAdd(&fill_d[m.ridx0 + pme], c);
        if (old + c <= m.cap) d = (int32_t)(pme * m.cap + old) - (int32_t)base;
        else *qover_d = 1u;
      }
      gdst[pme] = d;
    }
  } else {
    const uint32_t p0 = (uint32_t)tid * kPpt;
    uint32_t v[kPpt], sum = 0;
#pragma unroll
    for (int u = 0; u < kPpt; ++u) { v[u] = p0 + u < np ? hist[p0 + u] : 0u; sum += v[u]; }
    uint32_t inc = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      const uint32_t w = lane < kScThreads / 32 ? s_warp[lane] : 0u;
      uint32_t winc = w;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, winc, d); if (lane >= d) winc += t; }
      if (lane < kScThreads / 32) s_warp[lane] = winc - w;
    }
    __syncthreads();
    uint32_t base = s_warp[warp] + inc - sum;
#pragma unroll
    for (int u = 0; u < kPpt; ++u) {
      if (p0 + u < np) {
        const uint32_t c = v[u];
        hist[p0 + u] = base;
        int32_t d = INT32_MIN;
        if (c) {
          const uint32_t old = atomicAdd(&fill_d[m.ridx0 + p0 + u], c);
          if (old + c <= m.cap) d = (int32_t)((p0 + u) * m.cap + old) - (int32_t)base;
          else *qover_d = 1u;
        }
        gdst[p0 + u] = d;
        base += c;
      }
    }
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < kTpt; ++k) {
    const int i = iw + k * 32 + lane;
    if (i < n) idx[hist[pr[k] >> 13] + (pr[k] & 8191u)] = (uint16_t)i;
  }
  __syncthreads();
  uint64_t *__restrict__ reg = regions_d + m.reg_off;
  for (int t = tid; t < n; t += kScThreads) {
    const uint64_t tup = stage[idx[t]];
    const int32_t d = gdst[pv_part((uint32_t)(tup >> (kDiffBits + 1)), (uint32_t)(tup >> 1) & (uint32_t)kDiffMask, np)];
    if (d != INT32_MIN) reg[(int64_t)d + t] = tup;
  }
}

// ---- count ----------------------------------------------------------------------------------------------------
// exact-table slot word: (song 24 | diff 25) << 15 | count 15
__device__ __forceinline__ uint64_t pv_rank(uint64_t slot) {          // count desc, song asc, diff asc as ONE maximum
  if (slot == 0ull) return 0ull;
  const uint64_t key = slot >> 15;
  return ((slot & 0x7fffull) << 49) | ((kM24 - (key >> kDiffBits)) << kDiffBits) | (kDiffMask - (key & kDiffMask));
}
__device__ __forceinline__ uint64_t pv_rank1(uint64_t key) {          // the same for a bin of count 1
  return (1ull << 49) | ((kM24 - (key >> kDiffBits)) << kDiffBits) | (kDiffMask - (key & kDiffMask));
}
// bucket of a (song, diff) key in the duplicate filter / its slot hash in the exact table
__device__ __forceinline__ uint32_t pv_hash(uint64_t key) { return (uint32_t)(key >> kDiffBits) * 0x85ebca6bu + (uint32_t)key * 0xc2b2ae35u; }

// One CTA per region, two passes over its tuples (the second one reads them from L2):
//   mark   every tuple sets the "seen" bit of its bucket in a 2-bit duplicate filter (one atomicOr, no probing, no
//          divergence); an arrival in a bucket already seen sets "twice";
//   count  tuples of twice-hit buckets — every bin of count >= 2 is among them, plus the false positives of the filter
//          (~10 %) — are counted exactly in a small open-addressing table; all other tuples are bins of count 1 and
//          touch nothing;
//   top-n  by one warp from the bins that reached count 2; if fewer than topn songs have one, the bins of count 1
//          decide: the CTA scans the tuples themselves.
__device__ __forceinline__ void
pv_count_region(const uint32_t r, const uint64_t *__restrict__ regions, const uint32_t *__restrict__ fill,
                const PvQuery *__restrict__ pq, const uint32_t *__restrict__ reg_q, int q_lo, uint32_t *__restrict__ qover, int topn,
                uint64_t *__restrict__ cand, uint32_t *__restrict__ qbins) {
  extern __shared__ __align__(16) unsigned char pv_smem[];
  uint32_t *filt = reinterpret_cast<uint32_t *>(pv_smem);
  uint64_t *tab = reinterpret_cast<uint64_t *>(pv_smem + (size_t)kFiltWords * 4);
  __shared__ uint16_t s_dup[kDup];
  __shared__ uint32_t s_ndup, s_over;
  __shared__ uint64_t s_lw[kCntThreads / 32 + 1][kPvMaxTopn];       // per-warp winners; last row: the running winners
  __shared__ int s_nres;
  __shared__ uint64_t s_win[kPvMaxTopn];
  __shared__ uint64_t s_red[kCntThreads / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t n = fill[r];
  const int ql = (int)reg_q[r];
  const PvQuery m = pq[ql];
  const uint32_t p = r - m.ridx0;
  uint64_t *__restrict__ out = cand + (int64_t)r * topn;
  if (n == 0 || n > m.cap || qover[q_lo + ql]) {
    if (tid < topn) out[tid] = 0ull;
    return;
  }
  // filter: >= 8 buckets per tuple up to 2^17 buckets; table: every tuple fits while n <= 2048, else 4096 slots
  int fb = 10;
  while ((1u << fb) < 8 * n && fb < 17) ++fb;
  int tb = 6;
  while ((1u << tb) < 2 * n && tb < 12) ++tb;
  const uint32_t nw = 1u << (fb - 4), S = 1u << tb, tmask = S - 1;
  for (uint32_t i = tid; i < nw / 4; i += kCntThreads) reinterpret_cast<uint4 *>(filt)[i] = make_uint4(0u, 0u, 0u, 0u);
  for (uint32_t i = tid; i < S / 2; i += kCntThreads) reinterpret_cast<ulonglong2 *>(tab)[i] = make_ulonglong2(0ull, 0ull);
  if (tid == 0) { s_ndup = 0; s_over = 0; }
  const uint64_t *__restrict__ reg = regions + m.reg_off + (int64_t)p * m.cap;
  __syncthreads();
  // ---- mark ----
  for (uint32_t i0 = tid; i0 < n; i0 += 4 * kCntThreads) {
    uint64_t t[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) { const uint32_t i = i0 + u * kCntThreads; t[u] = i < n ? reg[i] : 0ull; }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (i0 + u * kCntThreads < n) {
        const uint32_t hb = pv_hash(t[u] >> 1) >> (32 - fb);
        const uint32_t seen = 1u << (2 * (hb & 15u));
        uint32_t *w = filt + (hb >> 4);
        const uint32_t old = atomicOr(w, seen);
        if ((old & (3u * seen)) == seen) atomicOr(w, seen << 1);        // second arrival: the bucket is hit twice
      }
    }
  }
  __syncthreads();
  // ---- count ----
  // The exact table holds ~3 300 distinct candidate keys.  A tie-heavy region (a long query against a self-similar
  // track) has more: its candidates are then counted in nsub sub-passes, each taking the keys of one residue class and
  // re-reading the tuples from L2; the running winners ride along.  nsub starts at 1 and doubles while a sub-pass
  // overflows, so the kernel cannot fail for a region that fits its slots.
  uint32_t nsub = 1;
  uint32_t fresh = 0;
  for (;;) {
    bool ok = true;
    fresh = 0;
    if (tid < kPvMaxTopn) s_lw[kCntThreads / 32][tid] = 0ull;          // the running winners of this attempt
    for (uint32_t sub = 0; sub < nsub; ++sub) {
      if (nsub > 1 || sub > 0) {
        __syncthreads();                                                 // the table of the previous sub-pass has been read
        for (uint32_t i = tid; i < S / 2; i += kCntThreads) reinterpret_cast<ulonglong2 *>(tab)[i] = make_ulonglong2(0ull, 0ull);
        if (tid == 0) { s_ndup = 0; s_over = 0; }
        __syncthreads();
      }
      for (uint32_t i0 = tid; i0 < n; i0 += 4 * kCntThreads) {
        uint64_t t[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) { const uint32_t i = i0 + u * kCntThreads; t[u] = i < n ? __ldcs(reg + i) : 0ull; }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (i0 + u * kCntThreads < n) {
            const uint64_t key = t[u] >> 1;
            const uint32_t hx = pv_hash(key), hb = hx >> (32 - fb);
            if (!(filt[hb >> 4] & (2u << (2 * (hb & 15u))))) { fresh += sub == 0; continue; }   // alone in its bucket: a bin of count 1
            if (((hx >> 3) & (nsub - 1)) != sub) continue;
            uint32_t h = mix32(hx) & tmask;
            for (uint32_t probes = 0;; ++probes) {
              if (probes == S) { s_over = 1u; break; }                  // the table is full
              const uint64_t cur = atomicCAS(reinterpret_cast<unsigned long long *>(tab + h), 0ull, (unsigned long long)((key << 15) | 1ull));
              if (cur == 0ull) { ++fresh; break; }
              if ((cur >> 15) == key) {
                const uint32_t old = atomicAdd(reinterpret_cast<uint32_t *>(tab + h), 1u);      // low word: key bits | count
                if ((old & 0x7fffu) == 1u) { const uint32_t d = atomicAdd(&s_ndup, 1u); if (d < (uint32_t)kDup) s_dup[d] = (uint16_t)h; }
                break;
              }
              h = (h + 1) & tmask;
            }
          }
        }
      }
      __syncthreads();
      if (s_ndup > (uint32_t)kDup || s_over) { ok = false; break; }
      // top-n songs from the bins that reached count 2: every warp ranks its share of the list (distinct songs), warp 0
      // merges the 16 x topn survivors and the running winners — the first occurrence of a song in descending order is
      // its best bin
      {
        const uint32_t nd = s_ndup;
        uint64_t *lw = s_lw[warp];
        int nl = 0;
        while (nl < topn) {
          uint64_t best = 0;
          for (uint32_t k = tid; k < nd; k += kCntThreads) {
            uint64_t c = pv_rank(tab[s_dup[k]]);
            if (c > best) {
              const uint64_t song = (c >> kDiffBits) & kM24;
              for (int w = 0; w < nl; ++w) if (((lw[w] >> kDiffBits) & kM24) == song) c = 0;
              if (c > best) best = c;
            }
          }
#pragma unroll
          for (int d = 16; d; d >>= 1) { const uint64_t o = __shfl_xor_sync(0xffffffffu, best, d); if (o > best) best = o; }
          if (best == 0ull) break;
          if (lane == 0) lw[nl] = best;
          ++nl;
          __syncwarp();
        }
        if (lane == 0) for (int w = nl; w < topn; ++w) lw[w] = 0ull;
      }
      __syncthreads();
      if (warp == 0) {
        const uint32_t total = (kCntThreads / 32 + 1) * (uint32_t)topn;
        int nres = 0;
        while (nres < topn) {
          uint64_t best = 0;
          for (uint32_t k = lane; k < total; k += 32) {
            uint64_t c = s_lw[k / (uint32_t)topn][k % (uint32_t)topn];
            if (c > best) {
              const uint64_t song = (c >> kDiffBits) & kM24;
              for (int w = 0; w < nres; ++w) if (((s_win[w] >> kDiffBits) & kM24) == song) c = 0;
              if (c > best) best = c;
            }
          }
#pragma unroll
          for (int d = 16; d; d >>= 1) { const uint64_t o = __shfl_xor_sync(0xffffffffu, best, d); if (o > best) best = o; }
          if (best == 0ull) break;
          if (lane == 0) s_win[nres] = best;
          ++nres;
          __syncwarp();
        }
        if (lane < topn) s_lw[kCntThreads / 32][lane] = lane < nres ? s_win[lane] : 0ull;
        if (lane == 0) s_nres = nres;
      }
    }
    if (ok) break;
    if (nsub >= 16) {                                                    // cannot happen for n <= 24576 (16 x 3328 keys); kept as a guard
      if (tid == 0) qover[q_lo + ql] = 1u;
      if (tid < topn) out[tid] = 0ull;
      return;
    }
    nsub <<= 1;
  }
  if (qbins) {
#pragma unroll
    for (int d = 16; d; d >>= 1) fresh += __shfl_xor_sync(0xffffffffu, fresh, d);
    if (lane == 0 && fresh) atomicAdd(&qbins[q_lo + ql], fresh);
  }
  __syncthreads();
  int nres = s_nres;
  // fewer than topn songs with a repeated bin: the remaining songs all rank by a bin of count 1 — (song asc, diff asc)
  // over the tuples themselves, winners' songs excluded (rare on a large index, the normal case on a tiny one)
  while (nres < topn) {
    uint64_t best = 0;
    for (uint32_t k = tid; k < n; k += kCntThreads) {
      uint64_t c = pv_rank1(reg[k] >> 1);
      if (c > best) {
        const uint64_t song = (c >> kDiffBits) & kM24;
        for (int w = 0; w < nres; ++w) if (((s_win[w] >> kDiffBits) & kM24) == song) c = 0;
        if (c > best) best = c;
      }
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) { const uint64_t o = __shfl_xor_sync(0xffffffffu, best, d); if (o > best) best = o; }
    if (lane == 0) s_red[warp] = best;
    __syncthreads();
    best = 0;
#pragma unroll
    for (int w = 0; w < kCntThreads / 32; ++w) { const uint64_t o = s_red[w]; if (o > best) best = o; }
    if (best == 0ull) break;
    if (tid == 0) s_win[nres] = best;
    ++nres;
    __syncthreads();
  }
  if (tid < topn) out[tid] = tid < nres ? s_win[tid] : 0ull;
}

// CTAs take up to kRegionsPerCta regions each from a shared counter (tot[2]): the grid is 1/8 of the host-side bound of the
// (device-side) number of regions
__global__ void __launch_bounds__(kCntThreads, 3)
pv_count_kernel(const uint64_t *__restrict__ regions, const uint32_t *__restrict__ fill, const PvQuery *__restrict__ pq,
                const uint32_t *__restrict__ reg_q, uint32_t *__restrict__ tot, int q_lo, uint32_t *__restrict__ qover, int topn,
                uint64_t *__restrict__ cand, uint32_t *__restrict__ qbins) {
  __shared__ uint32_t s_next;
  const uint32_t n_regions = tot[0];
  for (int it = 0; it < kRegionsPerCta; ++it) {   // bounded: CTAs retire regularly, so kernels of other streams (NCCL) get SMs
    __syncthreads();                          // the previous region's shared state has been read
    if (threadIdx.x == 0) s_next = atomicAdd(&tot[2], 1u);
    __syncthreads();
    const uint32_t r = s_next;
    if (r >= n_regions) return;
    pv_count_region(r, regions, fill, pq, reg_q, q_lo, qover, topn, cand, qbins);
  }
}

// ---- merge ----------------------------------------------------------------------------------------------------
// one warp per query: top-n over its regions' candidates.  A song's bins are spread over the partitions, so the same
// song can come from several regions: in descending order its first occurrence is its best bin, later ones are skipped.
// (Exact: a song of the true top-n cannot be cut from its region's list, because the n songs ahead of it there each
// have a bin at least that good.)  out.rows is left 0: dedup_hashes is counted by the caller.
__global__ void __launch_bounds__(256)
pv_merge_kernel(const uint64_t *__restrict__ cand, const PvQuery *__restrict__ pq, int nq, int q_lo, int qid_base,
                const uint32_t *__restrict__ qover, int topn, PvOut out, uint32_t *__restrict__ over_count,
                const uint32_t *__restrict__ qbins, unsigned long long *__restrict__ n_bins) {
  const int lane = threadIdx.x & 31;
  const int ql = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  if (ql >= nq) return;
  const int q = q_lo + ql;
  if (qover[q]) { if (lane == 0 && over_count) atomicAdd(over_count, 1u); return; }
  if (lane == 0 && n_bins && qbins[q]) atomicAdd(n_bins, (unsigned long long)qbins[q]);   // distinct bins of the settled queries
  const PvQuery m = pq[ql];
  if (m.np == 0) return;                    // no tuples: the outputs are already zero
  const uint64_t *__restrict__ c = cand + (int64_t)m.ridx0 * topn;
  const uint32_t total = m.np * (uint32_t)topn;
  const int64_t obase = ((int64_t)q + qid_base) * topn;
  uint64_t prev = ~0ull;
  int nres = 0;
  while (nres < topn) {
    uint64_t best = 0;
    for (uint32_t i = lane; i < total; i += 32) { const uint64_t v = c[i]; if (v < prev && v > best) best = v; }
#pragma unroll
    for (int d = 16; d; d >>= 1) { const uint64_t o = __shfl_xor_sync(0xffffffffu, best, d); if (o > best) best = o; }
    if (best == 0ull) break;
    prev = best;
    const int32_t song = (int32_t)(kM24 - ((best >> kDiffBits) & kM24));
    bool taken = false;
    for (int w = 0; w < nres; ++w) taken = taken || out.song[obase + w] == song;
    if (taken) continue;                    // a lesser bin of a song that already has its place
    if (lane == 0) {
      out.song[obase + nres] = song;
      out.count[obase + nres] = (int32_t)(best >> 49);
      out.diff[obase + nres] = (int32_t)(kDiffMask - (best & kDiffMask)) - SIA_DIFF_BIAS;
      out.rows[obase + nres] = 0;
    }
    ++nres;
    __syncwarp();
  }
  if (lane == 0) out.nres[q + qid_base] = nres;
}

// dedup_hashes of the winners (recognizer.py:259-264) from the regions: one CTA per region counts the head tuples of
// its query's winning songs (the tuples of a song are spread over the query's regions)
__global__ void __launch_bounds__(256)
pv_rows_kernel(const uint64_t *__restrict__ regions, const uint32_t *__restrict__ fill, const PvQuery *__restrict__ pq,
               const uint32_t *__restrict__ reg_q, const uint32_t *__restrict__ tot, int q_lo, int qid_base,
               const uint32_t *__restrict__ qover, int topn, const int32_t *__restrict__ out_song,
               const int32_t *__restrict__ out_nres, int32_t *__restrict__ out_rows) {
  __shared__ uint32_t s_song[kPvMaxTopn], s_cnt[kPvMaxTopn];
  const uint32_t n_regions = tot[0];
  for (uint32_t r = blockIdx.x; r < n_regions; r += gridDim.x) {
    const int ql = (int)reg_q[r], q = q_lo + ql;
    const uint32_t n = fill[r];
    const int nres = out_nres[q + qid_base];
    const PvQuery m = pq[ql];
    if (n == 0 || nres == 0 || qover[q] || n > m.cap) continue;       // block-uniform
    const int64_t obase = ((int64_t)q + qid_base) * topn;
    __syncthreads();
    if ((int)threadIdx.x < nres) { s_song[threadIdx.x] = (uint32_t)out_song[obase + threadIdx.x]; s_cnt[threadIdx.x] = 0; }
    __syncthreads();
    const uint64_t *__restrict__ reg = regions + m.reg_off + (int64_t)(r - m.ridx0) * m.cap;
    for (uint32_t k = threadIdx.x; k < n; k += blockDim.x) {
      const uint64_t t = __ldcs(reg + k);
      if (t & 1ull) {
        const uint32_t song = (uint32_t)(t >> (kDiffBits + 1));
        for (int w = 0; w < nres; ++w) if (s_song[w] == song) atomicAdd(&s_cnt[w], 1u);
      }
    }
    __syncthreads();
    if ((int)threadIdx.x < nres && s_cnt[threadIdx.x]) atomicAdd(out_rows + obase + threadIdx.x, (int32_t)s_cnt[threadIdx.x]);
  }
}

// layout of every destination rank's queries from the TOTAL tuple counts (all shards): block d lays out the queries
// [d * qp, (d + 1) * qp) exactly as rank d does for itself, so senders and owner agree on every region without talking.
// dest_tot[2d] = regions, dest_tot[2d + 1] = tuple slots; an owner whose buffers are too small sets flag 4 in *info.
__global__ void __launch_bounds__(1024)
pv_layout_dest_kernel(const int64_t *__restrict__ t_total, int qp, PvTune tune, PvQuery *__restrict__ pq,
                      uint32_t *__restrict__ q_ridx0, int64_t *__restrict__ dest_tot, int64_t region_cap, int64_t fill_cap,
                      unsigned long long *__restrict__ info) {
  __shared__ int64_t s_reg[1024];
  __shared__ uint32_t s_idx[1024];
  const int d = blockIdx.x;
  const int64_t *__restrict__ tt = t_total + (int64_t)d * qp;
  PvQuery *__restrict__ pqd = pq + (int64_t)d * qp;
  const int per = (qp + 1023) / 1024;
  const int a = min(qp, (int)threadIdx.x * per), b = min(qp, a + per);
  int64_t reg = 0;
  uint32_t idx = 0;
  for (int q = a; q < b; ++q) {
    const uint64_t t = (uint64_t)tt[q];
    const uint32_t np = t ? pv_parts(t, tune.cap, tune.avg) : 0;
    idx += np;
    reg += (int64_t)np * pv_region_cap(t, tune.cap);
  }
  s_reg[threadIdx.x] = reg; s_idx[threadIdx.x] = idx;
  __syncthreads();
  if (threadIdx.x == 0) {
    int64_t r = 0; uint32_t i = 0;
    for (int j = 0; j < 1024; ++j) { const int64_t x = s_reg[j]; const uint32_t y = s_idx[j]; s_reg[j] = r; s_idx[j] = i; r += x; i += y; }
    dest_tot[2 * d] = i; dest_tot[2 * d + 1] = r;
    if (q_ridx0) q_ridx0[(int64_t)d * (qp + 1) + qp] = i;
    if (r > region_cap || (int64_t)i > fill_cap) atomicOr(info, 4ull);
    atomicMax(info + 3, (unsigned long long)r);
  }
  __syncthreads();
  reg = s_reg[threadIdx.x]; idx = s_idx[threadIdx.x];
  for (int q = a; q < b; ++q) {
    const uint64_t t = (uint64_t)tt[q];
    PvQuery m;
    m.np = t ? pv_parts(t, tune.cap, tune.avg) : 0;
    m.cap = pv_region_cap(t, tune.cap);
    m.nt = (uint32_t)min(t, (uint64_t)0xffffffffu);
    m.reg_off = reg; m.ridx0 = idx;
    pqd[q] = m;
    if (q_ridx0) q_ridx0[(int64_t)d * (qp + 1) + q] = idx;
    idx += m.np; reg += (int64_t)m.np * m.cap;
  }
}

// a pass whose regions do not fit some owner's buffers is not scattered / counted at all (every rank sees the same flag)
__global__ void pv_gate_kernel(const unsigned long long *__restrict__ info, uint32_t *__restrict__ tot, int which) {
  if (*info & 4ull) tot[which] = 0;
}
__global__ void pv_set_regions_kernel(const int64_t *__restrict__ dest_tot, uint32_t *__restrict__ tot) {
  tot[0] = (uint32_t)dest_tot[0]; tot[1] = 0; tot[2] = 0; tot[3] = 0;
}
__global__ void pv_blocks_only_kernel(const uint32_t *__restrict__ tot, uint32_t *__restrict__ tot2) { tot2[0] = 0; tot2[1] = tot[1]; }

struct PvScratch {
  int64_t *seg_lo; uint32_t *seg_cnt, *seg_blk0, *q_ridx0, *tot, *fill, *blk_seg, *reg_q;
  PvQuery *pq; uint64_t *regions, *cand;
};

size_t pv_scratch_bytes(int64_t n_seg, int64_t nq, int64_t regions, int64_t region_tuples, int64_t blocks, int topn) {
  return (size_t)n_seg * 16 + (size_t)(n_seg + nq + 2) * 4 + (size_t)nq * sizeof(PvQuery) + (size_t)regions * (8 + 8 * (size_t)topn) +
         (size_t)blocks * 4 + (size_t)region_tuples * 8 + 16 * 256 + 64;
}

bool pv_take(Arena &ar, PvScratch &S, int64_t n_seg, int64_t nq, int64_t regions, int64_t region_tuples, int64_t blocks, int topn) {
  S.seg_lo = ar.take<int64_t>(n_seg);
  S.seg_cnt = ar.take<uint32_t>(n_seg);
  S.seg_blk0 = ar.take<uint32_t>(n_seg + 1);
  S.q_ridx0 = ar.take<uint32_t>(nq + 1);
  S.tot = ar.take<uint32_t>(4);
  S.pq = ar.take<PvQuery>(nq);
  S.fill = ar.take<uint32_t>(regions);
  S.reg_q = ar.take<uint32_t>(regions);
  S.blk_seg = ar.take<uint32_t>(blocks);
  S.cand = ar.take<uint64_t>(regions * topn);
  S.regions = ar.take<uint64_t>(region_tuples);
  return S.seg_lo && S.seg_cnt && S.seg_blk0 && S.q_ridx0 && S.tot && S.pq && S.fill && S.reg_q && S.blk_seg && S.cand && S.regions;
}

int pv_attrs() {
  static bool done[64] = {false};
  int dev = 0;
  SIA_CUDA(cudaGetDevice(&dev));
  if (dev >= 0 && dev < 64 && done[dev]) return SIA_OK;
  SIA_CUDA(cudaFuncSetAttribute(pv_scatter_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kScatterSmem));
  SIA_CUDA(cudaFuncSetAttribute(pv_scatter_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kScatterSmem));
  SIA_CUDA(cudaFuncSetAttribute(pv_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCountSmem));
  if (dev >= 0 && dev < 64) done[dev] = true;
  return SIA_OK;
}

// worst case over all splits of `tuples` into nq queries: a query that fits one region takes its own size (rounded to 2),
// a larger one ceil(t / avg) <= t / avg + 1 regions of cap slots — and there are at most min(nq, tuples / cap) of those
void pv_bounds(int64_t tuples, int64_t nq, int n_src, const PvTune &t, int64_t &regions, int64_t &region_tuples, int64_t &blocks) {
  regions = tuples / t.avg + nq + 1;
  region_tuples = (tuples / t.avg + 1) * (int64_t)t.cap + std::min<int64_t>(nq * (int64_t)t.cap, tuples) + 2 * nq + t.cap;
  blocks = ceil_div(tuples, kBlk) + nq * n_src;
}

}  // namespace

namespace sia {

size_t pvote_bytes(int64_t tuples, int64_t nq, int n_src, int topn) {
  int64_t regions, region_tuples, blocks;
  pv_bounds(tuples, nq, n_src, pv_tune(), regions, region_tuples, blocks);
  return pv_scratch_bytes(nq * n_src, nq, regions, region_tuples, blocks, topn);
}

int pvote_entry_info(const Lookup &L, longlong2 *d_info, uint32_t *d_qh, cudaStream_t s) {
  if (L.n == 0) return SIA_OK;
  pv_entry_info_kernel<<<grid_for(L.n), 256, 0, s>>>(L.ent, L.first, L.off_all, L.cnt_head, L.n, d_info, d_qh);
  SIA_CHECK_LAUNCH();
  return SIA_OK;
}

int pvote_entries(Arena &ar, const Lookup &L, const longlong2 *d_info, const uint32_t *d_qh, const uint64_t *post, const int64_t *d_qs,
                  int64_t i0, const int64_t *d_goff, const int64_t *h_goff, int qa, int qb, int qid_base, int topn, const PvOut &out,
                  uint32_t *d_qover, uint32_t *d_qbins, unsigned long long *d_nbins, cudaStream_t s, StageEvents &tm) {
  const int nq = qb - qa;
  if (nq <= 0) return SIA_OK;
  int rc = pv_attrs();
  if (rc) return rc;
  const PvTune tune = pv_tune();
  int64_t regions = 0, region_tuples = 0, blocks = 0;
  uint32_t maxp = 1;
  for (int q = qa; q < qb; ++q) {
    const uint64_t t = (uint64_t)(h_goff[q + 1] - h_goff[q]);
    if (t == 0) continue;
    const uint32_t np = pv_parts(t, tune.cap, tune.avg);
    maxp = std::max(maxp, np);
    regions += np;
    region_tuples += (int64_t)np * pv_region_cap(t, tune.cap);
    blocks += (int64_t)ceil_div((int64_t)t, kBlk);
  }
  if (blocks == 0) return SIA_OK;
  SIA_REQUIRE(blocks < (1ll << 31) && regions < (1ll << 31), SIA_E_UNSUPPORTED, "vote: group too large");
  PvScratch S;
  SIA_REQUIRE(pv_take(ar, S, nq, nq, regions, region_tuples, blocks, topn), SIA_E_NOMEM,
              "index scratch arena too small (partitioned vote)");
  tm.mark(0, s);
  SIA_CUDA(cudaMemsetAsync(S.fill, 0, sizeof(uint32_t) * regions, s));
  pv_segs_entries_kernel<<<grid_for(nq), 256, 0, s>>>(d_goff, qa, nq, S.seg_lo, S.seg_cnt, 0, 0, 0);
  pv_layout_kernel<<<1, 1024, 0, s>>>(S.seg_cnt, nq, 1, tune, S.pq, S.q_ridx0, S.seg_blk0, S.tot);
  pv_maps_kernel<<<grid_for(regions + blocks), 256, 0, s>>>(S.seg_blk0, nq, S.q_ridx0, nq, S.tot, S.blk_seg, S.reg_q);
  ScatterArgs a{};
  a.seg_blk0 = S.seg_blk0; a.blk_seg = S.blk_seg; a.seg_lo = S.seg_lo; a.seg_cnt = S.seg_cnt; a.G = 1;
  a.pq = S.pq; a.tot = S.tot; a.regions = S.regions; a.fill = S.fill; a.qover = d_qover; a.q_lo = qa;
  a.maxp = (int)std::min<uint32_t>(kMaxParts, (maxp + 511u) & ~511u);
  a.off = L.off_all; a.info = d_info; a.qh = d_qh; a.post = post; a.q_ent = d_qs; a.i0 = i0;
  tm.mark(1, s);
  pv_scatter_kernel<0><<<(unsigned)blocks, kScThreads, scatter_smem(a.maxp), s>>>(a);
  tm.mark(2, s);
  pv_count_kernel<<<(unsigned)ceil_div(regions, kRegionsPerCta), kCntThreads, kCountSmem, s>>>(S.regions, S.fill, S.pq, S.reg_q, S.tot, qa, d_qover, topn, S.cand,
                                                                     d_nbins ? d_qbins : nullptr);
  pv_merge_kernel<<<(unsigned)ceil_div((int64_t)nq * 32, 256), 256, 0, s>>>(S.cand, S.pq, nq, qa, qid_base, d_qover, topn, out, nullptr,
                                                                            d_qbins, d_nbins);
  SIA_CHECK_LAUNCH();
  tm.mark(3, s);
  return SIA_OK;
}

int pvote_key_slots(Arena &ar, const uint64_t *d_keys, int n_slots, int64_t cap, const int64_t *d_counts, int nq, int topn,
                    const PvOut &out, uint32_t *d_qover, uint32_t *d_flags2, cudaStream_t s) {
  if (nq <= 0) return SIA_OK;
  int rc = pv_attrs();
  if (rc) return rc;
  const PvTune tune = pv_tune();
  const int64_t T = (int64_t)n_slots * cap;                 // upper bound of the keys
  int64_t regions, region_tuples, blocks;
  pv_bounds(T, nq, n_slots, tune, regions, region_tuples, blocks);
  SIA_REQUIRE(blocks < (1ll << 31) && regions < (1ll << 31), SIA_E_UNSUPPORTED, "vote: too many keys in one call");
  const int64_t n_seg = (int64_t)nq * n_slots;
  PvScratch S;
  SIA_REQUIRE(pv_take(ar, S, n_seg, nq, regions, region_tuples, blocks, topn), SIA_E_NOMEM, "vote scratch too small (partitioned vote)");
  SIA_CUDA(cudaMemsetAsync(S.fill, 0, sizeof(uint32_t) * regions, s));
  pv_segs_keys_kernel<<<grid_for(n_seg), 256, 0, s>>>(d_keys, cap, d_counts, n_slots, nq, S.seg_lo, S.seg_cnt, d_flags2);
  pv_layout_kernel<<<1, 1024, 0, s>>>(S.seg_cnt, nq, n_slots, tune, S.pq, S.q_ridx0, S.seg_blk0, S.tot);
  pv_maps_kernel<<<grid_for(regions + blocks), 256, 0, s>>>(S.seg_blk0, (int)n_seg, S.q_ridx0, nq, S.tot, S.blk_seg, S.reg_q);
  ScatterArgs a{};
  a.seg_blk0 = S.seg_blk0; a.blk_seg = S.blk_seg; a.seg_lo = S.seg_lo; a.seg_cnt = S.seg_cnt; a.G = n_slots;
  a.pq = S.pq; a.tot = S.tot; a.regions = S.regions; a.fill = S.fill; a.qover = d_qover; a.q_lo = 0;
  a.maxp = kMaxParts;                                       // the queries' sizes are only known on the device
  a.keys = d_keys; a.key_cap = cap; a.counts = d_counts; a.unsorted = d_flags2;
  pv_scatter_kernel<1><<<(unsigned)blocks, kScThreads, kScatterSmem, s>>>(a);
  pv_count_kernel<<<(unsigned)ceil_div(regions, kRegionsPerCta), kCntThreads, kCountSmem, s>>>(S.regions, S.fill, S.pq, S.reg_q, S.tot, 0, d_qover, topn, S.cand,
                                                                     nullptr);
  pv_merge_kernel<<<(unsigned)ceil_div((int64_t)nq * 32, 256), 256, 0, s>>>(S.cand, S.pq, nq, 0, 0, d_qover, topn, out, d_flags2 + 1,
                                                                            nullptr, nullptr);
  // dedup_hashes of the winners: the head tuples of their songs, from the regions (queries left to the table vote have
  // no winners yet and are skipped)
  pv_rows_kernel<<<(unsigned)std::min<int64_t>(regions, kNumSMs * 16), 256, 0, s>>>(S.regions, S.fill, S.pq, S.reg_q, S.tot, 0, 0, d_qover, topn, out.song, out.nres,
                                                   out.rows);
  SIA_CHECK_LAUNCH();
  return SIA_OK;
}

// ---- hash-prefix sharding over peer memory ----------------------------------------------------------------------
// Sender side: the posting runs of this shard's entries (queries of ALL ranks, numbered rank * qp + local) are scattered
// straight into the owners' regions through NVLink.  d_t_total: tuples of every global query over all shards (the
// all-reduced counts), from which every rank derives the same layout.
int pvote_scatter_peers(Arena &ar, const Lookup &L, const longlong2 *d_einfo, const uint32_t *d_qh, const uint64_t *post,
                        const int64_t *d_q_ent, const int64_t *d_goff, int world, int rank, int qp, const int64_t *d_t_total,
                        void *const *peer_regions, void *const *peer_fill, void *const *peer_qover, int64_t region_cap,
                        int64_t fill_cap, int64_t *d_info, cudaStream_t s) {
  SIA_REQUIRE(world >= 1 && world <= kPvMaxPeers && rank >= 0 && rank < world, SIA_E_UNSUPPORTED, "peer scatter: at most 16 ranks");
  int rc = pv_attrs();
  if (rc) return rc;
  const PvTune tune = pv_tune();
  const int nq = world * qp;
  const int64_t blocks = ceil_div(std::max<int64_t>(L.tuples, 1), kBlk) + nq;
  SIA_REQUIRE(blocks < (1ll << 31), SIA_E_UNSUPPORTED, "peer scatter: pass too large");
  int64_t *seg_lo = ar.take<int64_t>(nq);
  uint32_t *seg_cnt = ar.take<uint32_t>(nq), *seg_blk0 = ar.take<uint32_t>(nq + 1), *q_ridx2 = ar.take<uint32_t>(nq + 1);
  uint32_t *tot = ar.take<uint32_t>(4), *blk_seg = ar.take<uint32_t>(blocks), *reg_q2 = ar.take<uint32_t>(1);
  PvQuery *pq = ar.take<PvQuery>(nq), *pq2 = ar.take<PvQuery>(nq);
  int64_t *dest_tot = ar.take<int64_t>(2 * (size_t)world);
  SIA_REQUIRE(seg_lo && seg_cnt && seg_blk0 && q_ridx2 && tot && blk_seg && reg_q2 && pq && pq2 && dest_tot, SIA_E_NOMEM,
              "index scratch arena too small (peer scatter)");
  pv_segs_entries_kernel<<<grid_for(nq), 256, 0, s>>>(d_goff, 0, nq, seg_lo, seg_cnt, world, rank, qp);
  // blocks of the LOCAL tuples (pq2 / q_ridx2 are by-products nobody reads) ...
  pv_layout_kernel<<<1, 1024, 0, s>>>(seg_cnt, nq, 1, tune, pq2, q_ridx2, seg_blk0, tot);
  // ... regions from the TOTAL counts, per owner
  pv_layout_dest_kernel<<<world, 1024, 0, s>>>(d_t_total, qp, tune, pq, nullptr, dest_tot, region_cap, fill_cap,
                                               reinterpret_cast<unsigned long long *>(d_info));
  pv_gate_kernel<<<1, 1, 0, s>>>(reinterpret_cast<const unsigned long long *>(d_info), tot, 1);
  pv_blocks_only_kernel<<<1, 1, 0, s>>>(tot, tot + 2);                  // the block -> query map only (no regions here)
  pv_maps_kernel<<<grid_for(blocks), 256, 0, s>>>(seg_blk0, nq, q_ridx2, nq, tot + 2, blk_seg, reg_q2);
  ScatterArgs a{};
  a.seg_blk0 = seg_blk0; a.blk_seg = blk_seg; a.seg_lo = seg_lo; a.seg_cnt = seg_cnt; a.G = 1;
  a.pq = pq; a.tot = tot; a.q_lo = 0; a.maxp = kMaxParts;
  a.qp_dest = qp; a.il_world = world; a.il_rank = rank;
  for (int d = 0; d < world; ++d) {
    a.regions_p[d] = static_cast<uint64_t *>(peer_regions[d]);
    a.fill_p[d] = static_cast<uint32_t *>(peer_fill[d]);
    a.qover_p[d] = static_cast<uint32_t *>(peer_qover[d]);
  }
  a.off = L.off_all; a.info = d_einfo; a.qh = d_qh; a.post = post; a.q_ent = d_q_ent; a.i0 = 0;
  pv_scatter_kernel<0><<<(unsigned)blocks, kScThreads, kScatterSmem, s>>>(a);
  SIA_CHECK_LAUNCH();
  return SIA_OK;
}

// Owner side: count + merge + rows over the regions the shards filled.  d_t_total: this rank's qp queries.
int pvote_count_regions(Arena &ar, const int64_t *d_t_total, int nq, int topn, uint64_t *d_regions, uint32_t *d_fill,
                        uint32_t *d_qover, int64_t region_cap, int64_t fill_cap, const PvOut &out, int64_t *d_info,
                        uint32_t *d_over_count, cudaStream_t s) {
  if (nq <= 0) return SIA_OK;
  int rc = pv_attrs();
  if (rc) return rc;
  const PvTune tune = pv_tune();
  const int64_t regions = fill_cap;                       // upper bound of the grid; the kernels stop at tot[0]
  PvQuery *pq = ar.take<PvQuery>(nq);
  uint32_t *q_ridx0 = ar.take<uint32_t>(nq + 1), *tot = ar.take<uint32_t>(4), *reg_q = ar.take<uint32_t>(regions);
  uint32_t *blk_seg = ar.take<uint32_t>(1), *seg_blk0 = ar.take<uint32_t>(2);
  int64_t *dest_tot = ar.take<int64_t>(2);
  uint64_t *cand = ar.take<uint64_t>(regions * topn);
  SIA_REQUIRE(pq && q_ridx0 && tot && reg_q && blk_seg && seg_blk0 && dest_tot && cand, SIA_E_NOMEM, "vote scratch too small (regions)");
  pv_layout_dest_kernel<<<1, 1024, 0, s>>>(d_t_total, nq, tune, pq, q_ridx0, dest_tot, region_cap, fill_cap,
                                           reinterpret_cast<unsigned long long *>(d_info));
  pv_set_regions_kernel<<<1, 1, 0, s>>>(dest_tot, tot);
  pv_gate_kernel<<<1, 1, 0, s>>>(reinterpret_cast<const unsigned long long *>(d_info), tot, 0);
  SIA_CUDA(cudaMemsetAsync(seg_blk0, 0, 2 * sizeof(uint32_t), s));
  pv_maps_kernel<<<grid_for(regions), 256, 0, s>>>(seg_blk0, 1, q_ridx0, nq, tot, blk_seg, reg_q);
  pv_count_kernel<<<(unsigned)ceil_div(regions, kRegionsPerCta), kCntThreads, kCountSmem, s>>>(d_regions, d_fill, pq, reg_q, tot, 0, d_qover, topn, cand, nullptr);
  pv_merge_kernel<<<(unsigned)ceil_div((int64_t)nq * 32, 256), 256, 0, s>>>(cand, pq, nq, 0, 0, d_qover, topn, out, d_over_count, nullptr,
                                                                            nullptr);
  pv_rows_kernel<<<(unsigned)std::min<int64_t>(regions, kNumSMs * 16), 256, 0, s>>>(d_regions, d_fill, pq, reg_q, tot, 0, 0, d_qover, topn, out.song, out.nres, out.rows);
  SIA_CHECK_LAUNCH();
  return SIA_OK;
}

}  // namespace sia
