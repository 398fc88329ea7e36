// K4, build side — the `fingerprints` table (mysql_database.py:46-59) as key table + packed postings (index.cuh), its
// INSERT IGNORE (:62-68, 167-181), ON DELETE CASCADE (:56-57, 132-139) and the row export used for persistence.
//
// sia_index_finalize is INCREMENTAL: it sorts only the pending rows (LSD radix sort, 16-byte records), probes the
// table for each of them (directory + binary search -> posting position, duplicate?, new hash?), writes the merged key
// table into the second key buffer and shifts the postings in place, back to front, through a small staging chunk —
// O(pending · log) + one pass over the part of the table behind the first inserted row; no full re-sort and no
// table-sized allocation (the reference's ingest commits per song, __init__.py:381-386).
#include "index.cuh"

using namespace sia;

namespace {

constexpr int64_t kStageRows = 32ll << 20;     // postings per staging chunk (256 MB)
constexpr int kTile = 256;                     // rows per tile of the delete compaction

__global__ void __launch_bounds__(256)
pack_rows_kernel(const uint8_t *__restrict__ hash, const int32_t *__restrict__ off, const int32_t *__restrict__ song_arr,
                 int32_t song_const, int64_t n, ulonglong2 *__restrict__ out, int32_t *__restrict__ status) {
  int32_t smax = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    uint64_t hi; uint32_t lo16;
    load_digest(hash + i * SIA_HASH_BYTES, hi, lo16);
    const int32_t song = song_arr ? song_arr[i] : song_const;
    const int32_t o = off[i];
    if (song < 0 || song > (int32_t)kM24 || o < 0 || o > (int32_t)kM24) atomicOr(status, 1);
    else smax = max(smax, song);
    out[i] = make_ulonglong2(((uint64_t)lo16 << 48) | (((uint64_t)song & kM24) << 24) | ((uint64_t)o & kM24), hi);
  }
#pragma unroll
  for (int d = 16; d; d >>= 1) smax = max(smax, __shfl_xor_sync(0xffffffffu, smax, d));
  if ((threadIdx.x & 31) == 0 && smax > 0) atomicMax(status + 1, smax);
}

// dir[b] = first record whose bucket (top `bits` bits of the digest) is >= b; one binary search per bucket, so a
// skewed key set costs nothing extra
__global__ void __launch_bounds__(256)
build_dir_kernel(const ulonglong2 *__restrict__ r, int64_t n, int bits, uint32_t *__restrict__ dir) {
  const int64_t nb = 1ll << bits;
  for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b <= nb; b += (int64_t)gridDim.x * blockDim.x) {
    int64_t lo = 0, hi = n;
    if (b == nb) lo = n;
    else
      while (lo < hi) {
        const int64_t mid = lo + ((hi - lo) >> 1);
        if ((int64_t)(r[mid].y >> (64 - bits)) < b) lo = mid + 1; else hi = mid;
      }
    dir[b] = (uint32_t)lo;
  }
}

// One sorted pending row against the table: rank = the posting index it goes in front of, kidx = the first key whose
// hash is >= the row's, bit 63 of rank = the hash already has a key; keep = 0 for a duplicate of the previous pending
// row or of a stored row (INSERT IGNORE).
constexpr uint64_t kFound = 1ull << 63;

__global__ void __launch_bounds__(256)
probe_kernel(const ulonglong2 *__restrict__ p, int64_t m, const ulonglong2 *__restrict__ keys, int64_t n_keys,
             const uint32_t *__restrict__ dir, int bits, const uint64_t *__restrict__ post, uint32_t *__restrict__ keep,
             uint64_t *__restrict__ rank, uint32_t *__restrict__ kidx) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const ulonglong2 r = p[i];
    const uint32_t lo16 = (uint32_t)(r.x >> 48);
    const uint64_t so = r.x & kM48;
    bool dup = i > 0 && rec_eq(p[i - 1], r);
    const int64_t ki = hash_lower_bound_dir(keys, dir, bits, r.y, lo16);
    const ulonglong2 k = keys[ki];                       // ki == n_keys: the sentinel (start = n_rows)
    uint64_t rk = k.x & kM48;
    if (ki < n_keys && k.y == r.y && (uint32_t)(k.x >> 48) == lo16) {
      const int64_t e = (int64_t)(keys[ki + 1].x & kM48);
      const int64_t pos = lower_bound_u64(post, (int64_t)rk, e, so);
      if (pos < e && post[pos] == so) dup = true;
      rk = (uint64_t)pos | kFound;
    }
    keep[i] = dup ? 0u : 1u;
    rank[i] = rk;
    kidx[i] = (uint32_t)ki;
  }
}

__global__ void __launch_bounds__(256)
compact_pending_kernel(const ulonglong2 *__restrict__ p, const uint64_t *__restrict__ rank, const uint32_t *__restrict__ kidx,
                       const uint32_t *__restrict__ keep, const int64_t *__restrict__ pos, int64_t m,
                       ulonglong2 *__restrict__ q, uint64_t *__restrict__ rank2, uint32_t *__restrict__ kidx2) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x)
    if (keep[i]) { const int64_t o = pos[i]; q[o] = p[i]; rank2[o] = rank[i]; kidx2[o] = kidx[i]; }
}

// first pending row of a hash that has no key yet
__global__ void __launch_bounds__(256)
newkey_flag_kernel(const ulonglong2 *__restrict__ q, const uint64_t *__restrict__ rank, int64_t m, uint32_t *__restrict__ nk) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x)
    nk[i] = (!(rank[i] & kFound) && (i == 0 || !same_hash(q[i], q[i - 1]))) ? 1u : 0u;
}

// old key j (and the sentinel, j == n_keys) moves behind the new keys with a smaller hash; its run starts
// `a` postings later, a = pending rows with a smaller hash
__global__ void __launch_bounds__(256)
merge_old_keys_kernel(const ulonglong2 *__restrict__ keys, int64_t n_keys, const ulonglong2 *__restrict__ q, int64_t m,
                      const uint32_t *__restrict__ dirq, int bq, const int64_t *__restrict__ nkpos,
                      ulonglong2 *__restrict__ out) {
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j <= n_keys; j += (int64_t)gridDim.x * blockDim.x) {
    const ulonglong2 k = keys[j];
    const int64_t a = j == n_keys ? m : hash_lower_bound_dir(q, dirq, bq, k.y, (uint32_t)(k.x >> 48));
    out[j + nkpos[a]] = make_ulonglong2((k.x & ~kM48) | ((k.x & kM48) + (uint64_t)a), k.y);
  }
}

__global__ void __launch_bounds__(256)
merge_new_keys_kernel(const ulonglong2 *__restrict__ q, const uint64_t *__restrict__ rank, const uint32_t *__restrict__ kidx,
                      const uint32_t *__restrict__ nk, const int64_t *__restrict__ nkpos, int64_t m,
                      ulonglong2 *__restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x)
    if (nk[i]) {
      const ulonglong2 r = q[i];
      out[(int64_t)kidx[i] + nkpos[i]] = make_ulonglong2((r.x & ~kM48) | ((rank[i] & kM48) + (uint64_t)i), r.y);
    }
}

__device__ __forceinline__ int64_t upper_bound_rank(const uint64_t *__restrict__ rank, int64_t lo, int64_t hi, uint64_t p) {
  while (lo < hi) { const int64_t mid = lo + ((hi - lo) >> 1); if ((rank[mid] & kM48) <= p) lo = mid + 1; else hi = mid; }
  return lo;
}

// stored posting p moves to p + (pending rows that go in front of it); the chunk [a, b) was copied to `stage` first,
// chunks run back to front, so nothing that is still to be read is overwritten
__global__ void __launch_bounds__(256)
move_rows_kernel(const uint64_t *__restrict__ stage, int64_t a, int64_t b, const uint64_t *__restrict__ rank, int64_t m,
                 uint64_t *__restrict__ post) {
  __shared__ int64_t s_c[2];
  const int64_t p0 = a + (int64_t)blockIdx.x * 1024;
  const int64_t p1 = min(b, p0 + 1024);
  if (threadIdx.x < 2) s_c[threadIdx.x] = upper_bound_rank(rank, 0, m, (uint64_t)(threadIdx.x == 0 ? p0 : p1 - 1));
  __syncthreads();
  const int64_t c_lo = s_c[0], c_hi = s_c[1];
  for (int64_t p = p0 + threadIdx.x; p < p1; p += 256) {
    const int64_t c = c_lo == c_hi ? c_lo : upper_bound_rank(rank, c_lo, c_hi, (uint64_t)p);
    post[p + c] = stage[p - a];
  }
}

__global__ void __launch_bounds__(256)
scatter_pending_kernel(const ulonglong2 *__restrict__ q, const uint64_t *__restrict__ rank, int64_t m,
                       uint64_t *__restrict__ post) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x)
    post[(int64_t)(rank[i] & kM48) + i] = q[i].x & kM48;
}

// ---- delete (ON DELETE CASCADE) ---------------------------------------------------------------------------
// one block = one tile of 256 postings: keep bits (1 = the song stays) + kept rows of the tile
__global__ void __launch_bounds__(kTile)
flag_rows_kernel(const uint64_t *__restrict__ post, int64_t n, const uint32_t *__restrict__ dead, uint32_t *__restrict__ keepbits,
                 uint32_t *__restrict__ tile_cnt) {
  __shared__ uint32_t s_cnt[kTile / 32];
  const int64_t p = (int64_t)blockIdx.x * kTile + threadIdx.x;
  bool keep = false;
  if (p < n) {
    const uint32_t song = (uint32_t)(post[p] >> 24) & 0xffffffu;
    keep = !((dead[song >> 5] >> (song & 31)) & 1u);
  }
  const uint32_t bits = __ballot_sync(0xffffffffu, keep);
  if ((threadIdx.x & 31) == 0) { keepbits[p >> 5] = bits; s_cnt[threadIdx.x >> 5] = __popc(bits); }
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t c = 0;
#pragma unroll
    for (int w = 0; w < kTile / 32; ++w) c += s_cnt[w];
    tile_cnt[blockIdx.x] = c;
  }
}

// rows kept in front of posting index s (s <= n)
__device__ __forceinline__ int64_t kept_before(int64_t s, int64_t n, int64_t keep_total, const uint32_t *__restrict__ keepbits,
                                               const int64_t *__restrict__ tile_base) {
  if (s >= n) return keep_total;
  const int64_t t = s / kTile;
  int64_t c = tile_base[t];
  const int64_t w0 = t * (kTile / 32), w1 = s >> 5;
  for (int64_t w = w0; w < w1; ++w) c += __popc(keepbits[w]);
  return c + __popc(keepbits[w1] & ((1u << (s & 31)) - 1u));
}

__global__ void __launch_bounds__(256)
key_restart_kernel(const ulonglong2 *__restrict__ keys, int64_t n_keys, int64_t n, int64_t keep_total,
                   const uint32_t *__restrict__ keepbits, const int64_t *__restrict__ tile_base, int64_t *__restrict__ ns) {
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j <= n_keys; j += (int64_t)gridDim.x * blockDim.x)
    ns[j] = kept_before((int64_t)(keys[j].x & kM48), n, keep_total, keepbits, tile_base);
}

__global__ void __launch_bounds__(256)
key_alive_kernel(const int64_t *__restrict__ ns, int64_t n_keys, uint32_t *__restrict__ alive) {
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n_keys; j += (int64_t)gridDim.x * blockDim.x)
    alive[j] = ns[j + 1] > ns[j] ? 1u : 0u;
}

__global__ void __launch_bounds__(256)
compact_keys_kernel(const ulonglong2 *__restrict__ keys, int64_t n_keys, const int64_t *__restrict__ ns,
                    const uint32_t *__restrict__ alive, const int64_t *__restrict__ kpos, ulonglong2 *__restrict__ out) {
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j <= n_keys; j += (int64_t)gridDim.x * blockDim.x) {
    const ulonglong2 k = keys[j];
    if (j == n_keys || alive[j]) out[kpos[j]] = make_ulonglong2((k.x & ~kM48) | (uint64_t)ns[j], k.y);
  }
}

// kept postings of the staged chunk [a, b) (a is a multiple of the tile) move forward to their final position
__global__ void __launch_bounds__(kTile)
compact_rows_kernel(const uint64_t *__restrict__ stage, int64_t a, int64_t b, const uint32_t *__restrict__ keepbits,
                    const int64_t *__restrict__ tile_base, uint64_t *__restrict__ post) {
  const int64_t t = a / kTile + blockIdx.x;
  const int64_t p = t * kTile + threadIdx.x;
  if (p >= b) return;
  const int w = threadIdx.x >> 5;
  const uint32_t bits = keepbits[t * (kTile / 32) + w];
  if (!((bits >> (threadIdx.x & 31)) & 1u)) return;
  int64_t c = tile_base[t] + __popc(bits & ((1u << (threadIdx.x & 31)) - 1u));
  for (int u = 0; u < w; ++u) c += __popc(keepbits[t * (kTile / 32) + u]);
  post[c] = stage[p - a];
}

// ---- export / select -----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
export_rows_kernel(const ulonglong2 *__restrict__ keys, int64_t n_keys, const uint64_t *__restrict__ post, int64_t first_row,
                   int64_t n, uint8_t *__restrict__ hash, int32_t *__restrict__ song, int32_t *__restrict__ off) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t r = (uint64_t)(first_row + i);
    int64_t lo = 0, hi = n_keys;             // first key whose run starts behind row r; the row's key is the one before
    while (lo < hi) { const int64_t mid = lo + ((hi - lo) >> 1); if ((keys[mid].x & kM48) <= r) lo = mid + 1; else hi = mid; }
    const ulonglong2 k = keys[lo - 1];
    store_digest(hash + i * SIA_HASH_BYTES, k.y, (uint32_t)(k.x >> 48));
    const uint64_t v = post[r];
    song[i] = (int32_t)((v >> 24) & kM24);
    off[i] = (int32_t)(v & kM24);
  }
}

int set_device(const sia_index *ix) {
  SIA_CUDA(cudaSetDevice(ix->device));
  return SIA_OK;
}

int ensure_keys(sia_index *ix, int which, int64_t entries) {
  if (ix->keys_cap[which] >= entries) return SIA_OK;
  if (ix->keys[which]) cudaFree(ix->keys[which]);
  ix->keys[which] = nullptr; ix->keys_cap[which] = 0;
  const int64_t want = entries + (entries >> 2) + 1024;
  SIA_CUDA(cudaMalloc(&ix->keys[which], (size_t)want * sizeof(ulonglong2)));
  ix->keys_cap[which] = want;
  return SIA_OK;
}

int ensure_stage(sia_index *ix, int64_t rows) {
  if (ix->stage_cap >= rows) return SIA_OK;
  if (ix->stage) cudaFree(ix->stage);
  ix->stage = nullptr; ix->stage_cap = 0;
  SIA_CUDA(cudaMalloc(&ix->stage, (size_t)rows * sizeof(uint64_t)));
  ix->stage_cap = rows;
  return SIA_OK;
}

// directory over the current key table: ~8 keys per bucket
int rebuild_dir(sia_index *ix, cudaStream_t s) {
  int bits = 10;
  while (bits < 28 && (ix->n_keys >> bits) > 8) ++bits;
  const int64_t entries = (1ll << bits) + 1;
  if (entries > ix->dir_cap) {
    if (ix->dir) cudaFree(ix->dir);
    ix->dir = nullptr; ix->dir_cap = 0;
    SIA_CUDA(cudaMalloc(&ix->dir, (size_t)entries * sizeof(uint32_t)));
    ix->dir_cap = entries;
  }
  ix->dir_bits = bits;
  build_dir_kernel<<<grid_for(entries), 256, 0, s>>>(ix->keys[ix->cur], ix->n_keys, bits, ix->dir);
  SIA_CHECK_LAUNCH();
  return SIA_OK;
}

// sort the pending rows and merge them into the table (header comment)
int merge_pending(sia_index *ix, cudaStream_t s) {
  const int64_t M = ix->n_pending, N = ix->n_rows, D = ix->n_keys;
  SIA_REQUIRE(M < 0xfffffff0ll, SIA_E_CAPACITY, "finalize: 2^32 or more pending rows; call sia_index_finalize more often");
  int bq = 10;
  while (bq < 27 && (M >> bq) > 8) ++bq;
  int rc = ix->arena.reserve(radix_sort_tmp_bytes(M) + (size_t)M * (4 + 8 + 8 + 4 + 8 + 4) + 32 + scan_tmp_bytes(M) +
                             ((size_t)(1ll << bq) + 1) * 4 + (1 << 16));
  if (rc) return rc;
  Arena &ar = ix->arena;
  void *stmp = ar.take<char>(radix_sort_tmp_bytes(M));
  uint32_t *keep = ar.take<uint32_t>(M);
  int64_t *pos = ar.take<int64_t>(M + 1);
  void *sc = ar.take<char>(scan_tmp_bytes(M));
  uint64_t *rank = ar.take<uint64_t>(M), *rank2 = ar.take<uint64_t>(M);
  uint32_t *kidx = ar.take<uint32_t>(M), *kidx2 = ar.take<uint32_t>(M);
  uint32_t *dirq = ar.take<uint32_t>((size_t)(1ll << bq) + 1);
  SIA_REQUIRE(stmp && keep && pos && sc && rank && rank2 && kidx && kidx2 && dirq, SIA_E_NOMEM,
              "index scratch arena too small (finalize)");
  bool in_b = false;
  if ((rc = radix_sort(ix->pend[0], ix->pend[1], M, 16, 0, 16, stmp, s, &in_b))) return rc;
  const ulonglong2 *P = in_b ? ix->pend[1] : ix->pend[0];
  ulonglong2 *other = in_b ? ix->pend[0] : ix->pend[1];
  const ulonglong2 *keys = ix->keys[ix->cur];
  probe_kernel<<<grid_for(M), 256, 0, s>>>(P, M, keys, D, ix->dir, ix->dir_bits, ix->post, keep, rank, kidx);
  SIA_CHECK_LAUNCH();
  if ((rc = exclusive_scan_u32(keep, pos, M, sc, s))) return rc;
  int64_t Mk = 0;
  SIA_CUDA(cudaMemcpyAsync(&Mk, pos + M, sizeof Mk, cudaMemcpyDeviceToHost, s));
  SIA_CUDA(cudaStreamSynchronize(s));
  if (Mk == 0) { ix->n_pending = 0; return SIA_OK; }             // every pending row was already stored
  SIA_REQUIRE(N + Mk <= ix->capacity, SIA_E_CAPACITY, "index capacity exceeded");
  const ulonglong2 *Q = P;
  if (Mk != M) {
    compact_pending_kernel<<<grid_for(M), 256, 0, s>>>(P, rank, kidx, keep, pos, M, other, rank2, kidx2);
    SIA_CHECK_LAUNCH();
    Q = other; rank = rank2; kidx = kidx2;
  }
  // keys that do not exist yet (keep / pos are free again: reuse them for the flags and their scan)
  uint32_t *nk = keep;
  int64_t *nkpos = pos;
  newkey_flag_kernel<<<grid_for(Mk), 256, 0, s>>>(Q, rank, Mk, nk);
  SIA_CHECK_LAUNCH();
  if ((rc = exclusive_scan_u32(nk, nkpos, Mk, sc, s))) return rc;
  int64_t K = 0;
  uint64_t first_rank = 0;
  SIA_CUDA(cudaMemcpyAsync(&K, nkpos + Mk, sizeof K, cudaMemcpyDeviceToHost, s));
  SIA_CUDA(cudaMemcpyAsync(&first_rank, rank, sizeof first_rank, cudaMemcpyDeviceToHost, s));
  SIA_CUDA(cudaStreamSynchronize(s));
  SIA_REQUIRE(D + K < 0xfffffff0ll, SIA_E_CAPACITY, "index: 2^32 or more distinct hashes in one shard");
  bq = 10;
  while (bq < 27 && (Mk >> bq) > 8) ++bq;
  build_dir_kernel<<<grid_for((1ll << bq) + 1), 256, 0, s>>>(Q, Mk, bq, dirq);
  SIA_CHECK_LAUNCH();
  const int nxt = ix->cur ^ 1;
  if ((rc = ensure_keys(ix, nxt, D + K + 1))) return rc;
  merge_old_keys_kernel<<<grid_for(D + 1), 256, 0, s>>>(keys, D, Q, Mk, dirq, bq, nkpos, ix->keys[nxt]);
  SIA_CHECK_LAUNCH();
  if (K) {
    merge_new_keys_kernel<<<grid_for(Mk), 256, 0, s>>>(Q, rank, kidx, nk, nkpos, Mk, ix->keys[nxt]);
    SIA_CHECK_LAUNCH();
  }
  // postings: everything behind the first inserted row shifts, back to front through the staging chunk
  const int64_t lo_move = (int64_t)(first_rank & kM48);
  if (N > lo_move) {
    if ((rc = ensure_stage(ix, std::min<int64_t>(kStageRows, N - lo_move)))) return rc;
    for (int64_t b = N; b > lo_move;) {
      const int64_t a = std::max(lo_move, b - ix->stage_cap);
      SIA_CUDA(cudaMemcpyAsync(ix->stage, ix->post + a, (size_t)(b - a) * sizeof(uint64_t), cudaMemcpyDeviceToDevice, s));
      move_rows_kernel<<<(unsigned)ceil_div(b - a, 1024), 256, 0, s>>>(ix->stage, a, b, rank, Mk, ix->post);
      SIA_CHECK_LAUNCH();
      b = a;
    }
  }
  scatter_pending_kernel<<<grid_for(Mk), 256, 0, s>>>(Q, rank, Mk, ix->post);
  SIA_CHECK_LAUNCH();
  ix->cur = nxt;
  ix->n_keys = D + K;
  ix->n_rows = N + Mk;
  ix->n_pending = 0;
  if ((rc = rebuild_dir(ix, s))) return rc;
  SIA_CUDA(cudaStreamSynchronize(s));
  return SIA_OK;
}

int insert_common(sia_index *ix, const int32_t *d_song, int32_t song_const, const uint8_t *d_hash, const int32_t *d_off,
                  int64_t n, cudaStream_t s) {
  SIA_REQUIRE(ix != nullptr, SIA_E_INVALID, "index is NULL");
  SIA_REQUIRE(n >= 0, SIA_E_INVALID, "n < 0");
  if (n == 0) return SIA_OK;
  SIA_REQUIRE(d_hash && d_off, SIA_E_INVALID, "NULL argument");
  int rc = set_device(ix);
  if (rc) return rc;
  if (ix->n_rows + ix->n_pending + n > ix->capacity) {
    set_error("index capacity exceeded (capacity_rows counts stored + pending rows)");
    return SIA_E_CAPACITY;
  }
  if (ix->n_pending + n > ix->pend_cap) {          // grow the pending buffers (earlier inserts may still be in flight)
    const int64_t want = std::max<int64_t>({ix->n_pending + n, ix->pend_cap + (ix->pend_cap >> 1), 1ll << 16});
    ulonglong2 *nb[2] = {nullptr, nullptr};
    SIA_CUDA(cudaDeviceSynchronize());
    for (int k = 0; k < 2; ++k) {
      cudaError_t e = cudaMalloc(&nb[k], (size_t)want * sizeof(ulonglong2));
      if (e != cudaSuccess) { if (nb[0]) cudaFree(nb[0]); return cuda_fail(e, "pending buffer", __FILE__, __LINE__); }
    }
    if (ix->n_pending)
      SIA_CUDA(cudaMemcpy(nb[0], ix->pend[0], (size_t)ix->n_pending * sizeof(ulonglong2), cudaMemcpyDeviceToDevice));
    for (int k = 0; k < 2; ++k) { if (ix->pend[k]) cudaFree(ix->pend[k]); ix->pend[k] = nb[k]; }
    ix->pend_cap = want;
  }
  pack_rows_kernel<<<grid_for(n), 256, 0, s>>>(d_hash, d_off, d_song, song_const, n, ix->pend[0] + ix->n_pending, ix->status);
  SIA_CHECK_LAUNCH();
  SIA_CUDA(cudaEventRecord(ix->insert_done, s));
  ix->n_pending += n;
  return SIA_OK;
}

}  // namespace

extern "C" {

int sia_index_create(int device, int64_t capacity_rows, sia_index **out) {
  SIA_REQUIRE(out != nullptr, SIA_E_INVALID, "out is NULL");
  *out = nullptr;
  SIA_REQUIRE(capacity_rows > 0 && capacity_rows < (1ll << 40), SIA_E_INVALID, "capacity_rows must be in 1 .. 2^40-1");
  int ndev = 0;
  SIA_CUDA(cudaGetDeviceCount(&ndev));
  SIA_REQUIRE(device >= 0 && device < ndev, SIA_E_INVALID, "no such CUDA device");
  SIA_CUDA(cudaSetDevice(device));
  sia_index *ix = new (std::nothrow) sia_index();
  SIA_REQUIRE(ix != nullptr, SIA_E_NOMEM, "out of host memory");
  ix->device = device;
  ix->capacity = capacity_rows;
  const ulonglong2 sentinel = make_ulonglong2(0xffffull << 48, ~0ull);       // all-ones hash, start 0
  cudaError_t e = cudaMalloc(&ix->post, (size_t)capacity_rows * sizeof(uint64_t));
  if (e == cudaSuccess) e = cudaMalloc(&ix->status, 2 * sizeof(int32_t));
  if (e == cudaSuccess) e = cudaMemset(ix->status, 0, 2 * sizeof(int32_t));
  if (e == cudaSuccess) e = cudaMalloc(&ix->keys[0], 1024 * sizeof(ulonglong2));
  if (e == cudaSuccess) e = cudaMemcpy(ix->keys[0], &sentinel, sizeof sentinel, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix->insert_done, cudaEventDisableTiming);
  if (e != cudaSuccess) {
    int rc = cuda_fail(e, "index allocation", __FILE__, __LINE__);
    sia_index_destroy(ix);
    return rc;
  }
  ix->keys_cap[0] = 1024;
  int rc = rebuild_dir(ix, nullptr);
  if (!rc && cudaDeviceSynchronize() != cudaSuccess) rc = cuda_fail(cudaGetLastError(), "index create", __FILE__, __LINE__);
  if (rc) { sia_index_destroy(ix); return rc; }
  *out = ix;
  return SIA_OK;
}

int sia_index_destroy(sia_index *ix) {
  if (!ix) return SIA_OK;
  cudaSetDevice(ix->device);
  cudaDeviceSynchronize();
  if (ix->post) cudaFree(ix->post);
  for (int k = 0; k < 2; ++k) { if (ix->keys[k]) cudaFree(ix->keys[k]); if (ix->pend[k]) cudaFree(ix->pend[k]); }
  if (ix->dir) cudaFree(ix->dir);
  if (ix->status) cudaFree(ix->status);
  if (ix->stage) cudaFree(ix->stage);
  if (ix->insert_done) cudaEventDestroy(ix->insert_done);
  for (cudaEvent_t e : ix->ev_q) if (e) cudaEventDestroy(e);
  ix->ev_stage.release();
  ix->arena.release();
  ix->arena3.release();
  delete ix;
  return SIA_OK;
}

int64_t sia_index_rows(const sia_index *ix) { return ix ? ix->n_rows : 0; }
int64_t sia_index_keys(const sia_index *ix) { return ix ? ix->n_keys : 0; }
int32_t sia_index_max_song(const sia_index *ix) { return ix ? ix->max_song : 0; }

int sia_index_insert(sia_index *ix, int32_t song_id, const uint8_t *d_hash, const int32_t *d_off, int64_t n, void *stream) {
  SIA_REQUIRE(song_id >= 0 && song_id <= (int32_t)kM24, SIA_E_INVALID, "song_id outside MEDIUMINT UNSIGNED (0..2^24-1)");
  return insert_common(ix, nullptr, song_id, d_hash, d_off, n, (cudaStream_t)stream);
}

int sia_index_insert_rows(sia_index *ix, const int32_t *d_song, const uint8_t *d_hash, const int32_t *d_off, int64_t n,
                          void *stream) {
  SIA_REQUIRE(d_song != nullptr || n == 0, SIA_E_INVALID, "NULL argument");
  return insert_common(ix, d_song, 0, d_hash, d_off, n, (cudaStream_t)stream);
}

int sia_index_insert_host(sia_index *ix, int32_t song_id, const uint8_t *h_hash, const int32_t *h_off, int64_t n) {
  SIA_REQUIRE(ix != nullptr, SIA_E_INVALID, "index is NULL");
  if (n == 0) return SIA_OK;
  SIA_REQUIRE(h_hash && h_off && n > 0, SIA_E_INVALID, "bad argument");
  int rc = set_device(ix);
  if (rc) return rc;
  SIA_CUDA(cudaDeviceSynchronize());               // the arena may still be read by an earlier call's kernels
  if ((rc = ix->arena.reserve((size_t)n * (SIA_HASH_BYTES + 4) + 4096))) return rc;
  uint8_t *dh = ix->arena.take<uint8_t>((size_t)n * SIA_HASH_BYTES);
  int32_t *dof = ix->arena.take<int32_t>(n);
  SIA_CUDA(cudaMemcpy(dh, h_hash, (size_t)n * SIA_HASH_BYTES, cudaMemcpyHostToDevice));
  SIA_CUDA(cudaMemcpy(dof, h_off, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice));
  rc = sia_index_insert(ix, song_id, dh, dof, n, nullptr);
  if (rc) return rc;
  SIA_CUDA(cudaDeviceSynchronize());
  return SIA_OK;
}

int sia_index_finalize(sia_index *ix, int64_t *h_rows) {
  SIA_REQUIRE(ix != nullptr, SIA_E_INVALID, "index is NULL");
  int rc = set_device(ix);
  if (rc) return rc;
  SIA_CUDA(cudaEventSynchronize(ix->insert_done));        // inserts may have been enqueued on any stream
  cudaStream_t s = nullptr;
  int32_t st[2] = {0, 0};
  SIA_CUDA(cudaMemcpy(st, ix->status, sizeof st, cudaMemcpyDeviceToHost));
  if (st[0] & 1) {
    st[0] &= ~1;                                            // clear only this flag
    SIA_CUDA(cudaMemcpy(ix->status, st, sizeof(int32_t), cudaMemcpyHostToDevice));
    ix->n_pending = 0;                                      // drop the offending batch
    set_error("insert: song_id or offset outside 0..2^24-1");
    return SIA_E_INVALID;
  }
  ix->max_song = st[1];
  if (ix->n_pending > 0 && (rc = merge_pending(ix, s))) return rc;
  if (h_rows) *h_rows = ix->n_rows;
  return SIA_OK;
}

int sia_index_delete_songs(sia_index *ix, const int32_t *h_song_ids, int32_t n, int64_t *h_rows) {
  SIA_REQUIRE(ix != nullptr, SIA_E_INVALID, "index is NULL");
  SIA_REQUIRE(ix->n_pending == 0, SIA_E_INVALID, "index has pending rows: call sia_index_finalize first");
  if (h_rows) *h_rows = ix->n_rows;
  if (n <= 0 || ix->n_rows == 0) return SIA_OK;
  SIA_REQUIRE(h_song_ids != nullptr, SIA_E_INVALID, "NULL argument");
  int rc = set_device(ix);
  if (rc) return rc;
  cudaStream_t s = nullptr;
  SIA_CUDA(cudaDeviceSynchronize());
  std::vector<uint32_t> bitmap((1u << 24) / 32, 0u);
  for (int i = 0; i < n; ++i) {
    SIA_REQUIRE(h_song_ids[i] >= 0 && h_song_ids[i] <= (int32_t)kM24, SIA_E_INVALID, "song id out of range");
    bitmap[h_song_ids[i] >> 5] |= 1u << (h_song_ids[i] & 31);
  }
  const int64_t N = ix->n_rows, D = ix->n_keys;
  const int64_t tiles = ceil_div(N, kTile);
  const int64_t scan_n = std::max(tiles, D + 1);
  if ((rc = ix->arena.reserve(bitmap.size() * 4 + (size_t)tiles * (kTile / 8 + 4 + 8) + (size_t)(D + 2) * (8 + 4 + 8) +
                              scan_tmp_bytes(scan_n) + (1 << 16))))
    return rc;
  Arena &ar = ix->arena;
  uint32_t *d_bm = ar.take<uint32_t>(bitmap.size());
  uint32_t *keepbits = ar.take<uint32_t>((size_t)tiles * (kTile / 32));
  uint32_t *tile_cnt = ar.take<uint32_t>(tiles);
  int64_t *tile_base = ar.take<int64_t>(tiles + 1);
  int64_t *ns = ar.take<int64_t>(D + 1);
  uint32_t *alive = ar.take<uint32_t>(D + 1);
  int64_t *kpos = ar.take<int64_t>(D + 2);
  void *sc = ar.take<char>(scan_tmp_bytes(scan_n));
  SIA_REQUIRE(d_bm && keepbits && tile_cnt && tile_base && ns && alive && kpos && sc, SIA_E_NOMEM,
              "index scratch arena too small (delete)");
  SIA_CUDA(cudaMemcpyAsync(d_bm, bitmap.data(), bitmap.size() * 4, cudaMemcpyHostToDevice, s));
  flag_rows_kernel<<<(unsigned)tiles, kTile, 0, s>>>(ix->post, N, d_bm, keepbits, tile_cnt);
  SIA_CHECK_LAUNCH();
  if ((rc = exclusive_scan_u32(tile_cnt, tile_base, tiles, sc, s))) return rc;
  int64_t keep = 0;
  SIA_CUDA(cudaMemcpyAsync(&keep, tile_base + tiles, sizeof keep, cudaMemcpyDeviceToHost, s));
  SIA_CUDA(cudaStreamSynchronize(s));
  if (keep == N) return SIA_OK;
  // keys: new run starts; a key whose run is gone disappears
  const ulonglong2 *keys = ix->keys[ix->cur];
  key_restart_kernel<<<grid_for(D + 1), 256, 0, s>>>(keys, D, N, keep, keepbits, tile_base, ns);
  key_alive_kernel<<<grid_for(D), 256, 0, s>>>(ns, D, alive);
  SIA_CHECK_LAUNCH();
  if ((rc = exclusive_scan_u32(alive, kpos, D, sc, s))) return rc;        // kpos[D] = keys left = slot of the sentinel
  int64_t Dk = 0;
  SIA_CUDA(cudaMemcpyAsync(&Dk, kpos + D, sizeof Dk, cudaMemcpyDeviceToHost, s));
  SIA_CUDA(cudaStreamSynchronize(s));
  const int nxt = ix->cur ^ 1;
  if ((rc = ensure_keys(ix, nxt, Dk + 1))) return rc;
  compact_keys_kernel<<<grid_for(D + 1), 256, 0, s>>>(keys, D, ns, alive, kpos, ix->keys[nxt]);
  SIA_CHECK_LAUNCH();
  // postings: kept rows move forward, front to back through the staging chunk (chunks are whole tiles)
  if ((rc = ensure_stage(ix, std::min<int64_t>(kStageRows, tiles * kTile)))) return rc;
  const int64_t chunk = ix->stage_cap / kTile * kTile;
  for (int64_t a = 0; a < N; a += chunk) {
    const int64_t b = std::min(N, a + chunk);
    SIA_CUDA(cudaMemcpyAsync(ix->stage, ix->post + a, (size_t)(b - a) * sizeof(uint64_t), cudaMemcpyDeviceToDevice, s));
    compact_rows_kernel<<<(unsigned)ceil_div(b - a, kTile), kTile, 0, s>>>(ix->stage, a, b, keepbits, tile_base, ix->post);
    SIA_CHECK_LAUNCH();
  }
  ix->cur = nxt;
  ix->n_keys = Dk;
  ix->n_rows = keep;
  if ((rc = rebuild_dir(ix, s))) return rc;
  SIA_CUDA(cudaStreamSynchronize(s));
  if (h_rows) *h_rows = ix->n_rows;
  return SIA_OK;
}

int sia_index_trim(sia_index *ix) {
  SIA_REQUIRE(ix != nullptr, SIA_E_INVALID, "index is NULL");
  SIA_REQUIRE(ix->n_pending == 0, SIA_E_INVALID, "index has pending rows: call sia_index_finalize first");
  int rc = set_device(ix);
  if (rc) return rc;
  SIA_CUDA(cudaDeviceSynchronize());
  for (int k = 0; k < 2; ++k) { if (ix->pend[k]) cudaFree(ix->pend[k]); ix->pend[k] = nullptr; }
  ix->pend_cap = 0;
  const int other = ix->cur ^ 1;
  if (ix->keys[other]) cudaFree(ix->keys[other]);
  ix->keys[other] = nullptr; ix->keys_cap[other] = 0;
  if (ix->stage) cudaFree(ix->stage);
  ix->stage = nullptr; ix->stage_cap = 0;
  ix->arena.release();
  ix->arena3.release();
  vote_scratch_release(ix->device);
  return SIA_OK;
}

int sia_index_export(sia_index *ix, int64_t first_row, int64_t n, uint8_t *d_hash, int32_t *d_song, int32_t *d_off,
                     void *stream) {
  SIA_REQUIRE(ix != nullptr, SIA_E_INVALID, "index is NULL");
  SIA_REQUIRE(ix->n_pending == 0, SIA_E_INVALID, "index has pending rows: call sia_index_finalize first");
  SIA_REQUIRE(first_row >= 0 && n >= 0 && first_row + n <= ix->n_rows, SIA_E_INVALID, "export: row range outside the index");
  if (n == 0) return SIA_OK;
  SIA_REQUIRE(d_hash && d_song && d_off, SIA_E_INVALID, "NULL output");
  int rc = set_device(ix);
  if (rc) return rc;
  export_rows_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(ix->keys[ix->cur], ix->n_keys, ix->post, first_row, n,
                                                                    d_hash, d_song, d_off);
  SIA_CHECK_LAUNCH();
  return SIA_OK;
}

}  // extern "C"
