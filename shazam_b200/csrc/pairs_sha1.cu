// K3 — generate_hashes (__init__.py:179-210): for every peak i (in (t asc, f asc) order)
// and partner j = 1..fan_value-1 with i+j inside the same track and
// 0 <= t[i+j]-t[i] <= MAX_HASH_TIME_DELTA(200):
//     h = sha1(f"{f1}|{f2}|{dt}")    -> first 10 digest bytes (= hexdigest()[0:20]), t1
// emitted in the reference's list order (i major, j minor).
//
// Peaks are time-sorted, so dt >= 0 and the valid partners of a peak form a prefix
// j = 1..m_i.  pairs_count computes m_i, a scan turns it into output offsets, and
// pairs_sha1 runs one thread per (i, j): the decimal ASCII message is 5..13 bytes, i.e.
// always ONE 64-byte SHA-1 block, hashed with a 16-word rolling schedule in registers.
// The path is tiny in bytes (~15 KB per audio second) and bound by INT32 issue — unless the context holds the digest
// table (below), which turns it into a gather.
#include "sia_common.cuh"
#include "stft.cuh"

namespace sia {

namespace {

__global__ void __launch_bounds__(256)
pairs_count_kernel(const int32_t *__restrict__ peak_t, const int64_t *__restrict__ track_peak_starts, int n_tracks,
                   int fan_value, const int64_t *__restrict__ final_t, uint32_t *__restrict__ pair_count) {
  const int64_t n_peaks = track_peak_starts[n_tracks];
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_peaks; i += (int64_t)gridDim.x * blockDim.x) {
    const int trk = find_segment(track_peak_starts, n_tracks, i);
    const int64_t e = track_peak_starts[trk + 1];
    const int t1 = peak_t[i];
    int m = 0;
    // streaming: an anchor whose partners are not all known yet (fewer than fan_value-1 peaks behind it, and a later
    // peak could still lie within MAX_HASH_TIME_DELTA) gets no pairs in this pass
    if (final_t && i + fan_value - 1 >= e && t1 > final_t[trk]) { pair_count[i] = 0; continue; }
    for (int j = 1; j < fan_value; ++j) {
      if (i + j >= e) break;
      const int dt = peak_t[i + j] - t1;
      if (dt < 0 || dt > SIA_MAX_DT) break;   // MIN_HASH_TIME_DELTA <= dt <= MAX_HASH_TIME_DELTA
      ++m;
    }
    pair_count[i] = (uint32_t)m;
  }
}

__device__ __forceinline__ uint32_t rotl(uint32_t x, int n) { return __funnelshift_l(x, x, n); }

// message bytes accumulate big-endian in a 128-bit shift register
struct Msg {
  uint64_t hi = 0, lo = 0;
  int n = 0;
  __device__ __forceinline__ void push(uint32_t byte) {
    hi = (hi << 8) | (lo >> 56);
    lo = (lo << 8) | byte;
    ++n;
  }
  __device__ __forceinline__ void push_dec(uint32_t v) {   // decimal ASCII, no leading zeros, v < 100000
    if (v >= 10000) push('0' + v / 10000 % 10);
    if (v >= 1000) push('0' + v / 1000 % 10);
    if (v >= 100) push('0' + v / 100 % 10);
    if (v >= 10) push('0' + v / 10 % 10);
    push('0' + v % 10);
  }
};

// SHA-1 of a message of n <= 15 bytes held left-aligned in w0..w3 (0x80 already appended).
__device__ __forceinline__ void sha1_one_block(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3, uint32_t bitlen,
                                               uint32_t &h0, uint32_t &h1, uint32_t &h2) {
  uint32_t w[16] = {w0, w1, w2, w3, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, bitlen};
  uint32_t a = 0x67452301u, b = 0xEFCDAB89u, c = 0x98BADCFEu, d = 0x10325476u, e = 0xC3D2E1F0u;
#pragma unroll
  for (int t = 0; t < 80; ++t) {
    if (t >= 16) w[t & 15] = rotl(w[(t + 13) & 15] ^ w[(t + 8) & 15] ^ w[(t + 2) & 15] ^ w[t & 15], 1);
    uint32_t f, k;
    if (t < 20) { f = (b & c) | (~b & d); k = 0x5A827999u; }
    else if (t < 40) { f = b ^ c ^ d; k = 0x6ED9EBA1u; }
    else if (t < 60) { f = (b & c) | (b & d) | (c & d); k = 0x8F1BBCDCu; }
    else { f = b ^ c ^ d; k = 0xCA62C1D6u; }
    const uint32_t tmp = rotl(a, 5) + f + e + k + w[t & 15];
    e = d; d = c; c = rotl(b, 30); b = a; a = tmp;
  }
  h0 = 0x67452301u + a;
  h1 = 0xEFCDAB89u + b;
  h2 = 0x98BADCFEu + c;
}

// first 10 digest bytes of sha1(f"{f1}|{f2}|{dt}") as five 16-bit words in memory order (f1, f2 < 100000, dt < 100000:
// the message is at most 17 bytes; 15 is the one-block limit of the 128-bit register, so callers bound the digits)
__device__ __forceinline__ void pair_digest(uint32_t f1, uint32_t f2, uint32_t dt, uint32_t &w01, uint32_t &w23, uint32_t &w4) {
  Msg m;
  m.push_dec(f1); m.push('|'); m.push_dec(f2); m.push('|'); m.push_dec(dt);
  const uint32_t bitlen = (uint32_t)m.n * 8u;
  m.push(0x80u);
  // left-align the m.n (<= 16) bytes in the 16-byte register
  const int sh = (16 - m.n) * 8;                 // 0..80 bits
  uint64_t hi = m.hi, lo = m.lo;
  if (sh >= 64) { hi = lo << (sh - 64); lo = 0; }
  else if (sh > 0) { hi = (hi << sh) | (lo >> (64 - sh)); lo <<= sh; }
  uint32_t h0, h1, h2;
  sha1_one_block((uint32_t)(hi >> 32), (uint32_t)hi, (uint32_t)(lo >> 32), (uint32_t)lo, bitlen, h0, h1, h2);
  // big-endian digest bytes as little-endian 16-bit pairs
  const uint32_t d0 = ((h0 >> 24) & 0xff) | ((h0 >> 8) & 0xff00), d1 = ((h0 >> 8) & 0xff) | ((h0 << 8) & 0xff00);
  const uint32_t d2 = ((h1 >> 24) & 0xff) | ((h1 >> 8) & 0xff00), d3 = ((h1 >> 8) & 0xff) | ((h1 << 8) & 0xff00);
  w01 = d0 | (d1 << 16); w23 = d2 | (d3 << 16);
  w4 = ((h2 >> 24) & 0xff) | ((h2 >> 8) & 0xff00);
}

// Digest table: the whole pre-image space of the pipeline's hashes — f1, f2 in 0..2048, dt in 0..200 — is
// 2049 * 2049 * 201 = 8.4e8 messages; one 16-byte entry each (10 digest bytes + padding, one aligned load) is 13.5 GB of
// a 180 GB HBM.  It is filled once per context by the SHA-1 code above, after which K3 is a gather (one 32-byte DRAM
// sector per hash) instead of 80 rounds of integer ALU work per hash.
constexpr int64_t kTabF = SIA_NBINS, kTabDt = SIA_MAX_DT + 1;
__device__ __forceinline__ int64_t table_index(uint32_t f1, uint32_t f2, uint32_t dt) {
  return ((int64_t)f1 * kTabF + f2) * kTabDt + dt;
}

__global__ void __launch_bounds__(256)
digest_table_kernel(uint4 *__restrict__ table, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t dt = (uint32_t)(i % kTabDt);
    const int64_t ff = i / kTabDt;
    uint4 v;
    pair_digest((uint32_t)(ff / kTabF), (uint32_t)(ff % kTabF), dt, v.x, v.y, v.z);
    v.w = 0;
    table[i] = v;
  }
}

__global__ void __launch_bounds__(256)
pairs_sha1_kernel(const int32_t *__restrict__ peak_t, const int32_t *__restrict__ peak_f,
                  const int64_t *__restrict__ track_peak_starts, int n_tracks, int fan_value,
                  const uint32_t *__restrict__ pair_count, const int64_t *__restrict__ pair_off,
                  int64_t hash_base_static, const int64_t *__restrict__ d_hash_base, const uint4 *__restrict__ table,
                  uint8_t *__restrict__ out_hash, int32_t *__restrict__ out_t1, int64_t cap, int32_t *__restrict__ status) {
  const int64_t n_peaks = track_peak_starts[n_tracks];
  const int fan1 = fan_value - 1;
  const int64_t n_tasks = n_peaks * fan1;
  const int64_t hash_base = hash_base_static + (d_hash_base ? *d_hash_base : 0);
  for (int64_t task = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; task < n_tasks;
       task += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = task / fan1;
    const int j = (int)(task - i * fan1);          // partner i + j + 1
    if ((uint32_t)j >= pair_count[i]) continue;
    const uint32_t f1 = (uint32_t)peak_f[i], f2 = (uint32_t)peak_f[i + j + 1];
    const int t1 = peak_t[i];
    const uint32_t dt = (uint32_t)(peak_t[i + j + 1] - t1);
    const int64_t o = hash_base + pair_off[i] + j;
    if (o >= cap) { atomicOr(status, 2); continue; }
    if (f1 > 99999u || f2 > 99999u) { atomicOr(status, 4); continue; }     // outside the one-block message (see header)
    uint32_t w01, w23, w4;
    if (table && f1 < (uint32_t)kTabF && f2 < (uint32_t)kTabF) {
      const uint4 v = __ldg(table + table_index(f1, f2, dt));
      w01 = v.x; w23 = v.y; w4 = v.z;
    } else {
      pair_digest(f1, f2, dt, w01, w23, w4);
    }
    // digest bytes 0..9; o*10 is 2-byte aligned
    uint16_t *dst = reinterpret_cast<uint16_t *>(out_hash + o * SIA_HASH_BYTES);
    dst[0] = (uint16_t)w01; dst[1] = (uint16_t)(w01 >> 16);
    dst[2] = (uint16_t)w23; dst[3] = (uint16_t)(w23 >> 16);
    dst[4] = (uint16_t)w4;
    out_t1[o] = t1;
  }
}

__global__ void track_hash_starts_kernel(const int64_t *__restrict__ track_peak_starts, int n_tracks,
                                         const int64_t *__restrict__ pair_off, int64_t hash_base_static,
                                         const int64_t *__restrict__ d_hash_base, int64_t *__restrict__ track_hash_starts) {
  const int64_t hash_base = hash_base_static + (d_hash_base ? *d_hash_base : 0);
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b <= n_tracks; b += gridDim.x * blockDim.x)
    track_hash_starts[b] = hash_base + pair_off[track_peak_starts[b]];
}

}  // namespace

int pairs_count_launch(const int32_t *d_peak_t, const int64_t *d_track_peak_starts, int n_tracks,
                       int64_t n_peaks_max, int fan_value, uint32_t *d_pair_count, cudaStream_t s,
                       const int64_t *d_final_t) {
  if (n_peaks_max == 0) return SIA_OK;
  int64_t blocks = ceil_div(n_peaks_max, 256);
  if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
  pairs_count_kernel<<<(unsigned)blocks, 256, 0, s>>>(d_peak_t, d_track_peak_starts, n_tracks, fan_value, d_final_t,
                                                      d_pair_count);
  SIA_CHECK_LAUNCH();
  return SIA_OK;
}

int pairs_sha1_launch(const int32_t *d_peak_t, const int32_t *d_peak_f, const int64_t *d_track_peak_starts,
                      int n_tracks, int64_t n_peaks_max, int fan_value, const uint32_t *d_pair_count,
                      const int64_t *d_pair_off, int64_t hash_base_static, const int64_t *d_hash_base,
                      const void *d_digest_table, uint8_t *d_hash, int32_t *d_t1, int64_t cap_hashes,
                      int64_t *d_track_hash_starts, int32_t *d_status, cudaStream_t s) {
  if (n_peaks_max > 0 && fan_value > 1) {
    int64_t blocks = ceil_div(n_peaks_max * (fan_value - 1), 256);
    if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
    pairs_sha1_kernel<<<(unsigned)blocks, 256, 0, s>>>(d_peak_t, d_peak_f, d_track_peak_starts, n_tracks, fan_value,
                                                     d_pair_count, d_pair_off, hash_base_static, d_hash_base,
                                                     static_cast<const uint4 *>(d_digest_table), d_hash, d_t1, cap_hashes,
                                                     d_status);
    SIA_CHECK_LAUNCH();
  }
  if (d_track_hash_starts) {
    track_hash_starts_kernel<<<(unsigned)ceil_div(n_tracks + 1, 256), 256, 0, s>>>(
        d_track_peak_starts, n_tracks, d_pair_off, hash_base_static, d_hash_base, d_track_hash_starts);
    SIA_CHECK_LAUNCH();
  }
  return SIA_OK;
}

size_t digest_table_bytes() { return (size_t)(kTabF * kTabF * kTabDt) * sizeof(uint4); }

int digest_table_build(void *d_table, cudaStream_t s) {
  const int64_t n = kTabF * kTabF * kTabDt;
  digest_table_kernel<<<kNumSMs * 16, 256, 0, s>>>(static_cast<uint4 *>(d_table), n);
  SIA_CHECK_LAUNCH();
  return SIA_OK;
}

}  // namespace sia
